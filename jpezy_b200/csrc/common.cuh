// common.cuh -- device-side constants and small helpers of libjpezy_b200.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>

#include "../../include/jpezy_b200.h"
#include "tables.h"

namespace jz {

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch: the pipelines are chains of 10-20 short kernels on one stream, and on a single image
// the gaps between them (kernel drain + launch latency) add up to more than a tenth of the step.  Every kernel starts
// with pdl_wait() (griddepcontrol.wait: all prerequisite grids complete, their writes visible), so a launch made with
// jz_launch() may be staged while its predecessor still runs.  The wait is a no-op for ordinary launches.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
inline bool pdl_enabled()
{
    static const bool on = [] { const char* e = std::getenv("JPEZY_B200_PDL"); return !e || e[0] != '0'; }();
    return on;
}
template <typename... KArgs, typename... Args>
inline cudaError_t jz_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args)
{
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at, cfg.numAttrs = pdl_enabled() ? 1u : 0u;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---------------------------------------------------------------------------------------------
// Constant bank: everything the transform kernels index with compile-time (uniform) indices.
// ---------------------------------------------------------------------------------------------
struct DevConst {
    double cos_ref[64];    // the reference's table, used by the exact-order recompute path
    double inv_sqrt2_ref;  // 1.0/sqrt(2.0) as the reference evaluates it
    float cosf_[64];       // ideal cosines in float (fast paths)
    uint16_t quant[2][64]; // [0]=luma, [1]=chroma, natural order (Annex K, src/jpezy.hpp:131-152)
    float rquant[2][64];   // 1/q
    uint8_t zz[64];        // zig-zag position -> natural position (src/jpezy.hpp:36-45)
    uint8_t izz[64];       // natural position -> zig-zag position
};
static __constant__ DevConst cC;   // single translation unit (capi.cu)
// the same cosine table in global memory, for the fix-up phases whose lanes index it divergently (a constant-bank
// load serialises per distinct address; an L1 load does not)
static __device__ double gCosRef[64];

// Huffman encoder LUT, one per table class (0 = luma tables, 1 = chroma tables).
// ac[(run << 4) | size] and dc[category]; entry = (code << 5) | length, 0 = invalid.
struct HuffEncLut {
    uint32_t ac[256];
    uint32_t dc[16];
};


// 32-bit load through a shared-space address (no generic-address arithmetic)
__device__ __forceinline__ uint32_t lds32(uint32_t saddr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}

// number of 16x16 MCUs along one dimension
__host__ __device__ inline uint32_t mcu_units(uint32_t n) { return (n + 15u) >> 4; }

__device__ __forceinline__ int bit_length(int a)  // number of significant bits of a >= 0
{
    return 32 - __clz(a);
}

}  // namespace jz
