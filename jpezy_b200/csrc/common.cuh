// common.cuh -- device-side constants, small helpers and the context of libjpezy_b200.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <string>

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

#define JZ_CUDA_TRY(ctx, expr)                                                                  \
    do {                                                                                        \
        cudaError_t e__ = (expr);                                                               \
        if (e__ != cudaSuccess) return (ctx)->fail_cuda(e__, #expr, __LINE__);                  \
    } while (0)

}  // namespace jz

// Growable device buffer owned by the context
struct jz_devbuf {
    void* p = nullptr;
    size_t cap = 0;
};

struct jpezyb200_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t aux_stream = nullptr;          // side stream of the decoder: zero-fills overlap the synchronisation kernels
    cudaEvent_t aux_fork = nullptr, aux_join = nullptr;
    std::string err;
    int pad_ones = 1;
    bool fp64_transforms = false;   // JPEZYB200_OPT_TRANSFORM = 1: the FP64 validation kernels
    int sync_guesses = 0;     // JPEZYB200_OPT_SYNC_GUESSES
    int sync_rounds = 3;      // launches behind launch 0 (which checks the CTA boundaries itself): two that repair, one that verifies
    int64_t shard_scratch = 0;                 // JPEZYB200_OPT_SHARD_SCRATCH_BYTES (0 = 3 bytes per pixel)
    int64_t group_bytes = int64_t(96) << 20;   // host<->device bytes per stage of the pipelined host batches
    uint64_t launches = 0;
    bool inv_attr_set = false, fwd_attr_set = false, inv2_attr_set = false;
    int num_sms = 148;                         // SMs of the device
    static constexpr int kInv2Slots = 4;       // tables of k_inv_transform2 per set of quantisation tables (capi_decode.inc)
    void* inv2_tab[kInv2Slots] = {};
    uint16_t inv2_key[kInv2Slots][3][64] = {};
    int inv2_next = 0;
    void* invg_tab[kInv2Slots] = {};           // ... and of k_idct_blocks (general frame layouts)
    uint16_t invg_key[kInv2Slots][3][64] = {};
    int invg_next = 0;
    bool invg_attr_set = false;
    jz_devbuf inv_samples;                     // [nimg][blocks][64] int16 between k_idct_blocks and k_colour_general

    // device-resident tables
    jz::HuffEncLut* d_enc_lut = nullptr;  // [2]
    // decoder tables are built per frame descriptor (cached by hash): [4] = DC luma, DC chroma, AC luma, AC chroma
    void* d_dec_lut = nullptr;
    uint64_t dec_lut_key = 0;

    // counters on the device: [0] guard_fwd, [1] guard_inv, [2] sync rounds, [3] scratch
    unsigned long long* d_counters = nullptr;
    int8_t* d_y_exact = nullptr;   // 64 KiB table of the exact luma cases (enc_transform.cuh)

    // scratch
    jz_devbuf coefs, blk_off, tile_sum, tile_base, img_bits, ustream, ff_sum, ff_base, planes_in, planes_out, scan_io, sizes_io;
    jz_devbuf dec_scanbytes, dec_chunk_cnt, dec_chunk_base, dec_ubytes, dec_state, dec_dirty, dec_subblk, dec_dc, dec_dcd, blk_meta, dec_status, dec_changed, dec_flags, dec_mcnt, dec_mbase, dec_seg;
    jz_devbuf sym_hist, huff_lut;  // optimised Huffman tables (enc_huffopt.cuh): symbol counts (zeroed when allocated), [nimg][2] LUTs
    jz_devbuf shard_geom;      // ShardGeom + scratch of the MCU-row sharded encoder (enc_shard.cuh)
    void* batch_pipe = nullptr;    // streams, events and double buffers of the pipelined host batches (capi_batch.inc)
    void* shard_state = nullptr;   // host copy of the launch parameters between the phases (capi_shard.inc)
    uint64_t* h_sizes = nullptr;   // pinned, 8192 values (jpezyb200_read_sizes)
    uint64_t* h_words = nullptr;   // pinned, 8 words: sizes / status read back by jpezyb200_encode / jpezyb200_decode
    void* h_huff = nullptr;        // pinned, kHuffReadback bytes: sizes + the four tables read back by jpezyb200_encode_optimized
    void* h_pinned = nullptr;
    size_t h_pinned_cap = 0;

    int fail_cuda(cudaError_t e, const char* what, int line)
    {
        char buf[512];
        snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s [capi.cu:%d]", int(e), cudaGetErrorString(e), what, line);
        err = buf;
        cudaGetLastError();
        return JPEZYB200_ECUDA;
    }
    int fail(int code, const char* msg)
    {
        err = msg;
        return code;
    }
    int ensure(jz_devbuf& b, size_t bytes)
    {
        if (bytes <= b.cap) return JPEZYB200_OK;
        if (b.p) cudaFree(b.p);
        b.p = nullptr, b.cap = 0;
        size_t want = bytes + (bytes >> 3) + 256;
        cudaError_t e = cudaMalloc(&b.p, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            err = "cudaMalloc failed for scratch buffer";
            return JPEZYB200_ENOMEM;
        }
        b.cap = want;
        return JPEZYB200_OK;
    }
    int ensure_pinned(size_t bytes)
    {
        if (bytes <= h_pinned_cap) return JPEZYB200_OK;
        if (h_pinned) cudaFreeHost(h_pinned);
        h_pinned = nullptr, h_pinned_cap = 0;
        if (cudaMallocHost(&h_pinned, bytes + 4096) != cudaSuccess) {
            cudaGetLastError();
            err = "cudaMallocHost failed";
            return JPEZYB200_ENOMEM;
        }
        h_pinned_cap = bytes + 4096;
        return JPEZYB200_OK;
    }
};
