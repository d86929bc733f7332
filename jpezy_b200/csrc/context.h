// context.h -- the context behind the C ABI and the host-side state it owns.  Host code only: capi.cu includes it after
// the kernel headers, whose launch parameter types it holds.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <string>

#include "../../include/jpezy_b200.h"

#define JZ_CUDA_TRY(ctx, expr)                                                                  \
    do {                                                                                        \
        cudaError_t e__ = (expr);                                                               \
        if (e__ != cudaSuccess) return (ctx)->fail_cuda(e__, #expr, __LINE__);                  \
    } while (0)

// Growable device buffer owned by the context
struct jz_devbuf {
    void* p = nullptr;
    size_t cap = 0;
    jz_devbuf() = default;
    jz_devbuf(const jz_devbuf&) = delete;
    jz_devbuf& operator=(const jz_devbuf&) = delete;
    ~jz_devbuf()
    {
        if (p) cudaFree(p);
    }
};

namespace jz {

// host copy of the launch parameters between the phases of the MCU-row sharded encoder (capi_shard.inc)
struct ShardState {
    bool valid = false;
    int phase = 0;          // last completed phase: 1 = A, 2 = B, 3 = C
    ShardParams sp{};
    uint32_t nmcu = 0;
};

// streams, events and double buffers of the pipelined host batches (capi_batch.inc); the streams and events are created
// by the first batch
struct BatchPipe {
    cudaStream_t h2d = nullptr, d2h = nullptr;
    cudaEvent_t e_in[2] = {nullptr, nullptr}, e_k[2] = {nullptr, nullptr}, e_sz[2] = {nullptr, nullptr}, e_out[2] = {nullptr, nullptr};
    jz_devbuf in[2], mid[2], out[2], sz[2];
    uint64_t* h_sz[2] = {nullptr, nullptr};     // pinned
    size_t h_sz_cap = 0;

    void destroy_handles()
    {
        for (cudaStream_t* s : {&h2d, &d2h})
            if (*s) cudaStreamDestroy(*s), *s = nullptr;
        for (int j = 0; j < 2; ++j)
            for (cudaEvent_t* e : {&e_in[j], &e_k[j], &e_sz[j], &e_out[j]})
                if (*e) cudaEventDestroy(*e), *e = nullptr;
    }
    ~BatchPipe()
    {
        destroy_handles();
        for (uint64_t* h : h_sz)
            if (h) cudaFreeHost(h);
    }
};

// per-frame tables of an inverse-transform kernel, keyed by the quantisation tables (cached_table, capi_decode.inc)
struct TableCache {
    static constexpr int kSlots = 4;
    void* tab[kSlots] = {};
    uint16_t key[kSlots][3][64] = {};
    int next = 0;
    ~TableCache()
    {
        for (void* t : tab)
            if (t) cudaFree(t);
    }
};

}  // namespace jz

struct jpezyb200_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t aux_stream = nullptr;          // side stream of the decoder: zero-fills overlap the synchronisation kernels
    cudaEvent_t aux_fork = nullptr, aux_join = nullptr;
    std::string err;
    int pad_ones = 1;
    uint32_t restart_interval = 0;   // JPEZYB200_OPT_RESTART_INTERVAL: MCUs per restart interval of the encoders, 0 = none
    bool fp64_transforms = false;   // JPEZYB200_OPT_TRANSFORM = 1: the FP64 validation kernels
    int sync_guesses = 0;     // JPEZYB200_OPT_SYNC_GUESSES
    int sync_rounds = 3;      // launches behind launch 0 (which checks the CTA boundaries itself): two that repair, one that verifies
    int64_t shard_scratch = 0;                 // JPEZYB200_OPT_SHARD_SCRATCH_BYTES (0 = 3 bytes per pixel)
    int64_t group_bytes = int64_t(96) << 20;   // host<->device bytes per stage of the pipelined host batches
    uint64_t launches = 0;
    int num_sms = 148;                         // SMs of the device
    jz::TableCache inv2_tabs, invg_tabs;       // tables of k_inv_transform2 and of k_idct_blocks (general frame layouts)
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
    jz_devbuf rst_base;        // [nimg][intervals + 1] byte bases of the restart intervals (enc_entropy.cuh)
    jz_devbuf sym_hist, huff_lut;  // optimised Huffman tables (enc_huffopt.cuh): symbol counts (zeroed when allocated), [nimg][2] LUTs
    jz_devbuf shard_geom;      // ShardGeom + scratch of the MCU-row sharded encoder (enc_shard.cuh)
    jz::BatchPipe pipe;
    jz::ShardState shard;
    // pinned, kReadbackWords words: what a call reads back to the host before it returns (sizes, status, Huffman tables).
    // One is enough: the context serves one host thread at a time, and every such call synchronises before it returns.
    static constexpr size_t kReadbackWords = 8192;
    uint64_t* h_readback = nullptr;

    ~jpezyb200_ctx()
    {
        if (h_readback) cudaFreeHost(h_readback);
        if (d_enc_lut) cudaFree(d_enc_lut);
        if (d_dec_lut) cudaFree(d_dec_lut);
        if (d_counters) cudaFree(d_counters);
        if (d_y_exact) cudaFree(d_y_exact);
        if (aux_fork) cudaEventDestroy(aux_fork);
        if (aux_join) cudaEventDestroy(aux_join);
        if (aux_stream) cudaStreamDestroy(aux_stream);
        if (stream) cudaStreamDestroy(stream);
    }

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
    // the pinned read-back buffer, allocated by the first call that needs it
    int readback(uint64_t** out)
    {
        if (!h_readback) JZ_CUDA_TRY(this, cudaMallocHost(reinterpret_cast<void**>(&h_readback), kReadbackWords * sizeof(uint64_t)));
        *out = h_readback;
        return JPEZYB200_OK;
    }
};
