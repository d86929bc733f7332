// capi.cu -- the C ABI of libjpezy_b200.so (include/jpezy_b200.h): context, table upload,
// kernel launches.  Single translation unit: all kernels are included here.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "common.cuh"
#include "dec_entropy.cuh"
#include "dec_transform.cuh"
#include "dec_transform2.cuh"
#include "dec_transform_g.cuh"
#include "enc_entropy.cuh"
#include "enc_huffopt.cuh"
#include "enc_transform.cuh"
#include "enc_shard.cuh"
#include "synth.cuh"
#include "context.h"

namespace jz {

// canonical Huffman code construction (T.81 Annex C.2); the same thing the reference's decoder
// does in analyze_dht (src/decoder/jpezy_decoder.hpp:223-239)
static void canonical_codes(const uint8_t bits[16], const uint8_t* vals, int nvals, uint16_t code_of[256], uint8_t len_of[256])
{
    std::memset(code_of, 0, 256 * sizeof(uint16_t));
    std::memset(len_of, 0, 256);
    int code = 0, k = 0;
    for (int len = 1; len <= 16; ++len) {
        for (int j = 0; j < bits[len - 1] && k < nvals; ++j, ++k) {
            code_of[vals[k]] = uint16_t(code++);
            len_of[vals[k]] = uint8_t(len);
        }
        code <<= 1;
    }
}

static void build_enc_lut(const HuffSpec& dc, const HuffSpec& ac, HuffEncLut* out)
{
    uint16_t code[256];
    uint8_t len[256];
    std::memset(out, 0, sizeof *out);
    canonical_codes(dc.bits, dc.vals, dc.nvals, code, len);
    for (int i = 0; i < 16; ++i) out->dc[i] = len[i] ? (uint32_t(code[i]) << 5) | len[i] : 0u;
    canonical_codes(ac.bits, ac.vals, ac.nvals, code, len);
    for (int i = 0; i < 256; ++i) out->ac[i] = len[i] ? (uint32_t(code[i]) << 5) | len[i] : 0u;
}

static cudaStream_t pick_stream(jpezyb200_ctx* ctx, void* s) { return s ? static_cast<cudaStream_t>(s) : ctx->stream; }

}  // namespace jz

using namespace jz;

extern "C" {

int jpezyb200_abi_version(void) { return JPEZYB200_ABI_VERSION; }

const char* jpezyb200_strerror(int code)
{
    switch (code) {
    case JPEZYB200_OK: return "ok";
    case JPEZYB200_EINVAL: return "invalid argument";
    case JPEZYB200_ECAPACITY: return "output buffer too small";
    case JPEZYB200_ECUDA: return "CUDA error";
    case JPEZYB200_ENCCL: return "collective error";
    case JPEZYB200_ECORRUPT: return "corrupt entropy-coded segment";
    case JPEZYB200_ENODEVICE: return "no CUDA device (libjpezy_b200 has no CPU path)";
    case JPEZYB200_ENOMEM: return "out of memory";
    case JPEZYB200_EUNSUPPORTED: return "unsupported frame layout";
    case JPEZYB200_EAGAIN: return "parallel Huffman decoder needs more synchronisation rounds";
    default: return "unknown error";
    }
}

const char* jpezyb200_last_error(const jpezyb200_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int jpezyb200_ctx_create(int device, jpezyb200_ctx** out)
{
    if (!out) return JPEZYB200_EINVAL;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        cudaGetLastError();
        return JPEZYB200_ENODEVICE;
    }
    if (device < 0 || device >= ndev) return JPEZYB200_EINVAL;
    jpezyb200_ctx* ctx = new (std::nothrow) jpezyb200_ctx();
    if (!ctx) return JPEZYB200_ENOMEM;
    ctx->device = device;
    if (cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || ctx->num_sms < 1) ctx->num_sms = 148;
    if (const char* e = std::getenv("JPEZY_B200_SYNC_ROUNDS")) ctx->sync_rounds = std::atoi(e);
    if (const char* e = std::getenv("JPEZY_B200_DEC_HYP")) ctx->sync_guesses = std::max(0, std::min(2, std::atoi(e)));      // (JPEZYB200_OPT_SYNC_GUESSES of every new context)      // (debugging: JPEZYB200_OPT_SYNC_ROUNDS of every new context)
    int rc = [&]() -> int {
        JZ_CUDA_TRY(ctx, cudaSetDevice(device));
        // static + dynamic shared memory of these kernels exceed 48 KiB: opt in once per context
        JZ_CUDA_TRY(ctx, cudaFuncSetAttribute(k_fwd_transform, cudaFuncAttributeMaxDynamicSharedMemorySize, kFwdTrSmem));
        JZ_CUDA_TRY(ctx, cudaFuncSetAttribute(k_inv_transform, cudaFuncAttributeMaxDynamicSharedMemorySize, kInvSmem));
        JZ_CUDA_TRY(ctx, cudaFuncSetAttribute(k_inv_transform2<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, Inv2<8>::kSmem));
        JZ_CUDA_TRY(ctx, cudaFuncSetAttribute(k_idct_blocks, cudaFuncAttributeMaxDynamicSharedMemorySize, InvG::kSmem));
        JZ_CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        DevConst h{};
        for (int i = 0; i < 64; ++i) {
            h.cos_ref[i] = kCosRef[i];
            h.cosf_[i] = float(std::cos((2 * (i & 7) + 1) * (i >> 3) * 3.14159265358979323846 / 16));
            h.quant[0][i] = kQuantLuma[i], h.quant[1][i] = kQuantChroma[i];
            h.rquant[0][i] = 1.0f / float(kQuantLuma[i]), h.rquant[1][i] = 1.0f / float(kQuantChroma[i]);
            h.zz[i] = kZigzag[i];
            h.izz[kZigzag[i]] = uint8_t(i);
        }
        h.inv_sqrt2_ref = kInvSqrt2Ref;
        JZ_CUDA_TRY(ctx, cudaMemcpyToSymbol(cC, &h, sizeof h));
        JZ_CUDA_TRY(ctx, cudaMemcpyToSymbol(gCosRef, h.cos_ref, sizeof h.cos_ref));
        {
            // constants of the FP32 AAN path per (class, column j): K folds the AAN scale factors, the /8 and 1/q; G is the guard
            // band (1.25 x worst-case flowgraph error + the rounding of w itself) in w units; T the "quantises to 0" test
            double aan[8];
            aan[0] = 1.0;
            for (int k = 1; k < 8; ++k) aan[k] = std::cos(k * 3.14159265358979323846 / 16) * std::sqrt(2.0);
            QuantCol col[2][8];
            uint2 izzc[8];
            for (int j = 0; j < 8; ++j) {
                uint8_t zb[8];
                for (int i = 0; i < 8; ++i) {
                    for (int c = 0; c < 2; ++c) {
                        const double q = c ? kQuantChroma[i * 8 + j] : kQuantLuma[i * 8 + j];
                        const double K = 1.0 / (8.0 * aan[i] * aan[j] * q);
                        const double Gd = (1.25 * kAanErrBound[i * 8 + j] + 5e-4) / q;
                        col[c][j].K[i] = float(K);
                        col[c][j].G[i] = float(Gd);
                        col[c][j].T[i] = float((1.0 - 2.0 * Gd) / K);
                    }
                    zb[i] = h.izz[i * 8 + j];
                }
                izzc[j].x = uint32_t(zb[0]) | (uint32_t(zb[1]) << 8) | (uint32_t(zb[2]) << 16) | (uint32_t(zb[3]) << 24);
                izzc[j].y = uint32_t(zb[4]) | (uint32_t(zb[5]) << 8) | (uint32_t(zb[6]) << 16) | (uint32_t(zb[7]) << 24);
            }
            JZ_CUDA_TRY(ctx, cudaMemcpyToSymbol(gQcol, col, sizeof col));
            JZ_CUDA_TRY(ctx, cudaMemcpyToSymbol(gIzzCol, izzc, sizeof izzc));
        }
        HuffEncLut lut[2];
        build_enc_lut(kDcLuma, kAcLuma, &lut[0]);
        build_enc_lut(kDcChroma, kAcChroma, &lut[1]);
        JZ_CUDA_TRY(ctx, cudaMalloc(&ctx->d_enc_lut, sizeof lut));
        JZ_CUDA_TRY(ctx, cudaMemcpy(ctx->d_enc_lut, lut, sizeof lut, cudaMemcpyHostToDevice));
        JZ_CUDA_TRY(ctx, cudaMalloc(&ctx->d_y_exact, 65536));
        k_build_y_exact<<<256, 256, 0, ctx->stream>>>(ctx->d_y_exact);
        JZ_CUDA_TRY(ctx, cudaGetLastError());
        JZ_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        JZ_CUDA_TRY(ctx, cudaMalloc(&ctx->d_counters, 8 * sizeof(unsigned long long)));
        JZ_CUDA_TRY(ctx, cudaMemset(ctx->d_counters, 0, 8 * sizeof(unsigned long long)));
        return JPEZYB200_OK;
    }();
    if (rc != JPEZYB200_OK) {
        jpezyb200_ctx_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return JPEZYB200_OK;
}

void jpezyb200_ctx_destroy(jpezyb200_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (cudaStream_t st : {ctx->stream, ctx->aux_stream, ctx->pipe.h2d, ctx->pipe.d2h})
        if (st) cudaStreamSynchronize(st);
    delete ctx;     // (the context's members release what they own)
}

int jpezyb200_set_option(jpezyb200_ctx* ctx, int option, int64_t value)
{
    if (!ctx) return JPEZYB200_EINVAL;
    switch (option) {
    case JPEZYB200_OPT_PAD_ONES: ctx->pad_ones = value ? 1 : 0; return JPEZYB200_OK;
    case JPEZYB200_OPT_RESTART_INTERVAL:
        if (value < 0 || value > 65535) return ctx->fail(JPEZYB200_EINVAL, "restart interval: 0 (none) or 1..65535 MCUs");
        ctx->restart_interval = uint32_t(value);
        return JPEZYB200_OK;
    case JPEZYB200_OPT_TRANSFORM:
        if (value != 0 && value != 1) return ctx->fail(JPEZYB200_EINVAL, "transform: 0 (production kernels) or 1 (FP64 validation kernels)");
        ctx->fp64_transforms = value == 1;
        return JPEZYB200_OK;
    case JPEZYB200_OPT_BATCH_GROUP_BYTES:
        if (value < 1) return ctx->fail(JPEZYB200_EINVAL, "group bytes must be positive");
        ctx->group_bytes = value;
        return JPEZYB200_OK;
    case JPEZYB200_OPT_SHARD_SCRATCH_BYTES:
        if (value < 0) return ctx->fail(JPEZYB200_EINVAL, "scratch bytes must be >= 0");
        ctx->shard_scratch = value;
        return JPEZYB200_OK;
    case JPEZYB200_OPT_SYNC_GUESSES:
        if (value < 0 || value > 2) return ctx->fail(JPEZYB200_EINVAL, "sync guesses: 0 (one per subsequence), 1 (one per block position on latency-bound inputs), 2 (always)");
        ctx->sync_guesses = int(value);
        return JPEZYB200_OK;
    case JPEZYB200_OPT_SYNC_ROUNDS:
        if (value < 0 || value > 64) return ctx->fail(JPEZYB200_EINVAL, "sync rounds must be in 0..64");
        ctx->sync_rounds = int(value);
        return JPEZYB200_OK;
    default: return ctx->fail(JPEZYB200_EINVAL, "unknown option");
    }
}

int jpezyb200_get_stat(jpezyb200_ctx* ctx, int stat, uint64_t* value)
{
    if (!ctx || !value) return JPEZYB200_EINVAL;
    if (stat == JPEZYB200_STAT_KERNEL_LAUNCHES) {
        *value = ctx->launches;
        return JPEZYB200_OK;
    }
    int idx = stat == JPEZYB200_STAT_GUARD_FWD ? 0 : stat == JPEZYB200_STAT_GUARD_INV ? 1 : stat == JPEZYB200_STAT_SYNC_ROUNDS ? 2 :
              stat == JPEZYB200_STAT_SYNC_ITERS0 ? 4 : stat == JPEZYB200_STAT_SYNC_ITERS1 ? 5 : -1;
    if (idx < 0) return ctx->fail(JPEZYB200_EINVAL, "unknown stat");
    JZ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    unsigned long long v = 0;
    JZ_CUDA_TRY(ctx, cudaMemcpy(&v, ctx->d_counters + idx, sizeof v, cudaMemcpyDeviceToHost));
    *value = v;
    return JPEZYB200_OK;
}

// -------------------------------------------------------------------------------------------------
// encoder
// -------------------------------------------------------------------------------------------------
static int check_geometry(jpezyb200_ctx* ctx, uint32_t W, uint32_t H, uint32_t nimg)
{
    if (!ctx) return JPEZYB200_EINVAL;
    // SOF0 carries 16-bit sizes (src/encoder/jpezy_writer.hpp:70-71)
    if (W == 0 || H == 0 || W > 65535u || H > 65535u) return ctx->fail(JPEZYB200_EINVAL, "width/height must be in 1..65535");
    if (nimg == 0 || nimg > 65535u) return ctx->fail(JPEZYB200_EINVAL, "nimg must be in 1..65535");
    return JPEZYB200_OK;
}

// picks the forward-transform kernel (JPEZYB200_OPT_TRANSFORM) and launches it
static int launch_fwd_kernel(jpezyb200_ctx* ctx, const FwdParams& p, uint32_t nimg, cudaStream_t st)
{
    if (ctx->fp64_transforms) {
        dim3 grid((p.HU + kMcuPerCta - 1) / kMcuPerCta, p.VU, nimg);
        k_fwd_transform_f64<<<grid, kFwdThreads, 0, st>>>(p);
    } else {
        (void)jz_launch(k_fwd_transform, dim3((p.HU + kTileMcu - 1) / kTileMcu, p.VU, nimg), dim3(256), kFwdTrSmem, st, p);
    }
    ++ctx->launches;
    JZ_CUDA_TRY(ctx, cudaGetLastError());
    return JPEZYB200_OK;
}

static int launch_fwd(jpezyb200_ctx* ctx, const uint8_t* d_r, const uint8_t* d_g, const uint8_t* d_b, uint32_t W, uint32_t H,
                      uint32_t nimg, int gray, int16_t* d_coefs, cudaStream_t st, bool with_meta = false)
{
    FwdParams p{};
    p.r = d_r, p.g = d_g, p.b = d_b;
    p.plane_stride = size_t(W) * H;
    p.W = W, p.H = H;
    p.HU = mcu_units(W), p.VU = mcu_units(H);
    p.coefs = d_coefs;
    p.coef_stride = size_t(p.HU) * p.VU * 384;
    p.row0 = 0, p.y_origin = 0;
    p.gray = gray;
    p.guard_counter = ctx->d_counters + 0;
    p.y_exact = ctx->d_y_exact;
    if (with_meta && !ctx->fp64_transforms) {     // side information for launch_entropy (same context, same images)
        int rc;
        if ((rc = ctx->ensure(ctx->blk_meta, size_t(nimg) * (p.coef_stride >> 6) * 4))) return rc;
        p.bmeta = static_cast<uint32_t*>(ctx->blk_meta.p);
    }
    return launch_fwd_kernel(ctx, p, nimg, st);
}

static size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// the entropy coder's scratch for nimg images of p.nblk blocks, p.ntile tiles, p.uslot un-stuffed bytes and p.nchunk
// stuffing chunks each, and of r->nint restart intervals when r is given; sets p's (and r's) pointers to it
static int ensure_entropy_scratch(jpezyb200_ctx* ctx, EntParams& p, uint32_t nimg, RstParams* r = nullptr)
{
    int rc;
    if (r) {
        if ((rc = ctx->ensure(ctx->rst_base, size_t(nimg) * (size_t(r->nint) + 1) * 8))) return rc;
        r->base = static_cast<uint64_t*>(ctx->rst_base.p);
    }
    if ((rc = ctx->ensure(ctx->blk_off, size_t(nimg) * p.nblk * 4))) return rc;
    if ((rc = ctx->ensure(ctx->tile_sum, size_t(nimg) * p.ntile * 4))) return rc;
    if ((rc = ctx->ensure(ctx->tile_base, size_t(nimg) * p.ntile * 8))) return rc;
    if ((rc = ctx->ensure(ctx->img_bits, size_t(nimg) * 16))) return rc;
    if ((rc = ctx->ensure(ctx->ustream, size_t(nimg) * p.uslot))) return rc;
    if ((rc = ctx->ensure(ctx->ff_sum, size_t(nimg) * p.nchunk * 4))) return rc;
    if ((rc = ctx->ensure(ctx->ff_base, size_t(nimg) * p.nchunk * 8))) return rc;
    p.blk_off = static_cast<uint32_t*>(ctx->blk_off.p);
    p.tile_sum = static_cast<uint32_t*>(ctx->tile_sum.p);
    p.tile_base = static_cast<uint64_t*>(ctx->tile_base.p);
    p.img_bits = static_cast<uint64_t*>(ctx->img_bits.p);
    p.img_bytes = p.img_bits + nimg;
    p.ustream = static_cast<uint8_t*>(ctx->ustream.p);
    p.ff_sum = static_cast<uint32_t*>(ctx->ff_sum.p);
    p.ff_base = static_cast<uint64_t*>(ctx->ff_base.p);
    return JPEZYB200_OK;
}

// d_ht != nullptr: code every image with its own optimised tables (enc_huffopt.cuh) and write them to d_ht[nimg][2][2]
static int launch_entropy(jpezyb200_ctx* ctx, const int16_t* d_coefs, uint32_t W, uint32_t H, uint32_t nimg, uint8_t* d_scan,
                          size_t slot_bytes, uint64_t* d_scan_bytes, uint64_t* d_scan_bits, cudaStream_t st, bool with_meta = false,
                          jpezyb200_huff* d_ht = nullptr)
{
    const uint32_t HU = mcu_units(W), VU = mcu_units(H);
    const size_t nmcu = size_t(HU) * VU;
    if (nmcu * 6 > 0xffffff00ull) return ctx->fail(JPEZYB200_EINVAL, "too many blocks");
    EntParams p{};
    p.coefs = d_coefs;
    p.coef_stride = nmcu * 384;
    p.bmeta = with_meta && !ctx->fp64_transforms ? static_cast<const uint32_t*>(ctx->blk_meta.p) : nullptr;
    p.nblk = uint32_t(nmcu * 6);
    p.ntile = (p.nblk + kEntThreads - 1) / kEntThreads;
    p.uslot = round_up(slot_bytes + 64, 16);
    p.nchunk = uint32_t((p.uslot + kStuffChunk - 1) / kStuffChunk) + 1;
    p.slot = slot_bytes;
    p.out = d_scan;
    p.out_bytes = d_scan_bytes, p.out_bits = d_scan_bits;
    p.lut = ctx->d_enc_lut;
    p.dc_init = nullptr;
    p.pad_ones = ctx->pad_ones;
    RstParams r{};
    r.rst = ctx->restart_interval;
    r.nint = r.rst ? uint32_t((nmcu + r.rst - 1) / r.rst) : 0;
    const bool rst = r.rst != 0;
    int rc;
    if ((rc = ensure_entropy_scratch(ctx, p, nimg, rst ? &r : nullptr))) return rc;
    if (d_ht) {
        const size_t hist_bytes = size_t(nimg) * 2 * kHistBins * sizeof(unsigned long long);
        const bool fresh = hist_bytes > ctx->sym_hist.cap;
        if ((rc = ctx->ensure(ctx->sym_hist, hist_bytes))) return rc;
        if (fresh) JZ_CUDA_TRY(ctx, cudaMemsetAsync(ctx->sym_hist.p, 0, ctx->sym_hist.cap, st));   // k_huff_build keeps it zeroed
        if ((rc = ctx->ensure(ctx->huff_lut, size_t(nimg) * 2 * sizeof(HuffEncLut)))) return rc;
        unsigned long long* counts = static_cast<unsigned long long*>(ctx->sym_hist.p);
        HuffEncLut* lut = static_cast<HuffEncLut*>(ctx->huff_lut.p);
        (void)jz_launch(rst ? k_sym_hist<true> : k_sym_hist<false>, dim3(p.ntile, nimg), dim3(kEntThreads), 0, st, p, counts, r);
        (void)jz_launch(k_huff_build, dim3(nimg), dim3(128), 0, st, counts, lut, d_ht);
        ctx->launches += 2;
        p.lut = lut;
        p.lut_stride = 2;
    }
    (void)jz_launch(rst ? k_block_bits<true> : k_block_bits<false>, dim3(p.ntile, nimg), dim3(kEntThreads), 0, st, p, r);
    (void)jz_launch(k_scan_tiles, dim3(nimg), dim3(1024), 0, st, p);
    if (rst) {
        (void)jz_launch(k_rst_intervals, dim3(nimg), dim3(1024), 0, st, p, r);
        ++ctx->launches;
    }
    // grid-stride helpers: enough CTAs to fill the machine, split evenly over the images
    const uint32_t per_img = std::max<uint32_t>(1u, std::min<uint32_t>(p.nchunk, (uint32_t(ctx->num_sms) * 8u + nimg - 1) / nimg));
    (void)jz_launch(k_zero_ustream, dim3(per_img, nimg), dim3(256), 0, st, p);
    (void)jz_launch(rst ? k_scatter<true> : k_scatter<false>, dim3(p.ntile, nimg), dim3(kEntThreads), 0, st, p, r);
    (void)jz_launch(k_ff_count, dim3(per_img, nimg), dim3(kStuffThreads), 0, st, p);
    (void)jz_launch(rst ? k_scan_ff<true> : k_scan_ff<false>, dim3(nimg), dim3(1024), 0, st, p, r);
    (void)jz_launch(rst ? k_stuff_write<true> : k_stuff_write<false>, dim3(per_img, nimg), dim3(kStuffThreads), 0, st, p, r);
    ctx->launches += 7;
    JZ_CUDA_TRY(ctx, cudaGetLastError());
    return JPEZYB200_OK;
}

// the fused encode of nimg device images (d_ht: as launch_entropy)
static int encode_dev(jpezyb200_ctx* ctx, const uint8_t* d_r, const uint8_t* d_g, const uint8_t* d_b, uint32_t W, uint32_t H, uint32_t nimg,
                      int gray, uint8_t* d_scan, size_t slot_bytes, uint64_t* d_scan_bytes, uint64_t* d_scan_bits, cudaStream_t st,
                      jpezyb200_huff* d_ht)
{
    int rc;
    if ((rc = ctx->ensure(ctx->coefs, size_t(mcu_units(W)) * mcu_units(H) * 384 * nimg * sizeof(int16_t)))) return rc;
    int16_t* d_coefs = static_cast<int16_t*>(ctx->coefs.p);
    if ((rc = launch_fwd(ctx, d_r, d_g, d_b, W, H, nimg, gray, d_coefs, st, true))) return rc;
    return launch_entropy(ctx, d_coefs, W, H, nimg, d_scan, slot_bytes, d_scan_bytes, d_scan_bits, st, true, d_ht);
}

// the encode of one host image on the context's stream; ht != nullptr: with optimised tables, read back into ht
static int encode_host(jpezyb200_ctx* ctx, const uint8_t* r, const uint8_t* g, const uint8_t* b, uint32_t W, uint32_t H, int gray,
                       uint8_t* scan_out, size_t scan_cap, size_t* scan_bytes, uint64_t* scan_bits, jpezyb200_huff (*ht)[2])
{
    // the sizes (2 words) and the four table records side by side: one device-to-host copy before the segment's
    const size_t readback = 16 + (ht ? 4 * sizeof(jpezyb200_huff) : 0);
    const size_t npx = size_t(W) * H;
    int rc;
    if ((rc = ctx->ensure(ctx->planes_in, 3 * npx))) return rc;
    if ((rc = ctx->ensure(ctx->scan_io, scan_cap))) return rc;
    if ((rc = ctx->ensure(ctx->sizes_io, readback))) return rc;
    uint64_t* h;
    if ((rc = ctx->readback(&h))) return rc;
    uint8_t* d_in = static_cast<uint8_t*>(ctx->planes_in.p);
    uint64_t* d_sz = static_cast<uint64_t*>(ctx->sizes_io.p);
    cudaStream_t st = ctx->stream;
    // (copies and transform on one stream: bands of MCU rows whose copies overlap the transform measured slower on a 4K frame,
    // 6.23-6.49 GPix/s for 2-8 bands against 6.48 for one -- the round trip is bound by the PCIe copies)
    JZ_CUDA_TRY(ctx, cudaMemcpyAsync(d_in, r, npx, cudaMemcpyHostToDevice, st));
    JZ_CUDA_TRY(ctx, cudaMemcpyAsync(d_in + npx, g, npx, cudaMemcpyHostToDevice, st));
    JZ_CUDA_TRY(ctx, cudaMemcpyAsync(d_in + 2 * npx, b, npx, cudaMemcpyHostToDevice, st));
    if ((rc = encode_dev(ctx, d_in, d_in + npx, d_in + 2 * npx, W, H, 1, gray, static_cast<uint8_t*>(ctx->scan_io.p), scan_cap, d_sz, d_sz + 1,
                         st, ht ? reinterpret_cast<jpezyb200_huff*>(d_sz + 2) : nullptr)))
        return rc;
    JZ_CUDA_TRY(ctx, cudaMemcpyAsync(h, d_sz, readback, cudaMemcpyDeviceToHost, st));
    JZ_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (h[0] == ~0ull || h[0] > scan_cap) return ctx->fail(JPEZYB200_ECAPACITY, "entropy-coded segment does not fit in scan_cap");
    JZ_CUDA_TRY(ctx, cudaMemcpyAsync(scan_out, ctx->scan_io.p, h[0], cudaMemcpyDeviceToHost, st));
    JZ_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    if (ht) std::memcpy(&ht[0][0], h + 2, 4 * sizeof(jpezyb200_huff));
    *scan_bytes = size_t(h[0]);
    if (scan_bits) *scan_bits = h[1];
    return JPEZYB200_OK;
}

int jpezyb200_read_sizes(jpezyb200_ctx* ctx, const uint64_t* d_values, uint32_t n, uint64_t* h_out, void* stream)
{
    if (!ctx) return JPEZYB200_EINVAL;
    if (!d_values || !h_out || n == 0 || n > jpezyb200_ctx::kReadbackWords) return ctx->fail(JPEZYB200_EINVAL, "null pointer / bad count");
    JZ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    uint64_t* h;
    int rc = ctx->readback(&h);
    if (rc) return rc;
    cudaStream_t st = pick_stream(ctx, stream);
    JZ_CUDA_TRY(ctx, cudaMemcpyAsync(h, d_values, size_t(n) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    JZ_CUDA_TRY(ctx, cudaStreamSynchronize(st));
    std::memcpy(h_out, h, size_t(n) * sizeof(uint64_t));
    return JPEZYB200_OK;
}

int jpezyb200_transform_fwd_dev(jpezyb200_ctx* ctx, const uint8_t* d_r, const uint8_t* d_g, const uint8_t* d_b, uint32_t W,
                                uint32_t H, uint32_t nimg, int gray, int16_t* d_coefs, void* stream)
{
    int rc = check_geometry(ctx, W, H, nimg);
    if (rc) return rc;
    if (!d_r || !d_g || !d_b || !d_coefs) return ctx->fail(JPEZYB200_EINVAL, "null pointer");
    JZ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return launch_fwd(ctx, d_r, d_g, d_b, W, H, nimg, gray, d_coefs, pick_stream(ctx, stream));
}

int jpezyb200_entropy_encode_dev(jpezyb200_ctx* ctx, const int16_t* d_coefs, uint32_t W, uint32_t H, uint32_t nimg, int gray,
                                 uint8_t* d_scan, size_t slot_bytes, uint64_t* d_scan_bytes, uint64_t* d_scan_bits, void* stream)
{
    (void)gray;
    int rc = check_geometry(ctx, W, H, nimg);
    if (rc) return rc;
    if (!d_coefs || !d_scan || slot_bytes == 0) return ctx->fail(JPEZYB200_EINVAL, "null pointer / empty slot");
    JZ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return launch_entropy(ctx, d_coefs, W, H, nimg, d_scan, slot_bytes, d_scan_bytes, d_scan_bits, pick_stream(ctx, stream));
}

int jpezyb200_entropy_encode_optimized_dev(jpezyb200_ctx* ctx, const int16_t* d_coefs, uint32_t W, uint32_t H, uint32_t nimg, int gray,
                                           uint8_t* d_scan, size_t slot_bytes, uint64_t* d_scan_bytes, uint64_t* d_scan_bits,
                                           jpezyb200_huff* d_ht, void* stream)
{
    (void)gray;
    int rc = check_geometry(ctx, W, H, nimg);
    if (rc) return rc;
    if (!d_coefs || !d_scan || !d_ht || slot_bytes == 0) return ctx->fail(JPEZYB200_EINVAL, "null pointer / empty slot");
    JZ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return launch_entropy(ctx, d_coefs, W, H, nimg, d_scan, slot_bytes, d_scan_bytes, d_scan_bits, pick_stream(ctx, stream), false, d_ht);
}

int jpezyb200_encode_batch_dev(jpezyb200_ctx* ctx, const uint8_t* d_r, const uint8_t* d_g, const uint8_t* d_b, uint32_t W,
                               uint32_t H, uint32_t nimg, int gray, uint8_t* d_scan, size_t slot_bytes, uint64_t* d_scan_bytes,
                               uint64_t* d_scan_bits, void* stream)
{
    int rc = check_geometry(ctx, W, H, nimg);
    if (rc) return rc;
    if (!d_r || !d_g || !d_b || !d_scan || slot_bytes == 0) return ctx->fail(JPEZYB200_EINVAL, "null pointer / empty slot");
    JZ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return encode_dev(ctx, d_r, d_g, d_b, W, H, nimg, gray, d_scan, slot_bytes, d_scan_bytes, d_scan_bits, pick_stream(ctx, stream), nullptr);
}

int jpezyb200_encode_batch_optimized_dev(jpezyb200_ctx* ctx, const uint8_t* d_r, const uint8_t* d_g, const uint8_t* d_b, uint32_t W,
                                         uint32_t H, uint32_t nimg, int gray, uint8_t* d_scan, size_t slot_bytes, uint64_t* d_scan_bytes,
                                         uint64_t* d_scan_bits, jpezyb200_huff* d_ht, void* stream)
{
    int rc = check_geometry(ctx, W, H, nimg);
    if (rc) return rc;
    if (!d_r || !d_g || !d_b || !d_scan || !d_ht || slot_bytes == 0) return ctx->fail(JPEZYB200_EINVAL, "null pointer / empty slot");
    JZ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return encode_dev(ctx, d_r, d_g, d_b, W, H, nimg, gray, d_scan, slot_bytes, d_scan_bytes, d_scan_bits, pick_stream(ctx, stream), d_ht);
}

int jpezyb200_encode(jpezyb200_ctx* ctx, const uint8_t* r, const uint8_t* g, const uint8_t* b, uint32_t W, uint32_t H, int gray,
                     uint8_t* scan_out, size_t scan_cap, size_t* scan_bytes, uint64_t* scan_bits)
{
    int rc = check_geometry(ctx, W, H, 1);
    if (rc) return rc;
    if (!r || !g || !b || !scan_out || !scan_bytes || scan_cap == 0) return ctx->fail(JPEZYB200_EINVAL, "null pointer / empty buffer");
    JZ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return encode_host(ctx, r, g, b, W, H, gray, scan_out, scan_cap, scan_bytes, scan_bits, nullptr);
}

int jpezyb200_encode_optimized(jpezyb200_ctx* ctx, const uint8_t* r, const uint8_t* g, const uint8_t* b, uint32_t W, uint32_t H, int gray,
                               uint8_t* scan_out, size_t scan_cap, size_t* scan_bytes, uint64_t* scan_bits, jpezyb200_huff ht[2][2])
{
    int rc = check_geometry(ctx, W, H, 1);
    if (rc) return rc;
    if (!r || !g || !b || !scan_out || !scan_bytes || !ht || scan_cap == 0) return ctx->fail(JPEZYB200_EINVAL, "null pointer / empty buffer");
    JZ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return encode_host(ctx, r, g, b, W, H, gray, scan_out, scan_cap, scan_bytes, scan_bits, ht);
}

// -------------------------------------------------------------------------------------------------
// synthetic input
// -------------------------------------------------------------------------------------------------
int jpezyb200_synth_dev(jpezyb200_ctx* ctx, uint8_t* d_r, uint8_t* d_g, uint8_t* d_b, uint32_t W, uint32_t H, uint32_t nimg,
                        uint32_t first_frame, int family, void* stream)
{
    int rc = check_geometry(ctx, W, H, nimg);
    if (rc) return rc;
    if (!d_r || !d_g || !d_b) return ctx->fail(JPEZYB200_EINVAL, "null pointer");
    JZ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t npx = size_t(W) * H;
    const uint32_t gx = uint32_t(std::min<size_t>((npx + 255) / 256, size_t(ctx->num_sms) * 16));
    k_synth<<<dim3(gx, nimg), 256, 0, pick_stream(ctx, stream)>>>(d_r, d_g, d_b, W, H, first_frame, family, 0u);
    ++ctx->launches;
    JZ_CUDA_TRY(ctx, cudaGetLastError());
    return JPEZYB200_OK;
}

int jpezyb200_synth_rows_dev(jpezyb200_ctx* ctx, uint8_t* d_r, uint8_t* d_g, uint8_t* d_b, uint32_t W, uint32_t y0, uint32_t nrows,
                             uint32_t frame, int family, void* stream)
{
    int rc = check_geometry(ctx, W, nrows, 1);
    if (rc) return rc;
    if (!d_r || !d_g || !d_b) return ctx->fail(JPEZYB200_EINVAL, "null pointer");
    JZ_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t npx = size_t(W) * nrows;
    const uint32_t gx = uint32_t(std::min<size_t>((npx + 255) / 256, size_t(ctx->num_sms) * 16));
    k_synth<<<dim3(gx, 1), 256, 0, pick_stream(ctx, stream)>>>(d_r, d_g, d_b, W, nrows, frame, family, y0);
    ++ctx->launches;
    JZ_CUDA_TRY(ctx, cudaGetLastError());
    return JPEZYB200_OK;
}

}  // extern "C"

#include "capi_decode.inc"
#include "capi_shard.inc"
#include "capi_batch.inc"
#include "capi_group.inc"
