// dec_transform_g.cuh -- stages D2+D3 for the frame layouts jpezy's own encoder never writes but its decoder accepts
// (1 or 3 components, luma sampling 1x1 / 2x1 / 1x2, chroma 1x1: 4:4:4, 4:2:2, 4:4:0, single-component gray).
//
// Replaces inverse_quantization (src/decoder/jpezy_decoder.hpp:645-650), inverse_dct (:652-670), the pixel replication of
// decode_mcu (:519-524) and make_rgb / to_r,g,b / revise_value (:531-578, :672-676) like the kernels of dec_transform2.cuh,
// which are specialised for 2x2 / 1x1 / 1x1.  Round 1 sent these layouts through the FP64 validation kernel
// (k_inv_transform_f64): 500-630 us for a 3840x2160 frame against 35 us for 4:2:0.  Two kernels here:
//
//  * k_idct_blocks: the block pipeline of k_inv_transform2 -- eight lanes per block PAIR, packed f32x2 AAN flowgraphs, floor by
//    FADD2.RM, per-block guard band, DC-only blocks in the reference's order, FP64 fix-up queue with the exact-order tier --
//    over the image's blocks in scan order, whatever component they belong to: a pair is two consecutive blocks, its constants
//    come from the table of its (component A, component B) class.  The 8x8 samples of every block go to a scratch array
//    (int16, 128 bytes per block, scan order).  A block with a sample outside the int16 range (kWideSample) is written as
//    kWideMark in every sample instead: k_colour_general recomputes its pixels from the coefficients.
//  * k_colour_general: one thread per 8 pixels of a row: gathers the Y, Cb, Cr samples through the MCU geometry (replication =
//    index arithmetic), evaluates the reference's FP64 expressions (40 TFLOP/s of FP64 make that 8 us for a 4K frame), stores
//    8 bytes per plane.
// Numerics: as dec_transform2.cuh (same flowgraphs, same guard band, same tiers).  Decoded samples identical to the reference
// decoder's (tests/test_general_decode_gpu.py).
#pragma once
#include "dec_transform2.cuh"

namespace jz {

// constants per (component of block A, component of block B) class c = 3 A + B
struct InvGTab {
    float2 M[9][8][8];     // [class][u][v]
    float2 Wg[9][8][8];
    uint2 zoff[8];
};

__global__ void k_build_invg_tab(const InvParams p, InvGTab* __restrict__ tab)
{
    pdl_wait();
    const int t = threadIdx.x;      // 576 threads: class, natural position
    const int c = t >> 6, nat = t & 63, v = nat >> 3, u = nat & 7;
    const int ca = c / 3, cb = c % 3;
    tab->M[c][u][v] = make_float2(p.M[ca][nat], p.M[cb][nat]);
    tab->Wg[c][u][v] = make_float2(p.Wg[ca][nat], p.Wg[cb][nat]);
    if (t < 8) {
        uint32_t w[2] = {0, 0};
        for (int vv = 0; vv < 8; ++vv) w[vv >> 2] |= uint32_t(cC.izz[vv * 8 + t] * 2) << (8 * (vv & 3));
        tab->zoff[t] = make_uint2(w[0], w[1]);
    }
}

constexpr int kGBlk = 48;                       // blocks per CTA
constexpr int16_t kWideMark = -32768;           // every sample of a block whose samples leave the int16 range (never a sample otherwise)
constexpr int kGThreads = kGBlk * 4;            // eight lanes per pair
struct InvG {
    static constexpr int kCoef = kGBlk * 128;
    static constexpr int kPairRow = 80, kPair = 8 * kPairRow + 64;
    static constexpr int kMid = (kGBlk / 2) * kPair;
    static constexpr int kSmp = kGBlk * 128;
    static constexpr int kSmem = kCoef + kMid + kSmp + kFixCap * 2 + 16 + kGBlk + 16;
};

// blocks [blk_lo, blk_hi) of every image (scan order; a shard of MCU rows is a contiguous range); samples: [nimg][nblk][64] int16
__global__ void __launch_bounds__(kGThreads, 5) k_idct_blocks(const __grid_constant__ InvParams p, const InvGTab* __restrict__ tab,
                                                              int16_t* __restrict__ samples, const uint32_t blk_lo, const uint32_t blk_hi)
{
    using C = InvG;
    extern __shared__ __align__(16) uint8_t smem[];
    uint8_t* s_coef = smem;                                  // [kGBlk][64] int16, zig-zag
    uint8_t* s_mid = s_coef + C::kCoef;                      // [kGBlk / 2 pairs][8][kPairRow] transpose scratch
    uint8_t* s_smp = s_mid + C::kMid;                        // [kGBlk][64] int16 samples, row-major
    uint16_t* s_fix = reinterpret_cast<uint16_t*>(s_smp + C::kSmp);
    uint32_t* s_nfix = reinterpret_cast<uint32_t*>(s_fix + kFixCap);
    const uint32_t bar = smem_u32(s_nfix + 2);
    uint8_t* s_mask = reinterpret_cast<uint8_t*>(s_nfix + 4);    // [kGBlk] non-zero zig-zag groups of every block
    unsigned long long* s_wide = reinterpret_cast<unsigned long long*>(s_mask + kGBlk);     // blocks with samples outside int16

    const int t = threadIdx.x, lane = t & 31;
    const size_t img = blockIdx.y;
    const uint32_t blk0 = blk_lo + blockIdx.x * kGBlk;
    const uint32_t nvalid = min(uint32_t(kGBlk), blk_hi - blk0);
    if (t == 0) {
        mbar_init(bar, 1);
        *s_nfix = 0;
        *s_wide = 0;
        mbar_fence_init();
    }
    __syncthreads();
    pdl_wait();
    if (t == 0) {
        mbar_expect_tx(bar, nvalid * 128u);
        bulk_g2s(smem_u32(s_coef), p.coefs + img * p.coef_stride + size_t(blk0) * 64, nvalid * 128u, bar);
    }
    const uint32_t pr = uint32_t(t) >> 3, sub = uint32_t(t) & 7u;
    const uint32_t blkA = 2u * pr, blkB = blkA + 1u;
    const bool validA = blkA < nvalid, validB = blkB < nvalid;
    const uint32_t kA = (blk0 + blkA) % p.nb, kB = (blk0 + blkB) % p.nb;
    const int compA = kA < p.ny ? 0 : int(kA - p.ny) + 1, compB = kB < p.ny ? 0 : int(kB - p.ny) + 1;
    const int cls = compA * 3 + compB;
    uint8_t* mid = s_mid + pr * C::kPair;
    mbar_wait_wd(bar, 0);

    {
        const uint8_t* cA = s_coef + blkA * 128u;
        constexpr uint32_t dAB = 128u;
        uint4 gA = make_uint4(0, 0, 0, 0), gB = gA;
        if (validA) gA = *reinterpret_cast<const uint4*>(cA + sub * 16u);
        if (validB) gB = *reinterpret_cast<const uint4*>(cA + dAB + sub * 16u);
        int dcA = 0, dcB = 0;
        if (sub == 0) {
            dcA = int(short(gA.x & 0xffffu)), dcB = int(short(gB.x & 0xffffu));
            gA.x &= 0xffff0000u, gB.x &= 0xffff0000u;
        }
        const uint32_t balA = __ballot_sync(0xffffffffu, (gA.x | gA.y | gA.z | gA.w) != 0u);
        const uint32_t balB = __ballot_sync(0xffffffffu, (gB.x | gB.y | gB.z | gB.w) != 0u);
        const uint32_t maskA = (balA >> (lane & 24)) & 0xffu, maskB = (balB >> (lane & 24)) & 0xffu;
        if (sub == 0) {
            if (validA) s_mask[blkA] = uint8_t(maskA);
            if (validB) s_mask[blkB] = uint8_t(maskB);
        }
        const int qA = int(p.qt[compA][0]), qB = int(p.qt[compB][0]);
        dcA = __shfl_sync(0xffffffffu, dcA, lane & 24), dcB = __shfl_sync(0xffffffffu, dcB, lane & 24);

        uint4 rowA, rowB;         // the 8 + 8 samples of row sub as int16 pairs
        bool wideA, wideB;        // a sample of this row leaves the int16 range
        if ((balA | balB) == 0u) {
            // every block of the warp is DC-only
            const int ia = dc_only_value(dcA, qA), ib = dc_only_value(dcB, qB);
            const uint32_t va = uint32_t(ia) & 0xffffu, vb = uint32_t(ib) & 0xffffu;
            rowA = make_uint4(va * 0x10001u, va * 0x10001u, va * 0x10001u, va * 0x10001u);
            rowB = make_uint4(vb * 0x10001u, vb * 0x10001u, vb * 0x10001u, vb * 0x10001u);
            wideA = wide_int(ia), wideB = wide_int(ib);
            if (lane == 0) atomicAdd(p.guard_counter, 32ull * 16ull);
        } else {
            const bool pruned = ((balA | balB) & 0xfefefefeu) == 0u;      // nothing beyond zig-zag position 7 in the warp
            const uint32_t u = sub;
            f32x2 d[8];
            f32x2 gs = pk2(0.0f, 0.0f);
            {
                const uint2 zo = __ldg(&tab->zoff[u]);
                const ulonglong2* mq = reinterpret_cast<const ulonglong2*>(&tab->M[cls][u][0]);
                const ulonglong2* wq = reinterpret_cast<const ulonglong2*>(&tab->Wg[cls][u][0]);
                const uint32_t base = smem_u32(cA);
#define JZ_LOAD_COEF(V, ZW, K, MM, WW)                                                                                   \
    {                                                                                                                     \
        const uint32_t ad = add_byte<K>(ZW, base);                                                                        \
        int ca, cb;                                                                                                       \
        asm volatile("ld.shared.s16 %0, [%1];" : "=r"(ca) : "r"(ad));                                                     \
        asm volatile("ld.shared.s16 %0, [%1];" : "=r"(cb) : "r"(ad + dAB));                                               \
        const f32x2 f = pk2(float(ca), float(cb));                                                                        \
        d[V] = mul2(f, MM);                                                                                               \
        const f32x2 g = mul2(f, WW);                                                                                      \
        gs = add2(gs, pk2(fabsf(lo2(g)), fabsf(hi2(g))));                                                                 \
    }
                const ulonglong2 m01 = __ldg(mq), m23 = __ldg(mq + 1), w01 = __ldg(wq), w23 = __ldg(wq + 1);
                JZ_LOAD_COEF(0, zo.x, 0, m01.x, w01.x)
                JZ_LOAD_COEF(1, zo.x, 1, m01.y, w01.y)
                JZ_LOAD_COEF(2, zo.x, 2, m23.x, w23.x)
                if (pruned) {
                    d[3] = d[4] = d[5] = d[6] = d[7] = pk2(0.0f, 0.0f);
                } else {
                    const ulonglong2 m45 = __ldg(mq + 2), m67 = __ldg(mq + 3), w45 = __ldg(wq + 2), w67 = __ldg(wq + 3);
                    JZ_LOAD_COEF(3, zo.x, 3, m23.y, w23.y)
                    JZ_LOAD_COEF(4, zo.y, 0, m45.x, w45.x)
                    JZ_LOAD_COEF(5, zo.y, 1, m45.y, w45.y)
                    JZ_LOAD_COEF(6, zo.y, 2, m67.x, w67.x)
                    JZ_LOAD_COEF(7, zo.y, 3, m67.y, w67.y)
                }
#undef JZ_LOAD_COEF
            }
            // (an absent block B reads the bytes behind the tile's last block: whatever they are, its samples are never stored)
            if (u == 0) d[0] = add2(d[0], pk2(128.0f, 128.0f));       // level shift rides on the DC term
            if (pruned) aan_idct8_in3_x2(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);
            else aan_idct8_x2(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);
#pragma unroll
            for (int y = 0; y < 8; ++y) *reinterpret_cast<f32x2*>(mid + y * C::kPairRow + u * 8u) = d[y];
            {
                float ga = lo2(gs), gb = hi2(gs);
                ga += __shfl_xor_sync(0xffffffffu, ga, 1), gb += __shfl_xor_sync(0xffffffffu, gb, 1);
                ga += __shfl_xor_sync(0xffffffffu, ga, 2), gb += __shfl_xor_sync(0xffffffffu, gb, 2);
                ga += __shfl_xor_sync(0xffffffffu, ga, 4), gb += __shfl_xor_sync(0xffffffffu, gb, 4);
                gs = pk2(ga + 2e-5f, gb + 2e-5f);
            }
            __syncwarp();
            {
                const ulonglong2* src = reinterpret_cast<const ulonglong2*>(mid + sub * C::kPairRow);
                const ulonglong2 a = src[0], b = src[1], c = src[2], e = src[3];
                d[0] = a.x, d[1] = a.y, d[2] = b.x, d[3] = b.y, d[4] = c.x, d[5] = c.y, d[6] = e.x, d[7] = e.y;
            }
            if (pruned) aan_idct8_in4_x2(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);
            else aan_idct8_x2(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);
            const f32x2 mg = pk2(kMagic15, kMagic15);
            uint32_t ia[8], ib[8];
            float ma = 1.0f, mb = 1.0f, va = 0.0f, vb = 0.0f;
#pragma unroll
            for (int x = 0; x < 8; x += 2) {
                const f32x2 f0 = add2_rm(d[x], mg), f1 = add2_rm(d[x + 1], mg);
                ia[x] = uint32_t(f0), ib[x] = uint32_t(f0 >> 32), ia[x + 1] = uint32_t(f1), ib[x + 1] = uint32_t(f1 >> 32);
                const f32x2 e0 = sub2(d[x], sub2(add2(d[x], mg), mg)), e1 = sub2(d[x + 1], sub2(add2(d[x + 1], mg), mg));
                ma = fmin3_abs(lo2(e0), lo2(e1), ma), mb = fmin3_abs(hi2(e0), hi2(e1), mb);
                va = fmax3_abs(lo2(d[x]), lo2(d[x + 1]), va), vb = fmax3_abs(hi2(d[x]), hi2(d[x + 1]), vb);
            }
            wideA = va >= kWideSample, wideB = vb >= kWideSample;
            rowA = make_uint4(__byte_perm(ia[0], ia[1], 0x5410), __byte_perm(ia[2], ia[3], 0x5410), __byte_perm(ia[4], ia[5], 0x5410), __byte_perm(ia[6], ia[7], 0x5410));
            rowB = make_uint4(__byte_perm(ib[0], ib[1], 0x5410), __byte_perm(ib[2], ib[3], 0x5410), __byte_perm(ib[4], ib[5], 0x5410), __byte_perm(ib[6], ib[7], 0x5410));
            const bool dcoA = maskA == 0u, dcoB = maskB == 0u;
            const bool negA = ((rowA.x | rowA.y | rowA.z | rowA.w) & 0x80008000u) != 0u, negB = ((rowB.x | rowB.y | rowB.z | rowB.w) & 0x80008000u) != 0u;
            uint32_t exact = 0;
            if (dcoA) {
                const uint32_t va = uint32_t(dc_only_value(dcA, qA)) & 0xffffu;
                rowA = make_uint4(va * 0x10001u, va * 0x10001u, va * 0x10001u, va * 0x10001u);
                exact += 8;
            } else if ((ma < lo2(gs) || negA) && validA) {
                rowA = inv_row_slow(lo2(d[0]), lo2(d[1]), lo2(d[2]), lo2(d[3]), lo2(d[4]), lo2(d[5]), lo2(d[6]), lo2(d[7]), lo2(gs), blkA, int(sub), s_nfix, s_fix);
            }
            if (dcoB) {
                const uint32_t vb = uint32_t(dc_only_value(dcB, qB)) & 0xffffu;
                rowB = make_uint4(vb * 0x10001u, vb * 0x10001u, vb * 0x10001u, vb * 0x10001u);
                exact += 8;
            } else if ((mb < hi2(gs) || negB) && validB) {
                rowB = inv_row_slow(hi2(d[0]), hi2(d[1]), hi2(d[2]), hi2(d[3]), hi2(d[4]), hi2(d[5]), hi2(d[6]), hi2(d[7]), hi2(gs), blkB, int(sub), s_nfix, s_fix);
            }
            exact = __reduce_add_sync(0xffffffffu, exact);
            if (lane == 0 && exact) atomicAdd(p.guard_counter, (unsigned long long)exact);
        }
        if (validA) *reinterpret_cast<uint4*>(s_smp + blkA * 128u + sub * 16u) = rowA;
        if (validB) *reinterpret_cast<uint4*>(s_smp + blkB * 128u + sub * 16u) = rowB;
        if ((wideA && validA) || (wideB && validB)) atomicOr(s_wide, (wideA && validA ? 1ull << blkA : 0ull) | (wideB && validB ? 1ull << blkB : 0ull));
    }
    __syncthreads();

    // ---- FP64 re-evaluation of the queue (guard-band samples) ----
    {
        const uint32_t nfix = *s_nfix;
        if (nfix) {
            const bool overflow = nfix > kFixCap;
            uint32_t exact_hits = 0;
            const uint32_t ntask = overflow ? nvalid * 8u : nfix * 8u;
            for (uint32_t task0 = 0; task0 < ntask; task0 += kGThreads) {
                const uint32_t task = task0 + uint32_t(t);
                // entry = blk << 7 | sample; overflow: row (task & 7) of block (task >> 3), every sample
                const uint32_t e = task >= ntask ? 0u : (overflow ? ((task >> 3) << 7) : uint32_t(s_fix[task >> 3]));
                const uint32_t blk = e >> 7, s8 = task & 7u;
                const uint32_t k = (blk0 + blk) % p.nb;
                const bool act = task < ntask;
                const int comp = k < p.ny ? 0 : int(k - p.ny) + 1;
                const int16_t* cz = reinterpret_cast<const int16_t*>(s_coef + blk * 128u);
                const int nlim = 8 * (32 - __clz(uint32_t(s_mask[blk]) | 1u));
                int16_t* smp = reinterpret_cast<int16_t*>(s_smp + blk * 128u);
                if (overflow) {
                    if (act)
                        for (int x = 0; x < 8; ++x) smp[s8 * 8 + x] = int16_t(idct_fix(cz, p.qt[comp], nlim, x, int(s8), &exact_hits));
                } else {
                    const int s = int(e & 63u);
                    double part = act ? idct_fix_part(cz, p.qt[comp], int(s8), 8, nlim, s & 7, s >> 3) : 0.0;
                    part += __shfl_xor_sync(0xffffffffu, part, 1);
                    part += __shfl_xor_sync(0xffffffffu, part, 2);
                    part += __shfl_xor_sync(0xffffffffu, part, 4);
                    if (act && s8 == 0) smp[s] = int16_t(idct_fix_finish(part, cz, p.qt[comp], nlim, s & 7, s >> 3, &exact_hits));
                }
            }
            exact_hits = __reduce_add_sync(0xffffffffu, exact_hits);
            if (lane == 0 && exact_hits) atomicAdd(p.guard_counter, (unsigned long long)exact_hits);
            __syncthreads();
        }
    }
    // ---- the samples leave, 16 bytes per thread and round ----
    uint4* dst = reinterpret_cast<uint4*>(samples + (img * (p.coef_stride >> 6) + blk0) * 64);
    const unsigned long long wide = *s_wide;
    constexpr uint32_t kMark2 = uint32_t(uint16_t(kWideMark)) * 0x10001u;
    for (uint32_t i = t; i < nvalid * 8u; i += kGThreads)
        dst[i] = (wide >> (i >> 3)) & 1ull ? make_uint4(kMark2, kMark2, kMark2, kMark2) : reinterpret_cast<const uint4*>(s_smp)[i];
}

// one thread per 8 pixels of a row of MCU rows [row0, row0 + rows).  The 8 pixels lie in one MCU and, per component, in one row of
// one block: 8 samples (factor 1) or 4 samples, each used twice (factor 2) -- one 16- or 8-byte load per component.
__device__ __forceinline__ void load_samples8(const int16_t* __restrict__ smp, size_t blk, uint32_t row, uint32_t px0, uint32_t dx, int (&v)[8])
{
    const uint32_t sx = px0 / dx;                         // first sample column: 0 (dx == 1), 0 or 4 (dx == 2)
    const int16_t* src = smp + (blk + (sx >> 3)) * 64 + row * 8 + (sx & 7u);
    if (dx == 1u) {
        const uint4 w = *reinterpret_cast<const uint4*>(src);
        v[0] = sx_lo(w.x), v[1] = sx_hi(w.x), v[2] = sx_lo(w.y), v[3] = sx_hi(w.y), v[4] = sx_lo(w.z), v[5] = sx_hi(w.z), v[6] = sx_lo(w.w), v[7] = sx_hi(w.w);
    } else {
        const uint2 w = *reinterpret_cast<const uint2*>(src);
        v[0] = v[1] = sx_lo(w.x), v[2] = v[3] = sx_hi(w.x), v[4] = v[5] = sx_lo(w.y), v[6] = v[7] = sx_hi(w.y);
    }
}

// the 8 pixels of k_colour_general, every sample by sample_ref from the coefficients (blocks marked kWideMark)
__device__ __noinline__ void colour_general_ref(const InvParams& p, size_t img, size_t mcu, uint32_t ry, uint32_t px0, uint32_t gx0, size_t idx)
{
    const int16_t* cz = p.coefs + img * p.coef_stride;
    for (uint32_t i = 0; i < 8 && gx0 + i < p.W; ++i) {
        const uint32_t px = px0 + i;
        int v[3] = {0, 128, 128};          // comp tiles of absent components stay 0x80 (src/decoder/jpezy_decoder.hpp:105)
        const int nc = (p.ncomp == 3 && !p.gray) ? 3 : 1;
        size_t first = mcu;
        for (int c = 0; c < nc; ++c) {
            const uint32_t sx = px / (p.hmax / p.hs[c]), sy = ry / (p.vmax / p.vs[c]);
            v[c] = sample_ref(cz + (first + (sy >> 3) * p.hs[c] + (sx >> 3)) * 64, p.qt[c], int(sx & 7u), int(sy & 7u));
            first += p.hs[c] * p.vs[c];
        }
        uint8_t* R = p.r + img * p.plane_stride + idx + i;
        uint8_t* G = p.g + img * p.plane_stride + idx + i;
        uint8_t* B = p.b + img * p.plane_stride + idx + i;
        if (p.gray) *R = *G = *B = revise(double(v[0]));
        else *R = ref_R(v[0], v[2]), *G = ref_G(v[0], v[1], v[2]), *B = ref_B(v[0], v[1]);
    }
}

__global__ void __launch_bounds__(256) k_colour_general(const __grid_constant__ InvParams p, const int16_t* __restrict__ samples, const uint32_t rows)
{
    pdl_wait();
    const size_t img = blockIdx.z;
    const uint32_t mw = 8 * p.hmax, mh = 8 * p.vmax;
    const uint32_t gx0 = (blockIdx.x * blockDim.x + threadIdx.x) * 8u;
    const uint32_t y = p.row0 * mh + blockIdx.y;                       // pixel row
    if (gx0 >= p.HU * mw || blockIdx.y >= rows * mh) return;
    const uint32_t my = y / mh, ry = y - my * mh;
    const uint32_t mx = gx0 / mw, px0 = gx0 - mx * mw;
    const size_t mcu = (size_t(my) * p.HU + mx) * p.nb;
    const int16_t* smp = samples + img * (p.coef_stride >> 6) * 64;
    const uint32_t dx0 = p.hmax / p.hs[0], dy0 = p.vmax / p.vs[0];
    int yv[8], cb[8], cr[8];
    {
        const uint32_t sy = ry / dy0;
        load_samples8(smp, mcu + (sy >> 3) * p.hs[0], sy & 7u, px0, dx0, yv);
    }
    if (p.ncomp == 3 && !p.gray) {
        const uint32_t dx1 = p.hmax / p.hs[1], dy1 = p.vmax / p.vs[1], dx2 = p.hmax / p.hs[2], dy2 = p.vmax / p.vs[2];
        const uint32_t sy1 = ry / dy1, sy2 = ry / dy2;
        load_samples8(smp, mcu + p.ny + (sy1 >> 3) * p.hs[1], sy1 & 7u, px0, dx1, cb);
        load_samples8(smp, mcu + p.ny + p.hs[1] * p.vs[1] + (sy2 >> 3) * p.hs[2], sy2 & 7u, px0, dx2, cr);
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) cb[i] = cr[i] = 128;      // comp tiles of absent components stay 0x80 (src/decoder/jpezy_decoder.hpp:105)
    }
    const size_t idx = size_t(y) * p.W + gx0;
    bool wide = false;
#pragma unroll
    for (int i = 0; i < 8; ++i) wide |= yv[i] == kWideMark || cb[i] == kWideMark || cr[i] == kWideMark;
    if (wide) {
        colour_general_ref(p, img, mcu, ry, px0, gx0, idx);
        atomicAdd(p.guard_counter, 8ull);     // (JPEZYB200_STAT_GUARD_INV: exact-order pixels)
        return;
    }
    uint32_t ro[2] = {0, 0}, go[2] = {0, 0}, bo[2] = {0, 0};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        uint32_t r, g, b;
        if (p.gray) r = g = b = revise(double(yv[i]));
        else r = ref_R(yv[i], cr[i]), g = ref_G(yv[i], cb[i], cr[i]), b = ref_B(yv[i], cb[i]);
        ro[i >> 2] |= r << (8 * (i & 3)), go[i >> 2] |= g << (8 * (i & 3)), bo[i >> 2] |= b << (8 * (i & 3));
    }
    uint8_t* R = p.r + img * p.plane_stride;
    uint8_t* G = p.g + img * p.plane_stride;
    uint8_t* B = p.b + img * p.plane_stride;
    if ((p.W & 7u) == 0 && gx0 + 8u <= p.W && ((reinterpret_cast<uintptr_t>(R) | reinterpret_cast<uintptr_t>(G) | reinterpret_cast<uintptr_t>(B) | p.plane_stride) & 7u) == 0) {
        *reinterpret_cast<uint2*>(R + idx) = make_uint2(ro[0], ro[1]);
        *reinterpret_cast<uint2*>(G + idx) = make_uint2(go[0], go[1]);
        *reinterpret_cast<uint2*>(B + idx) = make_uint2(bo[0], bo[1]);
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (gx0 + i < p.W) {
                R[idx + i] = uint8_t(ro[i >> 2] >> (8 * (i & 3)));
                G[idx + i] = uint8_t(go[i >> 2] >> (8 * (i & 3)));
                B[idx + i] = uint8_t(bo[i >> 2] >> (8 * (i & 3)));
            }
    }
}

}  // namespace jz
