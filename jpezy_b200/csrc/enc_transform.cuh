// enc_transform.cuh -- stages E1+E2: planar RGB -> quantised zig-zag int16 coefficients.
//
// Replaces make_YCC (src/encoder/jpezy_encoder.hpp:90-144), RGB::Y/Cb/Cr (:244-256), DCT (:146-166)
// and quantization (:168-172) of the reference.  One CTA transforms a strip of kMcuPerCta MCUs of
// one MCU row: colour conversion + 2:1 decimation into shared-memory MCU tiles, then the 8x8 DCTs,
// quantisation, zig-zag and a coalesced store in scan order (Y0 Y1 Y2 Y3 Cb Cr per MCU).
//
// Numerics: the reference truncates FP64 expressions, so results flip on 1-ulp differences when
// the exact value sits on a boundary.  The fast path computes the DCT with a separable transform;
// any coefficient whose value lies within kGuard of a non-zero multiple of its quantiser is
// recomputed in the reference's exact operation order (dct_exact), so the output is
// bit-identical to the reference's strict-IEEE evaluation.  Algorithmic HBM traffic: 3 B/px read
// + 3 B/px written (1.5 int16 coefficients per pixel) = 6 B/px.
#pragma once
#include "common.cuh"

namespace jz {

constexpr int kMcuPerCta = 8;                 // 128 x 16 pixels per CTA
constexpr int kBlkPerCta = kMcuPerCta * 6;    // 48 8x8 blocks
constexpr int kFwdThreads = 256;

struct FwdParams {
    const uint8_t *r, *g, *b;   // planes of image 0 (of the local rows when sharded)
    size_t plane_stride;        // bytes between consecutive images
    int16_t* coefs;
    size_t coef_stride;         // int16 elements between consecutive images
    uint32_t W, H;              // image size (H = full image height, used for edge replication)
    uint32_t HU, VU;            // MCUs per row / MCU rows handled by this launch
    uint32_t row0;              // first MCU row of this launch within the image (shards)
    uint32_t y_origin;          // image row stored at plane offset 0 (shards)
    int gray;
    unsigned long long* guard_counter;
    const int8_t* y_exact;      // [65536] correction of the exact luma cases, indexed r | g << 8 (k_build_y_exact)
    uint32_t* bmeta;            // nullptr, or per block (image stride coef_stride / 64): DC coefficient in bits 0..15, in bits
                                // 16..23 which 8-coefficient zig-zag groups hold a non-zero AC coefficient -- the entropy coder
                                // then reads only those groups of `coefs` (EntParams::bmeta)
};

// ---- colour conversion, bit-exact with src/encoder/jpezy_encoder.hpp:245-256 ------------------
// The reference evaluates left to right in double and truncates toward zero.
__device__ __forceinline__ int ref_Y(int r, int g, int b)
{
    double t = __dadd_rn(__dmul_rn(0.2990, double(r)), __dmul_rn(0.5870, double(g)));
    t = __dadd_rn(t, __dmul_rn(0.1140, double(b)));
    return __double2int_rz(__dadd_rn(t, -128.0));
}
__device__ __forceinline__ int ref_Cb(int r, int g, int b)
{
    double t = __dsub_rn(-__dmul_rn(0.1687, double(r)), __dmul_rn(0.3313, double(g)));
    return __double2int_rz(__dadd_rn(t, __dmul_rn(0.5000, double(b))));
}
__device__ __forceinline__ int ref_Cr(int r, int g, int b)
{
    double t = __dsub_rn(__dmul_rn(0.5000, double(r)), __dmul_rn(0.4187, double(g)));
    return __double2int_rz(__dsub_rn(t, __dmul_rn(0.0813, double(b))));
}

// Integer evaluation of the same formulas: the exact value is n/10000 with n integer, and the
// FP64 evaluation is within 1e-12 of it, so truncation agrees unless n is a multiple of 10000
// (exact integer result), where the FP64 rounding decides and ref_* is used instead.
__device__ __forceinline__ int fast_Y(int r, int g, int b)
{
    const int n = 2990 * r + 5870 * g + 1140 * b - 1280000;   // |n| <= 1.28e6
    const int q = n / 10000;
    return (n - q * 10000 == 0) ? ref_Y(r, g, b) : q;
}
__device__ __forceinline__ int fast_Cb(int r, int g, int b)
{
    const int n = -1687 * r - 3313 * g + 5000 * b;
    const int q = n / 10000;
    return (n - q * 10000 == 0) ? ref_Cb(r, g, b) : q;
}
__device__ __forceinline__ int fast_Cr(int r, int g, int b)
{
    const int n = 5000 * r - 4187 * g - 813 * b;
    const int q = n / 10000;
    return (n - q * 10000 == 0) ? ref_Cr(r, g, b) : q;
}

// ---- exact-order DCT of one coefficient (src/encoder/jpezy_encoder.hpp:146-166) ----------------
// F[i][j] = int( (sum_y sum_x ((pic*cos[j][x])*cos[i][y])) * cu * cv / 4 ), y outer, x inner.
__device__ __noinline__ double dct_exact(const int8_t* __restrict__ pic, int i, int j)
{
    double sum = 0.0;
    for (int y = 0; y < 8; ++y) {
        const double ci = cC.cos_ref[i * 8 + y];
#pragma unroll
        for (int x = 0; x < 8; ++x)
            sum = __dadd_rn(sum, __dmul_rn(__dmul_rn(double(pic[y * 8 + x]), cC.cos_ref[j * 8 + x]), ci));
    }
    const double cu = j ? 1.0 : cC.inv_sqrt2_ref;
    const double cv = i ? 1.0 : cC.inv_sqrt2_ref;
    return __dmul_rn(__dmul_rn(__dmul_rn(sum, cu), cv), 0.25);   // "/ 4" is exact
}

constexpr double kGuardF64 = 1e-6;   // fast-path FP64 error is < 1e-10; see DESIGN.md

// ---- validation build: FP64 separable DCT ---------------------------------------------------------
__global__ void __launch_bounds__(kFwdThreads) k_fwd_transform_f64(const FwdParams p)
{
    pdl_wait();
    __shared__ __align__(16) int8_t s_pix[kBlkPerCta][64];
    __shared__ double s_tmp[kBlkPerCta][64];
    __shared__ __align__(16) int16_t s_out[kBlkPerCta][64];

    const int t = threadIdx.x;
    const uint32_t mx0 = blockIdx.x * kMcuPerCta;
    const uint32_t my = blockIdx.y;
    const size_t img = blockIdx.z;
    const uint8_t* __restrict__ R = p.r + img * p.plane_stride;
    const uint8_t* __restrict__ G = p.g + img * p.plane_stride;
    const uint8_t* __restrict__ B = p.b + img * p.plane_stride;

    // ---- phase 1: colour conversion + decimation into MCU tiles ----
    {
        const int pr = t >> 5;    // row pair 0..7
        const int c4 = t & 31;    // group of 4 pixels
        const int mcu = c4 >> 2;
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const int ry = pr * 2 + rr;
            uint32_t gy = (p.row0 + my) * 16u + ry;
            if (gy > p.H - 1) gy = p.H - 1;
            const size_t rowoff = size_t(gy - p.y_origin) * p.W;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int cx = c4 * 4 + i;
                uint32_t gx = mx0 * 16u + cx;
                if (gx > p.W - 1) gx = p.W - 1;
                const int rv = __ldg(R + rowoff + gx), gv = __ldg(G + rowoff + gx), bv = __ldg(B + rowoff + gx);
                const int k = (ry >> 3) * 2 + ((cx & 15) >> 3);
                s_pix[mcu * 6 + k][(ry & 7) * 8 + (cx & 7)] = int8_t(fast_Y(rv, gv, bv));
                if (rr == 0 && (i & 1) == 0) {
                    const int pos = pr * 8 + ((cx & 15) >> 1);
                    s_pix[mcu * 6 + 4][pos] = p.gray ? int8_t(0) : int8_t(fast_Cb(rv, gv, bv));
                    s_pix[mcu * 6 + 5][pos] = p.gray ? int8_t(0) : int8_t(fast_Cr(rv, gv, bv));
                }
            }
        }
    }
    __syncthreads();

    // ---- phase 2a: row pass  tmp[y][j] = sum_x pic[y][x] cos[j][x] ----
    for (int task = t; task < kBlkPerCta * 8; task += kFwdThreads) {
        const int blk = task >> 3, y = task & 7;
        double px[8];
#pragma unroll
        for (int x = 0; x < 8; ++x) px[x] = double(s_pix[blk][y * 8 + x]);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            double s = 0.0;
#pragma unroll
            for (int x = 0; x < 8; ++x) s = fma(px[x], cC.cos_ref[j * 8 + x], s);
            s_tmp[blk][y * 8 + j] = s;
        }
    }
    __syncthreads();

    // ---- phase 2b: column pass + quantisation + zig-zag ----
    unsigned long long guard_hits = 0;
    for (int task = t; task < kBlkPerCta * 8; task += kFwdThreads) {
        const int blk = task >> 3, j = task & 7;
        const int cs = (blk % 6) >= 4;
        double col[8];
#pragma unroll
        for (int y = 0; y < 8; ++y) col[y] = s_tmp[blk][y * 8 + j];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            double s = 0.0;
#pragma unroll
            for (int y = 0; y < 8; ++y) s = fma(col[y], cC.cos_ref[i * 8 + y], s);
            const double scale = 0.25 * (i ? 1.0 : 0.70710678118654752440) * (j ? 1.0 : 0.70710678118654752440);
            double v = s * scale;
            const int q = cC.quant[cs][i * 8 + j];
            const double k = rint(v / double(q));
            if (k != 0.0 && fabs(v - k * double(q)) < kGuardF64) {
                v = dct_exact(&s_pix[blk][0], i, j);
                ++guard_hits;
            }
            s_out[blk][cC.izz[i * 8 + j]] = int16_t(__double2int_rz(v) / q);
        }
    }
    __syncthreads();
    if (guard_hits) atomicAdd(p.guard_counter, guard_hits);

    // ---- phase 3: coalesced store, scan order ----
    const uint32_t nvalid = min(uint32_t(kMcuPerCta), p.HU - mx0);
    const uint32_t nwords = nvalid * 6 * 32;   // uint32 words
    uint32_t* dst = reinterpret_cast<uint32_t*>(p.coefs + img * p.coef_stride + (size_t(my) * p.HU + mx0) * 384);
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&s_out[0][0]);
    for (uint32_t w = t; w < nwords; w += kFwdThreads) dst[w] = src[w];
}

// =====================================================================================================
// Production kernel: integer colour conversion + FP32 AAN DCT, eight lanes per 8x8 block.
//
//  * tile = 16 rows x 512 pixels (32 MCUs, 192 blocks) per CTA of 256 threads
//  * phase 1 (256 threads): lane = MCU, warp = row pair; 16-byte loads per plane and row; the weighted
//    sums 299r+587g+114b etc. come from IDP.2A (two 16-bit x 8-bit products per instruction); the integer
//    quotient is the reference's truncated value unless the weighted sum is an exact multiple of the
//    denominator, where the reference's FP64 rounding decides (ref_Y/ref_Cb/ref_Cr).  Results are stored
//    as value+128 bytes in row-major shared tiles (conflict-free 16-byte stores).
//  * phase 2 (256 threads): four blocks per warp and pass (4 luma passes, 2 chroma passes); lane j transforms
//    row j, the 8x8 transpose goes through a per-warp scratch, lane j transforms column j.  AAN flowgraph (5 mul
//    + 29 add per 1-D transform) in registers; the AAN scale factors and 1/q are folded into one multiplier.
//    w = y*K; coefficients with |w| < 1 - guard quantise to 0 without further work (whole-warp test per
//    natural row); otherwise trunc(w) and the guard test |w - k| < G, k != 0.  G covers the worst-case FP32
//    error of the flowgraph (tools/aan_error_bound.py); flagged coefficients are recomputed in FP64 (tier 2)
//    and, if still within 1e-9 of a multiple of q, in the reference's exact operation order (tier 3).
//  * phase 3 (256 threads): coalesced 16-byte stores of the tile's 24 KiB of coefficients.
// =====================================================================================================
constexpr int kTileMcu = 32;
constexpr int kTileBlk = kTileMcu * 6;
constexpr int kYStride = 528;      // bytes per row of the luma tile (512 + 16: keeps 16-byte alignment)
constexpr int kCStride = 272;      // bytes per row of a chroma tile (256 + 16)
constexpr int kOutStride = 144;    // bytes per block in the staging buffer (128 + 16)
constexpr int kFwdTrSmem = 8 * 4 * 72 * 4;   // dynamic shared memory of k_fwd_transform: the transpose scratch

// quantisation constants per (class, column j), for the DCT lanes that hold one column each (a constant-bank load with a
// lane-dependent index would serialise), coefficients (i, j), i = 0..7:
struct QuantCol {
    float K[8];   // 1 / (8 * aan_i * aan_j * q_ij)
    float T[8];   // |y| below this => |w| < 1 - 2G  => quantises to 0, cannot be flagged
    float G[8];   // guard band in w units
};
static __device__ QuantCol gQcol[2][8];
static __device__ uint2 gIzzCol[8];     // zig-zag positions of coefficients (0..7, j), one byte each

// worst-case first-order FP32 error of the AAN flowgraph in v units (tools/aan_error_bound.py), rounded up
static const float kAanErrBound[64] = {
    0.00e+00f, 4.00e-04f, 3.00e-04f, 3.90e-04f, 0.00e+00f, 4.80e-04f, 3.90e-04f, 1.20e-03f,
    2.40e-04f, 6.20e-04f, 5.00e-04f, 6.20e-04f, 2.40e-04f, 7.10e-04f, 6.10e-04f, 1.50e-03f,
    1.30e-04f, 4.60e-04f, 3.60e-04f, 4.50e-04f, 1.30e-04f, 5.30e-04f, 4.50e-04f, 1.20e-03f,
    2.30e-04f, 5.80e-04f, 4.70e-04f, 5.70e-04f, 2.30e-04f, 6.60e-04f, 5.70e-04f, 1.40e-03f,
    0.00e+00f, 4.00e-04f, 3.00e-04f, 3.90e-04f, 0.00e+00f, 4.80e-04f, 3.90e-04f, 1.20e-03f,
    3.10e-04f, 8.40e-04f, 6.70e-04f, 8.30e-04f, 3.10e-04f, 9.60e-04f, 8.20e-04f, 2.00e-03f,
    2.20e-04f, 1.10e-03f, 8.00e-04f, 1.10e-03f, 2.20e-04f, 1.20e-03f, 1.10e-03f, 2.70e-03f,
    9.50e-04f, 3.00e-03f, 2.30e-03f, 2.90e-03f, 9.50e-04f, 3.40e-03f, 2.90e-03f, 7.20e-03f};

__device__ __forceinline__ int dp2a_lo_su(int a, uint32_t b, int c)
{
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int dp2a_hi_su(int a, uint32_t b, int c)
{
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__host__ __device__ constexpr int zz_at(int n)   // zig-zag position -> natural position (src/jpezy.hpp:36-45)
{
    constexpr uint8_t t[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                               41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                               30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    return t[n];
}
__host__ __device__ constexpr int pack16(int lo, int hi) { return int((uint32_t(uint16_t(lo))) | (uint32_t(uint16_t(hi)) << 16)); }

// ---- exact cases of the luma formula -----------------------------------------------------------------
// 299r + 587g + 114b is a multiple of 1000 for at most one b per (r, g) (114 b = -(299 r + 587 g) mod 1000
// has period 500 in b).  For those triples the exact value is an integer and the reference's FP64 rounding
// decides; k_build_y_exact evaluates ref_Y once per (r, g) and stores (ref_Y + 128) - exact as a signed byte.
__global__ void k_build_y_exact(int8_t* __restrict__ tbl)
{
    pdl_wait();
    const int r = blockIdx.x, g = threadIdx.x;
    int8_t corr = 0;
    for (int b = 0; b < 256; ++b) {
        const int m = 299 * r + 587 * g + 114 * b;
        if (m % 1000 == 0) corr = int8_t(ref_Y(r, g, b) + 128 - m / 1000);
    }
    tbl[r | (g << 8)] = corr;
}

// Y + 128 for the 4 pixels held in (rw, gw, bw); exact (see fast_Y)
__device__ __forceinline__ uint32_t y4(uint32_t rw, uint32_t gw, uint32_t bw, const int8_t* __restrict__ yx)
{
    const uint32_t rg01 = __byte_perm(rw, gw, 0x5140), rg23 = __byte_perm(rw, gw, 0x7362);
    uint32_t m[4], q[4], lo[4];
    m[0] = dp2a_lo_su(pack16(299, 587), rg01, dp2a_lo_su(pack16(114, 0), bw, 0));
    m[1] = dp2a_hi_su(pack16(299, 587), rg01, dp2a_lo_su(pack16(0, 114), bw, 0));
    m[2] = dp2a_lo_su(pack16(299, 587), rg23, dp2a_hi_su(pack16(114, 0), bw, 0));
    m[3] = dp2a_hi_su(pack16(299, 587), rg23, dp2a_hi_su(pack16(0, 114), bw, 0));
    uint32_t lomin = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        // exact value (m - 128000) / 1000.  m * 4294968 = floor(m / 1000) * 2^32 + lo with lo <= 179520 iff m is a
        // multiple of 1000 and lo >= 4294968 otherwise (m < 2^18): one wide multiply gives quotient and exactness.
        const unsigned long long prod = (unsigned long long)m[i] * 4294968ull;
        q[i] = uint32_t(prod >> 32);
        lo[i] = uint32_t(prod);
        lomin = min(lomin, lo[i]);
        if (q[i] < 128u && lo[i] >= 1000000u) q[i] += 1;   // truncation toward zero of a negative, non-integer value
    }
    if (lomin < 1000000u) {                     // ~0.4 % of the calls: the reference's FP64 rounding decides (table)
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (lo[i] < 1000000u) {
                const uint32_t rg = (i < 2 ? rg01 : rg23) >> ((i & 1) * 16);
                q[i] += int(yx[rg & 0xffffu]);
            }
    }
    return q[0] | (q[1] << 8) | (q[2] << 16) | (q[3] << 24);
}

// (Cb + 128) and (Cr + 128) of pixels 0 and 2 of the word triple -> two bytes each (low 16 bits).
// Exact results sit on the truncation boundary whenever r == g (1687 + 3313 = 5000), i.e. for ~0.5 % of natural
// samples, so the chroma formulas are simply evaluated as the reference does (FP64, its operation order):
// 10 DP operations per sample on a quarter of the pixels.
__device__ __forceinline__ void c2(uint32_t rw, uint32_t gw, uint32_t bw, uint32_t& cb2, uint32_t& cr2)
{
    uint32_t q[4];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const double r = double((rw >> (16 * i)) & 255u), g = double((gw >> (16 * i)) & 255u), b = double((bw >> (16 * i)) & 255u);
        const double cb = __dadd_rn(__dsub_rn(-__dmul_rn(0.1687, r), __dmul_rn(0.3313, g)), __dmul_rn(0.5000, b));
        const double cr = __dsub_rn(__dsub_rn(__dmul_rn(0.5000, r), __dmul_rn(0.4187, g)), __dmul_rn(0.0813, b));
        q[i] = uint32_t(__double2int_rz(cb) + 128);
        q[2 + i] = uint32_t(__double2int_rz(cr) + 128);
    }
    cb2 = q[0] | (q[1] << 8);
    cr2 = q[2] | (q[3] << 8);
}

// AAN forward 1-D DCT on 8 registers (outputs scaled by 8*aan_k per dimension pair, see QuantCol::K)
__device__ __forceinline__ void aan_fdct8(float& d0, float& d1, float& d2, float& d3, float& d4, float& d5, float& d6, float& d7)
{
    const float t0 = d0 + d7, t7 = d0 - d7, t1 = d1 + d6, t6 = d1 - d6;
    const float t2 = d2 + d5, t5 = d2 - d5, t3 = d3 + d4, t4 = d3 - d4;
    const float t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    d0 = t10 + t11;
    d4 = t10 - t11;
    const float z1 = (t12 + t13) * 0.707106781186547524f;
    d2 = t13 + z1;
    d6 = t13 - z1;
    const float u10 = t4 + t5, u11 = t5 + t6, u12 = t6 + t7;
    const float z5 = (u10 - u12) * 0.382683432365089772f;
    const float z2 = fmaf(u10, 0.541196100146196985f, z5);
    const float z4 = fmaf(u12, 1.306562964876376528f, z5);
    const float z3 = u11 * 0.707106781186547524f;
    const float z11 = t7 + z3, z13 = t7 - z3;
    d5 = z13 + z2;
    d3 = z13 - z2;
    d1 = z11 + z4;
    d7 = z11 - z4;
}

// Fix-up queue: coefficients whose FP32 value is inside the guard band are not decided in the hot loop;
// (block, natural index) is pushed to shared memory and the whole CTA re-evaluates the queue afterwards.
constexpr int kFixCap = 1024;

__device__ __noinline__ void push_fix(uint32_t* s_nfix, uint16_t* s_fix, uint32_t blk_ij)
{
    const uint32_t idx = atomicAdd(s_nfix, 1u);
    if (idx < kFixCap) s_fix[idx] = uint16_t(blk_ij);
}

// tier 2 decision on the FP64 sum `acc` of coefficient (i, j); tier 3 (the reference's exact operation order, same
// arithmetic as dct_exact) when even that lands within 1e-9 of a quantiser multiple
__device__ __noinline__ int requant_finish(double acc, const uint8_t* __restrict__ tile, int stride, int i, int j, int q, unsigned long long* counter)
{
    double v = acc * 0.25 * (i ? 1.0 : 0.70710678118654752440) * (j ? 1.0 : 0.70710678118654752440);
    const double k = rint(v / double(q));
    if (k != 0.0 && fabs(v - k * double(q)) < 1e-9) {
        double sum = 0.0;
        for (int y = 0; y < 8; ++y) {
            const double ci = cC.cos_ref[i * 8 + y];
            for (int x = 0; x < 8; ++x)
                sum = __dadd_rn(sum, __dmul_rn(__dmul_rn(double(int(tile[y * stride + x]) - 128), cC.cos_ref[j * 8 + x]), ci));
        }
        const double cu = j ? 1.0 : cC.inv_sqrt2_ref, cv = i ? 1.0 : cC.inv_sqrt2_ref;
        v = __dmul_rn(__dmul_rn(__dmul_rn(sum, cu), cv), 0.25);
        atomicAdd(counter, 1ull);
    }
    return __double2int_rz(v) / q;
}

// tier 2 / tier 3 of the guard: FP64 evaluation of one coefficient from the stored (value+128) samples
__device__ __noinline__ int requant_exact(const uint8_t* __restrict__ tile, int stride, int i, int j, int q, unsigned long long* counter)
{
    double acc = 0.0;
    for (int y = 0; y < 8; ++y) {
        double row = 0.0;
#pragma unroll
        for (int x = 0; x < 8; ++x) row = fma(double(int(tile[y * stride + x]) - 128), cC.cos_ref[j * 8 + x], row);
        acc = fma(row, cC.cos_ref[i * 8 + y], acc);
    }
    return requant_finish(acc, tile, stride, i, j, q, counter);
}

// location of block `blk` (= mcu*6 + k) of the tile in the shared sample tiles
__device__ __forceinline__ const uint8_t* block_samples(const uint8_t* s_y, const uint8_t* s_cb, const uint8_t* s_cr, uint32_t blk, int& stride)
{
    const uint32_t mcu = blk / 6u, k = blk - mcu * 6u;
    if (k < 4u) {
        stride = kYStride;
        return s_y + (k >> 1) * 8 * kYStride + mcu * 16 + (k & 1) * 8;
    }
    stride = kCStride;
    return (k == 4u ? s_cb : s_cr) + mcu * 8;
}

// Phase 2 works with eight lanes per block (one row, then one column each; the 8x8 transpose goes through a per-warp
// scratch in shared memory).  A thread then carries 8 samples instead of the 64 of one thread per block: half the
// registers, twice the resident warps -- the kernel is latency bound (ncu: issue slots 42 % busy at 16 warps per SM).
__global__ void __launch_bounds__(256, 4) k_fwd_transform(const FwdParams p)
{
    pdl_wait();
    extern __shared__ __align__(16) float s_tr[];                 // [warp][block of the pass][8 rows x 8 + 8 pad] (kFwdTrSmem)
    __shared__ __align__(16) uint8_t s_y[16 * kYStride];
    __shared__ __align__(16) uint8_t s_cb[8 * kCStride];
    __shared__ __align__(16) uint8_t s_cr[8 * kCStride];
    __shared__ __align__(16) uint8_t s_out[kTileBlk * kOutStride];
    __shared__ uint16_t s_fix[kFixCap];
    __shared__ uint32_t s_nfix;

    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const uint32_t mx0 = blockIdx.x * kTileMcu;
    const uint32_t my = blockIdx.y;
    const size_t img = blockIdx.z;
    const uint8_t* __restrict__ R = p.r + img * p.plane_stride;
    const uint8_t* __restrict__ G = p.g + img * p.plane_stride;
    const uint8_t* __restrict__ B = p.b + img * p.plane_stride;
    if (t == 0) s_nfix = 0;

    // ---- phase 1: colour conversion + decimation; warp = row pair, lane = MCU ----
    {
        const uint32_t mx = mx0 + lane;
        const uint32_t x0 = mx * 16u;
        const bool fast = ((p.W & 15u) == 0) && x0 + 16u <= p.W;
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const int ry = warp * 2 + rr;
            uint32_t gy = (p.row0 + my) * 16u + ry;
            if (gy > p.H - 1) gy = p.H - 1;
            const size_t rowoff = size_t(gy - p.y_origin) * p.W;
            uint4 rv, gv, bv;
            if (fast) {
                rv = __ldg(reinterpret_cast<const uint4*>(R + rowoff + x0));
                gv = __ldg(reinterpret_cast<const uint4*>(G + rowoff + x0));
                bv = __ldg(reinterpret_cast<const uint4*>(B + rowoff + x0));
            } else if (mx < p.HU) {
                uint32_t rw[4], gw[4], bw[4];
#pragma unroll 1
                for (int w = 0; w < 4; ++w) {
                    rw[w] = gw[w] = bw[w] = 0;
#pragma unroll 1
                    for (int i = 0; i < 4; ++i) {
                        uint32_t gx = x0 + w * 4 + i;
                        if (gx > p.W - 1) gx = p.W - 1;
                        rw[w] |= uint32_t(__ldg(R + rowoff + gx)) << (8 * i);
                        gw[w] |= uint32_t(__ldg(G + rowoff + gx)) << (8 * i);
                        bw[w] |= uint32_t(__ldg(B + rowoff + gx)) << (8 * i);
                    }
                }
                rv = make_uint4(rw[0], rw[1], rw[2], rw[3]);
                gv = make_uint4(gw[0], gw[1], gw[2], gw[3]);
                bv = make_uint4(bw[0], bw[1], bw[2], bw[3]);
            } else {
                rv = gv = bv = make_uint4(0, 0, 0, 0);
            }
            uint4 yv;
            yv.x = y4(rv.x, gv.x, bv.x, p.y_exact), yv.y = y4(rv.y, gv.y, bv.y, p.y_exact);
            yv.z = y4(rv.z, gv.z, bv.z, p.y_exact), yv.w = y4(rv.w, gv.w, bv.w, p.y_exact);
            *reinterpret_cast<uint4*>(&s_y[ry * kYStride + lane * 16]) = yv;
            if (rr == 0) {
                uint2 cbv = make_uint2(0x80808080u, 0x80808080u), crv = cbv;   // gray: Cb = Cr = 0 (stored +128)
                if (!p.gray) {
                    uint32_t b0, r0, b1, r1, b2, r2, b3, r3;
                    c2(rv.x, gv.x, bv.x, b0, r0);
                    c2(rv.y, gv.y, bv.y, b1, r1);
                    c2(rv.z, gv.z, bv.z, b2, r2);
                    c2(rv.w, gv.w, bv.w, b3, r3);
                    cbv = make_uint2(b0 | (b1 << 16), b2 | (b3 << 16));
                    crv = make_uint2(r0 | (r1 << 16), r2 | (r3 << 16));
                }
                *reinterpret_cast<uint2*>(&s_cb[warp * kCStride + lane * 8]) = cbv;
                *reinterpret_cast<uint2*>(&s_cr[warp * kCStride + lane * 8]) = crv;
            }
        }
    }
    __syncthreads();

    // ---- phase 2: DCT + quantisation, eight lanes per block, four blocks per warp and pass ----
    // passes 0..3: the 128 luma blocks (luma block lb = pass * 32 + warp * 4 + g: MCU lb >> 2, block lb & 3);
    // passes 4..5: the 32 Cb and the 32 Cr blocks
    const int g = lane >> 3, j = lane & 7;
    float* scr = &s_tr[(warp * 4 + g) * 72];
    const uint2 izz = gIzzCol[j];
#pragma unroll
    for (int cls = 0; cls < 2; ++cls) {
        float K[8], T[8];
        {
            const float4* q4 = reinterpret_cast<const float4*>(&gQcol[cls][j]);
            const float4 k0 = q4[0], k1 = q4[1], t0 = q4[2], t1 = q4[3];
            K[0] = k0.x, K[1] = k0.y, K[2] = k0.z, K[3] = k0.w, K[4] = k1.x, K[5] = k1.y, K[6] = k1.z, K[7] = k1.w;
            T[0] = t0.x, T[1] = t0.y, T[2] = t0.z, T[3] = t0.w, T[4] = t1.x, T[5] = t1.y, T[6] = t1.z, T[7] = t1.w;
            if (j == 0) T[0] = 3.0e38f;        // the DC coefficient takes its own path
        }
#pragma unroll 1
        for (int pass = 0; pass < (cls ? 2 : 4); ++pass) {
            const uint32_t n = uint32_t(pass) * 32u + uint32_t(warp) * 4u + uint32_t(g);
            uint32_t blk;
            const uint8_t* row;
            if (cls == 0) {
                const uint32_t mcu = n >> 2, k = n & 3u;
                blk = mcu * 6u + k;
                row = &s_y[((k >> 1) * 8 + j) * kYStride + mcu * 16 + (k & 1u) * 8];
            } else {
                const uint32_t mcu = n & 31u, comp = n >> 5;
                blk = mcu * 6u + 4u + comp;
                row = (comp ? s_cr : s_cb) + j * kCStride + mcu * 8;
            }
            float d[8];
            {
                const uint2 w = *reinterpret_cast<const uint2*>(row);
                d[0] = float(w.x & 255u), d[1] = float((w.x >> 8) & 255u), d[2] = float((w.x >> 16) & 255u), d[3] = float(w.x >> 24);
                d[4] = float(w.y & 255u), d[5] = float((w.y >> 8) & 255u), d[6] = float((w.y >> 16) & 255u), d[7] = float(w.y >> 24);
            }
            aan_fdct8(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);      // row j of the block
            *reinterpret_cast<float4*>(&scr[j * 8]) = make_float4(d[0], d[1], d[2], d[3]);
            *reinterpret_cast<float4*>(&scr[j * 8 + 4]) = make_float4(d[4], d[5], d[6], d[7]);
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i) d[i] = scr[i * 8 + j];
            __syncwarp();
            aan_fdct8(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);      // column j: d[i] = coefficient (i, j)
            int16_t* out = reinterpret_cast<int16_t*>(&s_out[blk * kOutStride]);
            // rows of coefficients in which some lane of the warp may quantise to a non-zero value (|y| >= T <=> |w| >= 1 - 2G)
            uint32_t lm = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) lm |= (fabsf(d[i]) >= T[i] ? 1u : 0u) << i;
            const uint32_t wm = __reduce_or_sync(0xffffffffu, lm);
            int qv[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                qv[i] = 0;
                if (wm & (1u << i)) {
                    const float w = d[i] * K[i];
                    qv[i] = __float2int_rz(w);
                    // distance of |w| to the nearest integer >= 1
                    const float a = fabsf(w) - 0.5f;
                    const float kf = (a + 12582912.0f) - 12582912.0f;      // rint(|w| - 0.5)
                    const float delta = a - kf;                             // frac(|w|) - 0.5 in [-0.5, 0.5]
                    if (fabsf(delta) > 0.5f - gQcol[cls][j].G[i] && fabsf(w) > 0.5f && (i | j) != 0)
                        push_fix(&s_nfix, s_fix, (blk << 6) | uint32_t(i * 8 + j));
                }
            }
            if (j == 0) {
                // DC: the reference's sum is an exact integer (cos row 0 is 1.0), so its value is ((S*c)*c)/4 exactly as
                // evaluated; level shift: the samples are stored as value + 128 (64 * 128, exact)
                const double v = __dmul_rn(__dmul_rn(__dmul_rn(double(d[0] - 8192.0f), cC.inv_sqrt2_ref), cC.inv_sqrt2_ref), 0.25);
                qv[0] = cls ? __double2int_rz(v) / 17 : __double2int_rz(v) / 16;
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) out[__byte_perm(i < 4 ? izz.x : izz.y, 0, 0x4440 + (i & 3))] = int16_t(qv[i]);
        }
    }
    __syncthreads();

    // ---- phase 2b: dense re-evaluation of the guard-band queue ----
    {
        const uint32_t nfix = s_nfix;
        if (nfix) {
            if (nfix > kFixCap) {
                // queue overflow (adversarial content): every coefficient of the tile is re-evaluated exactly
                for (uint32_t e = t; e < kTileBlk * 64u; e += 256) {
                    const uint32_t blk = e >> 6, ij = e & 63u;
                    int stride;
                    const uint8_t* tile = block_samples(s_y, s_cb, s_cr, blk, stride);
                    const int q = cC.quant[(blk % 6u) >= 4u][ij];
                    reinterpret_cast<int16_t*>(&s_out[blk * kOutStride])[cC.izz[ij]] = int16_t(requant_exact(tile, stride, ij >> 3, ij & 7, q, p.guard_counter));
                }
            } else {
                // eight lanes per queue entry: lane `sub` evaluates row `sub` of the separable sum, a 3-step butterfly adds
                // the rows (the tail of a tile is the latency of this phase, not its instruction count)
                const uint32_t sub = uint32_t(t) & 7u;
                for (uint32_t e0 = 0; e0 < nfix; e0 += 32) {
                    const uint32_t e = e0 + (uint32_t(t) >> 3);
                    const bool act = e < nfix;
                    const uint32_t ent = act ? uint32_t(s_fix[e]) : 0u;
                    const uint32_t blk = ent >> 6, ij = ent & 63u, i = ij >> 3, j = ij & 7u;
                    int stride;
                    const uint8_t* tile = block_samples(s_y, s_cb, s_cr, blk, stride);
                    const uint2 w = *reinterpret_cast<const uint2*>(tile + sub * stride);
                    const double* cj = &gCosRef[j * 8];
                    double row = double(int(w.x & 255u) - 128) * cj[0];
                    row = fma(double(int((w.x >> 8) & 255u) - 128), cj[1], row);
                    row = fma(double(int((w.x >> 16) & 255u) - 128), cj[2], row);
                    row = fma(double(int(w.x >> 24) - 128), cj[3], row);
                    row = fma(double(int(w.y & 255u) - 128), cj[4], row);
                    row = fma(double(int((w.y >> 8) & 255u) - 128), cj[5], row);
                    row = fma(double(int((w.y >> 16) & 255u) - 128), cj[6], row);
                    row = fma(double(int(w.y >> 24) - 128), cj[7], row);
                    double part = row * gCosRef[i * 8 + sub];
                    part += __shfl_xor_sync(0xffffffffu, part, 1);
                    part += __shfl_xor_sync(0xffffffffu, part, 2);
                    part += __shfl_xor_sync(0xffffffffu, part, 4);
                    if (act && sub == 0) {
                        const int q = cC.quant[(blk % 6u) >= 4u][ij];
                        reinterpret_cast<int16_t*>(&s_out[blk * kOutStride])[cC.izz[ij]] =
                            int16_t(requant_finish(part, tile, stride, int(i), int(j), q, p.guard_counter));
                    }
                }
            }
            __syncthreads();
        }
    }

    // ---- phase 3: coalesced store, scan order ----
    const uint32_t nvalid = min(uint32_t(kTileMcu), p.HU - mx0);
    const uint32_t nchunks = nvalid * 6 * 8;   // 16-byte chunks
    uint4* dst = reinterpret_cast<uint4*>(p.coefs + img * p.coef_stride + (size_t(my) * p.HU + mx0) * 384);
    uint32_t* meta = p.bmeta ? p.bmeta + img * (p.coef_stride >> 6) + (size_t(my) * p.HU + mx0) * 6 : nullptr;
#pragma unroll
    for (uint32_t c0 = 0; c0 < uint32_t(kTileBlk) * 8u; c0 += 256) {
        const uint32_t c = c0 + uint32_t(t);
        const uint4 v = *reinterpret_cast<const uint4*>(&s_out[(c >> 3) * kOutStride + (c & 7) * 16]);
        if (c < nchunks) dst[c] = v;
        if (meta) {
            const bool nz = (((c & 7u) ? v.x : (v.x >> 16)) | v.y | v.z | v.w) != 0u;      // (group 0 without the DC coefficient)
            const uint32_t nzb = __ballot_sync(0xffffffffu, nz);
            if ((lane & 7) == 0 && c < nchunks) meta[c >> 3] = (v.x & 0xffffu) | (((nzb >> lane) & 0xffu) << 16);
        }
    }
}

}  // namespace jz
