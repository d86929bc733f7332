// dec_transform2.cuh -- stages D2+D3, second generation: quantised coefficients -> planar RGB (2x2 / 1x1 / 1x1 frames).
//
// Replaces inverse_quantization (src/decoder/jpezy_decoder.hpp:645-650), inverse_dct (:652-670), the pixel replication of
// decode_mcu (:519-524) and make_rgb / to_r,g,b / revise_value (:531-578, :672-676), like k_inv_transform of dec_transform.cuh
// (which stays for buffers that are not 16-byte aligned).  ncu of round 1 showed that kernel bound by
// instruction issue and by its barriers (one thread per 8x8 block with 64 live samples, 96 registers, 25 % of the warp slots
// filled, four CTA-wide barriers with different numbers of threads working).  Here:
//
//  * a tile is T MCUs of one MCU row; its 768 T bytes of coefficients arrive through ONE bulk copy (cp.async.bulk +
//    mbarrier): no per-thread global loads on the input side;
//  * eight lanes per block PAIR (Y0|Y2, Y1|Y3, Cb|Cr), packed f32x2 arithmetic on the two blocks of the pair: lane u
//    de-zig-zags, dequantises and transforms column u, the 8x8 transpose goes through a padded conflict-free scratch that
//    belongs to the warp (__syncwarp, not a CTA barrier), lane y transforms row y and decides its 8 + 8 samples;
//  * when no block of the warp has a coefficient beyond zig-zag position 7 the flowgraphs are pruned to 3 inputs per column
//    and 4 per row (operations on structural zeros dropped: bit-identical to the full flowgraph);
//  * when no block of the warp has a coefficient beyond zig-zag position 2 (photographic content at normal quality: nearly
//    every warp) the sample is the separable sum F00 q00 / 8 + 128 + F10 Ly[y] + F01 Lx[x]: lane y evaluates its row of both
//    blocks with eight FFMA2, no column pass and no transpose, under a guard band of its own (tools/lowfreq_idct_error_bound.py);
//  * floor(v) is one FADD2.RM against 1.5 * 2^23 (the integer sits in the low mantissa bits), the distance to the nearest
//    integer three more packed adds; one 3-input-min chain per block row decides whether any sample is inside the guard
//    band; negative samples (where the reference's truncation is not floor) and guard hits take the slow row function;
//  * the chroma lanes turn their samples into the three integer colour offsets right away (dec_transform.cuh explains why
//    trunc(y + t) = y + floor(t)); the colour phase is integer adds and saturating packs on 16 pixels of one row per thread,
//    three 16-byte planar stores.
//
// Numerics: same AAN flowgraphs, same per-block guard band (tools/aan_idct_error_bound.py; the low-frequency class has its
// own), same FP64 fix-up queue and exact-order tier as k_inv_transform; DC-only blocks are evaluated in the reference's operation order.  Decoded samples are
// identical to the reference decoder's.  Algorithmic HBM traffic: 3 B/px read + 3 B/px written = 6 B/px.
#pragma once
#include "dec_transform.cuh"

namespace jz {

// ---- async proxy: the bulk copy of a tile's coefficients and its barrier ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completes `bytes` on the barrier
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// wait with a watchdog: a protocol error must trap, not hang the device
// (try_wait with a suspend-time hint: the warp sleeps in hardware until the phase completes instead of polling)
__device__ __forceinline__ void mbar_wait_wd(uint32_t bar, uint32_t parity)
{
    uint32_t ok, spins = 0;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity), "r"(1000000u) : "memory");
        if (!ok && ++spins > (1u << 16)) __trap();
    } while (!ok);
}

// ---- packed FP32 pairs (FADD2 / FMUL2 / FFMA2 of sm_100): the two blocks of a pair go through a flowgraph at once; every
// lane of a pair is an ordinary IEEE add / mul / fma, so the results equal the scalar flowgraph's bit for bit ----
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi)
{
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c)
{
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ float lo2(f32x2 v) { return __uint_as_float(uint32_t(v)); }
__device__ __forceinline__ float hi2(f32x2 v) { return __uint_as_float(uint32_t(v >> 32)); }

constexpr float kMagic15 = 12582912.0f;    // 1.5 * 2^23: float(kMagic15 + n) has the integer n in its low mantissa bits (|n| < 2^22)

// per frame descriptor (quantisation tables), laid out for the column lanes; built by k_build_inv2_tab when the tables change
struct Inv2Tab {
    float2 M[2][8][8];     // [pair class][u][v]: (M of block A, M of block B), M = q * aan_v * aan_u / 8 of coefficient (v, u);
                           // class 0 = two luma blocks, class 1 = Cb | Cr (their quantisation tables may differ)
    float2 Wg[2][8][8];    // [pair class][u][v]: guard-band weights per unit |coefficient|
    uint2 zoff[8];         // [u]: byte offsets (2 * zig-zag position) of coefficients (0..7, u), one byte each
    // blocks with nothing beyond zig-zag position 2: sample (x, y) = F(0,0) q / 8 + 128 + F(1,0) Ly[y] + F(0,1) Lx[x]
    float2 Lx[2][8];       // [pair class][x]: q(0,1) cos((2x+1) pi / 16) / (4 sqrt 2)
    float2 Ly[2][8];       // [pair class][y]: q(1,0) cos((2y+1) pi / 16) / (4 sqrt 2)
    float2 Lg[2][4];       // [pair class]: guard-band weights of zig-zag positions 0..2 per unit |coefficient|, then the constant term
};

// worst-case FP32 error of that evaluation per unit dequantised coefficient of zig-zag position 0, 1, 2 (units of 2^-24, margin
// 1.25 included) and its constant term, the level shift rounded three times (tools/lowfreq_idct_error_bound.py)
constexpr double kLowErrSens0 = 0.625, kLowErrSens1 = 0.434, kLowErrSens2 = 0.651;
constexpr float kLowGuard0 = 2.87e-5f;

__global__ void k_build_inv2_tab(const InvParams p, Inv2Tab* __restrict__ tab)
{
    pdl_wait();
    const int t = threadIdx.x;      // 128 threads: pair class, natural position
    const int c = t >> 6, nat = t & 63, v = nat >> 3, u = nat & 7;
    const int ca = c ? 1 : 0, cb = c ? 2 : 0;
    tab->M[c][u][v] = make_float2(p.M[ca][nat], p.M[cb][nat]);
    tab->Wg[c][u][v] = make_float2(p.Wg[ca][nat], p.Wg[cb][nat]);
    if (t < 8) {
        uint32_t w[2] = {0, 0};
        for (int vv = 0; vv < 8; ++vv) w[vv >> 2] |= uint32_t(cC.izz[vv * 8 + t] * 2) << (8 * (vv & 3));
        tab->zoff[t] = make_uint2(w[0], w[1]);
    }
    if (nat < 8) {      // the low-frequency class: column / row `nat`
        const double s = cC.cos_ref[8 + nat] * cC.inv_sqrt2_ref * 0.25;
        tab->Lx[c][nat] = make_float2(float(p.qt[ca][1] * s), float(p.qt[cb][1] * s));
        tab->Ly[c][nat] = make_float2(float(p.qt[ca][8] * s), float(p.qt[cb][8] * s));
        if (nat < 4) {
            const int n = nat == 2 ? 8 : nat;      // natural position of zig-zag position `nat`
            const double e = (nat == 0 ? kLowErrSens0 : nat == 1 ? kLowErrSens1 : kLowErrSens2) / 16777216.0;
            tab->Lg[c][nat] = nat == 3 ? make_float2(kLowGuard0, kLowGuard0) : make_float2(float(p.qt[ca][n] * e), float(p.qt[cb][n] * e));
        }
    }
}

__device__ __forceinline__ f32x2 add2_rm(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("add.rm.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ float fmin3_abs(float a, float b, float c)
{
    float r;
    asm("{\n\t.reg .f32 x, y;\n\tabs.f32 x, %1;\n\tabs.f32 y, %2;\n\tmin.f32 %0, x, y, %3;\n\t}" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}
__device__ __forceinline__ float fmax3_abs(float a, float b, float c)
{
    float r;
    asm("{\n\t.reg .f32 x, y;\n\tabs.f32 x, %1;\n\tabs.f32 y, %2;\n\tmax.f32 %0, x, y, %3;\n\t}" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}
// base + byte K of w (one IDP.4A)
template <int K>
__device__ __forceinline__ uint32_t add_byte(uint32_t w, uint32_t base)
{
    uint32_t d;
    asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(1u << (8 * K)), "r"(base));
    return d;
}

// ---- packed AAN inverse flowgraphs: aan_idct8 / aan_idct8_in3 / aan_idct8_in4 of dec_transform.cuh on two blocks at once.
// Where the scalar code subtracts inside an FMA (fmaf(a, c, -b)) the packed code carries the negated value (fma(a, -c, b))
// and flips the sign of its uses: round-to-nearest is symmetric, the results are the same bit for bit. ----
__device__ __forceinline__ void aan_idct8_x2(f32x2& d0, f32x2& d1, f32x2& d2, f32x2& d3, f32x2& d4, f32x2& d5, f32x2& d6, f32x2& d7)
{
    const f32x2 c1414 = pk2(1.414213562373095049f, 1.414213562373095049f), c1847 = pk2(1.847759065022573512f, 1.847759065022573512f);
    const f32x2 cm1082 = pk2(-1.082392200292393968f, -1.082392200292393968f), cm2613 = pk2(-2.613125929752753055f, -2.613125929752753055f);
    const f32x2 t10 = add2(d0, d4), t11 = sub2(d0, d4);
    const f32x2 t13 = add2(d2, d6);
    const f32x2 nt12 = fma2(sub2(d6, d2), c1414, t13);                 // -t12
    const f32x2 e0 = add2(t10, t13), e3 = sub2(t10, t13), e1 = sub2(t11, nt12), e2 = add2(t11, nt12);
    const f32x2 z13 = add2(d5, d3), z10 = sub2(d5, d3), z11 = add2(d1, d7), z12 = sub2(d1, d7);
    const f32x2 o7 = add2(z11, z13);
    const f32x2 o11 = mul2(sub2(z11, z13), c1414);
    const f32x2 z5 = mul2(add2(z10, z12), c1847);
    const f32x2 no10 = fma2(z12, cm1082, z5);                           // -o10
    const f32x2 o12 = fma2(z10, cm2613, z5);
    const f32x2 o6 = sub2(o12, o7);
    const f32x2 o5 = sub2(o11, o6);
    const f32x2 o4 = sub2(o5, no10);
    d0 = add2(e0, o7), d7 = sub2(e0, o7);
    d1 = add2(e1, o6), d6 = sub2(e1, o6);
    d2 = add2(e2, o5), d5 = sub2(e2, o5);
    d4 = add2(e3, o4), d3 = sub2(e3, o4);
}
// inputs d3..d7 == 0
__device__ __forceinline__ void aan_idct8_in3_x2(f32x2& d0, f32x2& d1, f32x2& d2, f32x2& d3, f32x2& d4, f32x2& d5, f32x2& d6, f32x2& d7)
{
    const f32x2 c1414 = pk2(1.414213562373095049f, 1.414213562373095049f), c1847 = pk2(1.847759065022573512f, 1.847759065022573512f);
    const f32x2 cm1414 = pk2(-1.414213562373095049f, -1.414213562373095049f), cm1082 = pk2(-1.082392200292393968f, -1.082392200292393968f);
    const f32x2 nt12 = fma2(d2, cm1414, d2);                            // -(d2 * 1.414 - d2)
    const f32x2 e0 = add2(d0, d2), e3 = sub2(d0, d2), e1 = sub2(d0, nt12), e2 = add2(d0, nt12);
    const f32x2 o7 = d1;
    const f32x2 o11 = mul2(d1, c1414);
    const f32x2 z5 = mul2(d1, c1847);
    const f32x2 no10 = fma2(d1, cm1082, z5);
    const f32x2 o6 = sub2(z5, o7);
    const f32x2 o5 = sub2(o11, o6);
    const f32x2 o4 = sub2(o5, no10);
    d0 = add2(e0, o7), d7 = sub2(e0, o7);
    d1 = add2(e1, o6), d6 = sub2(e1, o6);
    d2 = add2(e2, o5), d5 = sub2(e2, o5);
    d4 = add2(e3, o4), d3 = sub2(e3, o4);
}
// inputs d4..d7 == 0
__device__ __forceinline__ void aan_idct8_in4_x2(f32x2& d0, f32x2& d1, f32x2& d2, f32x2& d3, f32x2& d4, f32x2& d5, f32x2& d6, f32x2& d7)
{
    const f32x2 c1414 = pk2(1.414213562373095049f, 1.414213562373095049f), c1847 = pk2(1.847759065022573512f, 1.847759065022573512f);
    const f32x2 cm1414 = pk2(-1.414213562373095049f, -1.414213562373095049f), cm1082 = pk2(-1.082392200292393968f, -1.082392200292393968f);
    const f32x2 c2613 = pk2(2.613125929752753055f, 2.613125929752753055f);
    const f32x2 nt12 = fma2(d2, cm1414, d2);
    const f32x2 e0 = add2(d0, d2), e3 = sub2(d0, d2), e1 = sub2(d0, nt12), e2 = add2(d0, nt12);
    const f32x2 dm = sub2(d1, d3);
    const f32x2 o7 = add2(d1, d3);
    const f32x2 o11 = mul2(dm, c1414);
    const f32x2 z5 = mul2(dm, c1847);
    const f32x2 no10 = fma2(d1, cm1082, z5);
    const f32x2 o12 = fma2(d3, c2613, z5);
    const f32x2 o6 = sub2(o12, o7);
    const f32x2 o5 = sub2(o11, o6);
    const f32x2 o4 = sub2(o5, no10);
    d0 = add2(e0, o7), d7 = sub2(e0, o7);
    d1 = add2(e1, o6), d6 = sub2(e1, o6);
    d2 = add2(e2, o5), d5 = sub2(e2, o5);
    d4 = add2(e3, o4), d3 = sub2(e3, o4);
}

// the reference's value of every sample of a DC-only block: ((c*c)*F)*1*1, /4, +128 in its operation order (:657-668)
__device__ __forceinline__ int dc_only_value(int c, int q)
{
    const double term = __dmul_rn(__dmul_rn(cC.inv_sqrt2_ref, cC.inv_sqrt2_ref), double(c * q));
    return __double2int_rz(__dadd_rn(__dmul_rn(term, 0.25), 128.0));
}

// slow half of one block row: truncation toward zero of every sample (the fast path floors), guard-band samples queued.
// (The samples travel in registers: an array argument would be built in local memory on the hot path.)
__device__ __forceinline__ uint32_t inv_slow_sample(float v, float guard, uint32_t entry, uint32_t* s_nfix, uint16_t* s_fix)
{
    const float kf = (v + kMagic15) - kMagic15;
    if (fabsf(v - kf) < guard) push_fix16(s_nfix, s_fix, entry);
    return uint32_t(__float2int_rz(v)) & 0xffffu;
}
__device__ __noinline__ uint4 inv_row_slow(float v0, float v1, float v2, float v3, float v4, float v5, float v6, float v7, float guard, uint32_t blk,
                                           int y, uint32_t* s_nfix, uint16_t* s_fix)
{
    const uint32_t e = (blk << 7) | uint32_t(y * 8);
    uint4 w;
    w.x = inv_slow_sample(v0, guard, e, s_nfix, s_fix) | (inv_slow_sample(v1, guard, e + 1, s_nfix, s_fix) << 16);
    w.y = inv_slow_sample(v2, guard, e + 2, s_nfix, s_fix) | (inv_slow_sample(v3, guard, e + 3, s_nfix, s_fix) << 16);
    w.z = inv_slow_sample(v4, guard, e + 4, s_nfix, s_fix) | (inv_slow_sample(v5, guard, e + 5, s_nfix, s_fix) << 16);
    w.w = inv_slow_sample(v6, guard, e + 6, s_nfix, s_fix) | (inv_slow_sample(v7, guard, e + 7, s_nfix, s_fix) << 16);
    return w;
}
// colour_exact4 with the four luma samples in registers
__device__ __noinline__ uint32_t colour_exact4r(int y0, int y1, int y2, int y3, uint32_t cc0, uint32_t cc1, int which)
{
    const int y[4] = {y0, y1, y2, y3};
    return colour_exact4(y, sx_lo(cc0), sx_hi(cc0), sx_lo(cc1), sx_hi(cc1), which);
}

// the colour offsets of one chroma pair (as phase 1c of k_inv_transform computes them) from the packed samples cb | cr << 16: fr | fg << 16 and
// fb | suspect << 16.  No conversion instructions: floor(x) is the low mantissa bits of x + 1.5 * 2^23 rounded down (|x| < 2^22),
// two of the three offsets share packed instructions
__device__ __forceinline__ uint2 chroma_offsets_w(uint32_t ccw)
{
    const f32x2 ab = add2(pk2(float(sx_lo(ccw)), float(sx_hi(ccw))), pk2(-128.0f, -128.0f));       // (cb - 128, cr - 128)
    const f32x2 fl = add2_rm(mul2(ab, pk2(1.7718f, 1.4020f)), pk2(kMagic15, kMagic15));           // floor(a * 1.7718) | floor(b * 1.4020)
    const float a = lo2(ab), b = hi2(ab);
    const float tg = fmaf(b, -0.7139f, a * -0.3441f);
    float fgm;
    asm("add.rm.f32 %0, %1, %2;" : "=f"(fgm) : "f"(tg), "f"(kMagic15));
    const float kf = (tg + kMagic15) - kMagic15;
    const bool near_int = fabsf(tg - kf) < 7.5e-5f && ccw != 0x00800080u;
    const bool wild = fmaxf(fabsf(a), fabsf(b)) > 256.0f;
    return make_uint2(__byte_perm(uint32_t(fl >> 32), __float_as_uint(fgm), 0x5410), (uint32_t(fl) & 0xffffu) | ((near_int || wild) ? 0x10000u : 0u));
}

template <int T>
struct Inv2 {
    static constexpr int kThreads = T * 24;
    static constexpr int kCoef = T * 768;
    static constexpr int kPairRow = 80, kPair = 8 * kPairRow + 64;
    static constexpr int kMid = T * 3 * kPair;
    static constexpr int kYRow = T * 32 + 16;          // int16 luma samples, 16 rows
    static constexpr int kY = 16 * kYRow;
    static constexpr int kOffRow = T * 64 + 16;        // uint2 per chroma pair, 8 rows
    static constexpr int kOff = 8 * kOffRow;
    static constexpr int kCcRow = T * 32 + 16;         // (Cb, Cr) int16 per chroma pair, 8 rows
    static constexpr int kCc = 8 * kCcRow;
    static constexpr int kSmem = kCoef + kMid + kY + kOff + kCc + kFixCap * 2 + 16 + T * 6 + 16;
};

template <int T>
__global__ void __launch_bounds__(T * 24, T == 8 ? 5 : 2) k_inv_transform2(const __grid_constant__ InvParams p, const Inv2Tab* __restrict__ tab)
{
    using C = Inv2<T>;
    extern __shared__ __align__(16) uint8_t smem[];
    uint8_t* s_coef = smem;                                  // [6T blocks][64] int16, zig-zag, scan order
    uint8_t* s_mid = s_coef + C::kCoef;                      // [3T pairs][8][kPairRow] transpose scratch, (A, B) packed
    uint8_t* s_y = s_mid + C::kMid;                          // [16][kYRow] int16 luma samples
    uint8_t* s_off = s_y + C::kY;                            // [8][kOffRow] colour offsets per chroma pair
    uint8_t* s_cc = s_off + C::kOff;                         // [8][kCcRow] chroma samples (exact path, fix-up)
    uint16_t* s_fix = reinterpret_cast<uint16_t*>(s_cc + C::kCc);
    uint32_t* s_nfix = reinterpret_cast<uint32_t*>(s_fix + kFixCap);
    const uint32_t bar = smem_u32(s_nfix + 2);
    uint8_t* s_mask = reinterpret_cast<uint8_t*>(s_nfix + 4);    // [6T] non-zero zig-zag groups of every block

    const int t = threadIdx.x, lane = t & 31;
    const uint32_t mx0 = blockIdx.x * T, my = blockIdx.y + p.row0;
    const size_t img = blockIdx.z;
    const uint32_t nvalid = min(uint32_t(T), p.HU - mx0);
    const size_t mcu0 = size_t(my) * p.HU + mx0;

    if (t == 0) {
        mbar_init(bar, 1);
        s_nfix[0] = 0, s_nfix[1] = 0;      // fix-up count, "a sample leaves the int16 range" (kWideSample)
        mbar_fence_init();
    }
    __syncthreads();
    pdl_wait();
    if (t == 0) {
        mbar_expect_tx(bar, nvalid * 768u);
        bulk_g2s(smem_u32(s_coef), p.coefs + img * p.coef_stride + mcu0 * 384, nvalid * 768u, bar);
    }

    // ---- the item of this thread: block pair pr, column (then row) sub ----
    const uint32_t pr = uint32_t(t) >> 3, sub = uint32_t(t) & 7u;
    const bool luma = pr < 2u * T;
    const uint32_t mcu = luma ? (pr >> 1) : pr - 2u * T;
    const bool valid = mcu < nvalid;
    const uint32_t blkA = luma ? mcu * 6u + (pr & 1u) : mcu * 6u + 4u, blkB = luma ? blkA + 2u : blkA + 1u;
    const int compA = luma ? 0 : 1, compB = luma ? 0 : 2;
    uint8_t* mid = s_mid + pr * C::kPair;
    int dcA = 0, dcB = 0;
    if (p.dc && sub == 0 && valid) {
        const int16_t* dc = p.dc + img * (p.coef_stride >> 6) + mcu0 * 6;
        dcA = __ldg(dc + blkA), dcB = __ldg(dc + blkB);
    }

    mbar_wait_wd(bar, 0);

    if (luma || !p.gray) {
        // ---- masks of the non-zero zig-zag groups: lane sub looks at group sub of both blocks ----
        const uint8_t* cA = s_coef + blkA * 128u;
        const uint32_t dAB = (blkB - blkA) * 128u;
        uint4 gA = make_uint4(0, 0, 0, 0), gB = gA;
        if (valid) gA = *reinterpret_cast<const uint4*>(cA + sub * 16u), gB = *reinterpret_cast<const uint4*>(cA + dAB + sub * 16u);
        if (sub == 0) {
            if (!p.dc) dcA = int(short(gA.x & 0xffffu)), dcB = int(short(gB.x & 0xffffu));
            else if (valid) {       // the fix-up phase reads the block from shared memory: put the DC coefficient in place
                *reinterpret_cast<int16_t*>(s_coef + blkA * 128u) = int16_t(dcA);
                *reinterpret_cast<int16_t*>(s_coef + blkB * 128u) = int16_t(dcB);
            }
            gA.x &= 0xffff0000u, gB.x &= 0xffff0000u;
        }
        const uint32_t balA = __ballot_sync(0xffffffffu, (gA.x | gA.y | gA.z | gA.w) != 0u);
        const uint32_t balB = __ballot_sync(0xffffffffu, (gB.x | gB.y | gB.z | gB.w) != 0u);
        // zig-zag positions 3..7 (the high half of word y, words z and w of group 0)
        const uint32_t bal37 = __ballot_sync(0xffffffffu, sub == 0u && (((gA.y | gB.y) >> 16) | gA.z | gA.w | gB.z | gB.w) != 0u);
        const uint32_t maskA = (balA >> (lane & 24)) & 0xffu, maskB = (balB >> (lane & 24)) & 0xffu;
        if (sub == 0 && valid) s_mask[blkA] = uint8_t(maskA), s_mask[blkB] = uint8_t(maskB);
        const int qA = int(p.qt[compA][0]), qB = int(p.qt[compB][0]);
        dcA = __shfl_sync(0xffffffffu, dcA, lane & 24), dcB = __shfl_sync(0xffffffffu, dcB, lane & 24);

        uint4 rowA, rowB;         // the 8 + 8 samples of row sub as int16 pairs
        bool wide;                // a sample of this row of the two blocks leaves the int16 range
        if ((balA | balB) == 0u) {
            // every block of the warp is DC-only
            const int ia = dc_only_value(dcA, qA), ib = dc_only_value(dcB, qB);
            const uint32_t va = uint32_t(ia) & 0xffffu, vb = uint32_t(ib) & 0xffffu;
            rowA = make_uint4(va * 0x10001u, va * 0x10001u, va * 0x10001u, va * 0x10001u);
            rowB = make_uint4(vb * 0x10001u, vb * 0x10001u, vb * 0x10001u, vb * 0x10001u);
            wide = valid && (wide_int(ia) || wide_int(ib));
            if (lane == 0) atomicAdd(p.guard_counter, 32ull * 16ull);
        } else {
            const bool pruned = ((balA | balB) & 0xfefefefeu) == 0u;      // nothing beyond zig-zag position 7 in the warp
            f32x2 d[8];           // samples of row sub of both blocks, level shift included
            f32x2 gs;             // per-block guard band
            if (pruned && bal37 == 0u) {
                // ---- nothing beyond zig-zag position 2 in the warp: the sample is a separable sum, row sub evaluated directly
                // (no column pass, no transpose).  FP32 order: ((F00 M00 + 128) + F10 Ly[sub]) + F01 Lx[x], one rounding per
                // step; its own guard band (Lg) ----
                const int cls = luma ? 0 : 1;
                uint2 wA, wB;     // zig-zag 0..3 of both blocks (F(0,1) is the high half of x, F(1,0) the low half of y)
                asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(wA.x), "=r"(wA.y) : "r"(smem_u32(cA)));
                asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(wB.x), "=r"(wB.y) : "r"(smem_u32(cA) + dAB));
                const f32x2 fd = pk2(float(dcA), float(dcB));
                const f32x2 fa = pk2(float(sx_hi(wA.x)), float(sx_hi(wB.x))), fb = pk2(float(sx_lo(wA.y)), float(sx_lo(wB.y)));
                const f32x2 m00 = __ldg(reinterpret_cast<const unsigned long long*>(&tab->M[cls][0][0]));
                const f32x2 ly = __ldg(reinterpret_cast<const unsigned long long*>(&tab->Ly[cls][sub]));
                const ulonglong2* lx = reinterpret_cast<const ulonglong2*>(&tab->Lx[cls][0]);
                const ulonglong2* lg = reinterpret_cast<const ulonglong2*>(&tab->Lg[cls][0]);
                const ulonglong2 x01 = __ldg(lx), x23 = __ldg(lx + 1), x45 = __ldg(lx + 2), x67 = __ldg(lx + 3), g01 = __ldg(lg), g23 = __ldg(lg + 1);
                const f32x2 base = fma2(fb, ly, add2(mul2(fd, m00), pk2(128.0f, 128.0f)));
                d[0] = fma2(fa, x01.x, base), d[1] = fma2(fa, x01.y, base), d[2] = fma2(fa, x23.x, base), d[3] = fma2(fa, x23.y, base);
                d[4] = fma2(fa, x45.x, base), d[5] = fma2(fa, x45.y, base), d[6] = fma2(fa, x67.x, base), d[7] = fma2(fa, x67.y, base);
                constexpr f32x2 kAbs = 0x7fffffff7fffffffull;
                gs = fma2(fd & kAbs, g01.x, fma2(fa & kAbs, g01.y, fma2(fb & kAbs, g23.x, g23.y)));
            } else {
                const uint32_t u = sub;
                // ---- column u: de-zig-zag, dequantise (x AAN input scale), guard-band sum ----
                gs = pk2(0.0f, 0.0f);
                {
                    const uint2 zo = __ldg(&tab->zoff[u]);
                    const int cls = luma ? 0 : 1;
                    const ulonglong2* mq = reinterpret_cast<const ulonglong2*>(&tab->M[cls][u][0]);
                    const ulonglong2* wq = reinterpret_cast<const ulonglong2*>(&tab->Wg[cls][u][0]);
                    const uint32_t base = smem_u32(cA);
#define JZ_LOAD_COEF(V, ZW, K, MM, WW)                                                                                   \
    {                                                                                                                     \
        const uint32_t ad = add_byte<K>(ZW, base);                                                                        \
        int ca, cb;                            /* (32-bit destinations: I2FP instead of the quarter-rate I2F.S16) */        \
        asm volatile("ld.shared.s16 %0, [%1];" : "=r"(ca) : "r"(ad));                                                     \
        asm volatile("ld.shared.s16 %0, [%1];" : "=r"(cb) : "r"(ad + dAB));                                               \
        const f32x2 f = pk2(float(ca), float(cb));                                                                        \
        d[V] = mul2(f, MM);                                                                                               \
        const f32x2 g = mul2(f, WW);                                                                                      \
        gs = add2(gs, pk2(fabsf(lo2(g)), fabsf(hi2(g))));                                                                 \
        }
                    const ulonglong2 m01 = __ldg(mq), m23 = __ldg(mq + 1), w01 = __ldg(wq), w23 = __ldg(wq + 1);
                    JZ_LOAD_COEF(0, zo.x, 0, m01.x, w01.x)
                    if (u == 0) {      // the DC coefficient is in registers (dense array or position 0 of the block)
                        const f32x2 f = pk2(float(dcA), float(dcB));
                        d[0] = mul2(f, m01.x);
                        const f32x2 g = mul2(f, w01.x);
                        gs = pk2(fabsf(lo2(g)), fabsf(hi2(g)));
                    }
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
                if (u == 0) d[0] = add2(d[0], pk2(128.0f, 128.0f));       // level shift rides on the DC term (gain 1 through the flowgraph)
                if (pruned) aan_idct8_in3_x2(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);
                else aan_idct8_x2(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);
#pragma unroll
                for (int y = 0; y < 8; ++y) *reinterpret_cast<f32x2*>(mid + y * C::kPairRow + u * 8u) = d[y];
                // per-block guard band: sum over the eight columns
                {
                    float ga = lo2(gs), gb = hi2(gs);
                    ga += __shfl_xor_sync(0xffffffffu, ga, 1), gb += __shfl_xor_sync(0xffffffffu, gb, 1);
                    ga += __shfl_xor_sync(0xffffffffu, ga, 2), gb += __shfl_xor_sync(0xffffffffu, gb, 2);
                    ga += __shfl_xor_sync(0xffffffffu, ga, 4), gb += __shfl_xor_sync(0xffffffffu, gb, 4);
                    gs = pk2(ga + 2e-5f, gb + 2e-5f);
                }
                __syncwarp();
                // ---- row sub of both blocks ----
                {
                    const ulonglong2* src = reinterpret_cast<const ulonglong2*>(mid + sub * C::kPairRow);
                    const ulonglong2 a = src[0], b = src[1], c = src[2], e = src[3];
                    d[0] = a.x, d[1] = a.y, d[2] = b.x, d[3] = b.y, d[4] = c.x, d[5] = c.y, d[6] = e.x, d[7] = e.y;
                }
                if (pruned) aan_idct8_in4_x2(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);
                else aan_idct8_x2(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);
            }
            // floor (low mantissa bits of v + 1.5 * 2^23, rounded down) and distance to the nearest integer
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
            wide = valid && fmaxf(va, vb) >= kWideSample;
            rowA = make_uint4(__byte_perm(ia[0], ia[1], 0x5410), __byte_perm(ia[2], ia[3], 0x5410), __byte_perm(ia[4], ia[5], 0x5410), __byte_perm(ia[6], ia[7], 0x5410));
            rowB = make_uint4(__byte_perm(ib[0], ib[1], 0x5410), __byte_perm(ib[2], ib[3], 0x5410), __byte_perm(ib[4], ib[5], 0x5410), __byte_perm(ib[6], ib[7], 0x5410));
            const bool dcoA = maskA == 0u, dcoB = maskB == 0u;
            const bool negA = ((rowA.x | rowA.y | rowA.z | rowA.w) & 0x80008000u) != 0u, negB = ((rowB.x | rowB.y | rowB.z | rowB.w) & 0x80008000u) != 0u;
            uint32_t exact = 0;
            if (dcoA) {
                const uint32_t va = uint32_t(dc_only_value(dcA, qA)) & 0xffffu;
                rowA = make_uint4(va * 0x10001u, va * 0x10001u, va * 0x10001u, va * 0x10001u);
                exact += 8;
            } else if ((ma < lo2(gs) || negA) && valid) {
                rowA = inv_row_slow(lo2(d[0]), lo2(d[1]), lo2(d[2]), lo2(d[3]), lo2(d[4]), lo2(d[5]), lo2(d[6]), lo2(d[7]), lo2(gs), blkA, int(sub), s_nfix, s_fix);
            }
            if (dcoB) {
                const uint32_t vb = uint32_t(dc_only_value(dcB, qB)) & 0xffffu;
                rowB = make_uint4(vb * 0x10001u, vb * 0x10001u, vb * 0x10001u, vb * 0x10001u);
                exact += 8;
            } else if ((mb < hi2(gs) || negB) && valid) {
                rowB = inv_row_slow(hi2(d[0]), hi2(d[1]), hi2(d[2]), hi2(d[3]), hi2(d[4]), hi2(d[5]), hi2(d[6]), hi2(d[7]), hi2(gs), blkB, int(sub), s_nfix, s_fix);
            }
            exact = __reduce_add_sync(0xffffffffu, valid ? exact : 0u);
            if (lane == 0 && exact) atomicAdd(p.guard_counter, (unsigned long long)exact);
        }
        if (__any_sync(0xffffffffu, wide) && lane == 0) s_nfix[1] = 1;
        // ---- hand the row over: luma samples to the tile, chroma samples as colour offsets ----
        if (luma) {
            uint8_t* dst = s_y + sub * C::kYRow + (mcu * 16u + (pr & 1u) * 8u) * 2u;
            *reinterpret_cast<uint4*>(dst) = rowA;
            *reinterpret_cast<uint4*>(dst + 8 * C::kYRow) = rowB;
        } else {
            // the (Cb, Cr) samples, interleaved; the colour offsets are derived from them by the threads of the colour phase
            // (the chroma lanes would otherwise keep the luma warps waiting at the barrier)
            const uint32_t cbw[4] = {rowA.x, rowA.y, rowA.z, rowA.w}, crw[4] = {rowB.x, rowB.y, rowB.z, rowB.w};
            uint32_t cc[8];
#pragma unroll
            for (int k = 0; k < 4; ++k) cc[2 * k] = __byte_perm(cbw[k], crw[k], 0x5410), cc[2 * k + 1] = __byte_perm(cbw[k], crw[k], 0x7632);
            uint4* cd = reinterpret_cast<uint4*>(s_cc + sub * C::kCcRow + mcu * 32u);
            cd[0] = make_uint4(cc[0], cc[1], cc[2], cc[3]), cd[1] = make_uint4(cc[4], cc[5], cc[6], cc[7]);
        }
    }
    __syncthreads();

    uint8_t* R = p.r + img * p.plane_stride;
    uint8_t* G = p.g + img * p.plane_stride;
    uint8_t* B = p.b + img * p.plane_stride;
    if (s_nfix[1]) {
        // a sample outside the int16 range: every pixel of the tile from the coefficients (DC in place), as the reference computes it
        for (uint32_t e = t; e < nvalid * 256u; e += C::kThreads) {
            const uint32_t m = e >> 8, py = (e >> 4) & 15u, px = e & 15u, gx = (mx0 + m) * 16u + px;
            if (gx < p.W) pixel420_ref(p, s_coef + m * 768u, 128u, px, py, (size_t(my) * 16 + py) * p.W + gx, R, G, B);
        }
        if (t == 0) atomicAdd(p.guard_counter, nvalid * 256ull);     // (JPEZYB200_STAT_GUARD_INV: exact-order pixels)
        return;
    }

    // ---- phase 1b: dense FP64 re-evaluation of the queue (guard-band samples) ----
    {
        const uint32_t nfix = *s_nfix;
        if (nfix) {
            const bool overflow = nfix > kFixCap;
            uint32_t exact_hits = 0;
            const uint32_t ntask = overflow ? nvalid * 6u * 8u : nfix * 8u;
            for (uint32_t task0 = 0; task0 < ntask; task0 += C::kThreads) {
                const uint32_t task = task0 + uint32_t(t);
                // entry = blk << 7 | sample; overflow: row (task & 7) of block (task >> 3), every sample
                const uint32_t e = task >= ntask ? 0u : (overflow ? ((task >> 3) << 7) : uint32_t(s_fix[task >> 3]));
                const uint32_t blk = e >> 7, s8 = task & 7u;
                const uint32_t m = blk / 6u, k = blk - m * 6u;
                const bool act = task < ntask && !(p.gray && k >= 4u);      // (uniform over the eight lanes of an entry)
                const int comp = k < 4u ? 0 : int(k) - 3;
                const int16_t* cz = reinterpret_cast<const int16_t*>(s_coef + blk * 128u);
                const int nlim = 8 * (32 - __clz(uint32_t(s_mask[blk]) | 1u));
                auto put = [&](int y, int x, int val) {
                    if (k < 4u) {
                        *reinterpret_cast<int16_t*>(s_y + ((k >> 1) * 8 + y) * C::kYRow + (m * 16u + (k & 1u) * 8u + x) * 2u) = int16_t(val);
                    } else {
                        int16_t* cc = reinterpret_cast<int16_t*>(s_cc + y * C::kCcRow + (m * 8u + x) * 4u);
                        cc[k - 4u] = int16_t(val);
                    }
                };
                if (overflow) {
                    if (act)
                        for (int x = 0; x < 8; ++x) put(int(s8), x, idct_fix(cz, p.qt[comp], nlim, x, int(s8), &exact_hits));
                } else {
                    const int s = int(e & 63u);
                    double part = act ? idct_fix_part(cz, p.qt[comp], int(s8), 8, nlim, s & 7, s >> 3) : 0.0;
                    part += __shfl_xor_sync(0xffffffffu, part, 1);
                    part += __shfl_xor_sync(0xffffffffu, part, 2);
                    part += __shfl_xor_sync(0xffffffffu, part, 4);
                    if (act && s8 == 0) put(s >> 3, s & 7, idct_fix_finish(part, cz, p.qt[comp], nlim, s & 7, s >> 3, &exact_hits));
                }
            }
            exact_hits = __reduce_add_sync(0xffffffffu, exact_hits);
            if (lane == 0 && exact_hits) atomicAdd(p.guard_counter, (unsigned long long)exact_hits);
            __syncthreads();
        }
    }

    // ---- phase 2: colour + planar stores; one thread per (row, MCU) ----
    if (t < T * 16) {
        const uint32_t ry = uint32_t(t) / T, m = uint32_t(t) % T;
        const uint32_t x0 = (mx0 + m) * 16u;
        if (!p.gray) {
            // colour offsets of chroma row ry / 2: this thread derives pairs 0..3 (even ry) or 4..7 (odd ry), the thread of the other
            // row of the pair -- T lanes away, same warp -- the other four
            const uint32_t h4 = (ry & 1u) * 4u;
            const uint4 ccq = *reinterpret_cast<const uint4*>(s_cc + (ry >> 1) * C::kCcRow + (m * 8u + h4) * 4u);
            const uint2 f0 = chroma_offsets_w(ccq.x), f1 = chroma_offsets_w(ccq.y), f2 = chroma_offsets_w(ccq.z), f3 = chroma_offsets_w(ccq.w);
            uint4* od = reinterpret_cast<uint4*>(s_off + (ry >> 1) * C::kOffRow + (m * 8u + h4) * 8u);
            od[0] = make_uint4(f0.x, f0.y, f1.x, f1.y), od[1] = make_uint4(f2.x, f2.y, f3.x, f3.y);
            __syncwarp();
        }
        if (m < nvalid) {
            const uint4 ya = *reinterpret_cast<const uint4*>(s_y + ry * C::kYRow + m * 32u);
            const uint4 yb = *reinterpret_cast<const uint4*>(s_y + ry * C::kYRow + m * 32u + 16u);
            const uint32_t yw[8] = {ya.x, ya.y, ya.z, ya.w, yb.x, yb.y, yb.z, yb.w};
            uint32_t ro[4], go[4], bo[4];
            if (p.gray) {
#pragma unroll
                for (int q4 = 0; q4 < 4; ++q4)
                    ro[q4] = go[q4] = bo[q4] = pack_sat_u8x4(sx_lo(yw[q4 * 2]), sx_hi(yw[q4 * 2]), sx_lo(yw[q4 * 2 + 1]), sx_hi(yw[q4 * 2 + 1]));
            } else {
                const uint4* op = reinterpret_cast<const uint4*>(s_off + (ry >> 1) * C::kOffRow + m * 64u);
                const uint4 o0 = op[0], o1 = op[1], o2 = op[2], o3 = op[3];
                const uint32_t oa[8] = {o0.x, o0.z, o1.x, o1.z, o2.x, o2.z, o3.x, o3.z};
                const uint32_t ob[8] = {o0.y, o0.w, o1.y, o1.w, o2.y, o2.w, o3.y, o3.w};
#pragma unroll
                for (int q4 = 0; q4 < 4; ++q4) {       // 4 pixels = 2 chroma pairs
                    const int c0 = q4 * 2, c1 = q4 * 2 + 1;
                    const int y0 = sx_lo(yw[c0]), y1 = sx_hi(yw[c0]), y2 = sx_lo(yw[c1]), y3 = sx_hi(yw[c1]);
                    if ((ob[c0] | ob[c1]) & 0x10000u) {
                        // rare: the reference's FP64 expressions, from the stored chroma samples
                        const uint32_t* pcc = reinterpret_cast<const uint32_t*>(s_cc + (ry >> 1) * C::kCcRow + (m * 8u + c0) * 4u);
                        const uint32_t w0 = pcc[0], w1 = pcc[1];
                        ro[q4] = colour_exact4r(y0, y1, y2, y3, w0, w1, 0);
                        go[q4] = colour_exact4r(y0, y1, y2, y3, w0, w1, 1);
                        bo[q4] = colour_exact4r(y0, y1, y2, y3, w0, w1, 2);
                    } else {
                        const int fr0 = sx_lo(oa[c0]), fg0 = sx_hi(oa[c0]), fb0 = sx_lo(ob[c0]);
                        const int fr1 = sx_lo(oa[c1]), fg1 = sx_hi(oa[c1]), fb1 = sx_lo(ob[c1]);
                        ro[q4] = pack_sat_u8x4(y0 + fr0, y1 + fr0, y2 + fr1, y3 + fr1);
                        go[q4] = pack_sat_u8x4(y0 + fg0, y1 + fg0, y2 + fg1, y3 + fg1);
                        bo[q4] = pack_sat_u8x4(y0 + fb0, y1 + fb0, y2 + fb1, y3 + fb1);
                    }
                }
            }
            const size_t rowoff = (size_t(my) * 16 + ry) * p.W;
            if ((p.W & 15u) == 0 && x0 + 16u <= p.W) {
                *reinterpret_cast<uint4*>(R + rowoff + x0) = make_uint4(ro[0], ro[1], ro[2], ro[3]);
                *reinterpret_cast<uint4*>(G + rowoff + x0) = make_uint4(go[0], go[1], go[2], go[3]);
                *reinterpret_cast<uint4*>(B + rowoff + x0) = make_uint4(bo[0], bo[1], bo[2], bo[3]);
            } else {
#pragma unroll           // (fully unrolled: a run-time index would send the three arrays to local memory)
                for (int i = 0; i < 16; ++i) {
                    if (x0 + i < p.W) {
                        R[rowoff + x0 + i] = uint8_t(ro[i >> 2] >> (8 * (i & 3)));
                        G[rowoff + x0 + i] = uint8_t(go[i >> 2] >> (8 * (i & 3)));
                        B[rowoff + x0 + i] = uint8_t(bo[i >> 2] >> (8 * (i & 3)));
                    }
                }
            }
        }
    }
}

}  // namespace jz
