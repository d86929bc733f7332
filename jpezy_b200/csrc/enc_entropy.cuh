// enc_entropy.cuh -- stage E3: quantised coefficients -> byte-stuffed Huffman segment.
//
// Replaces encode_huffman (src/encoder/jpezy_encoder.hpp:174-225) and the behaviour of the bit
// writer it drives (srook::io::jpeg::bofstream: MSB-first, 0xFF -> 0xFF 0x00 on bit writes, the
// final partial byte completed when the EOI marker is written, src/encoder/jpezy_writer.hpp:101-105).
//
// Pipeline (all integer, exact):
//   E3a k_block_bits   one thread per 8x8 block: DC delta, run-length symbols, bit length; CTA scan
//   E3b k_scan_tiles   per image: exclusive scan of the tile sums (64-bit bit offsets)
//   E3c k_scatter      one thread per block: re-generate the code words and OR them into the
//                      (zeroed) un-stuffed stream at the block's bit offset; pads the last byte
//   E3d k_ff_count / k_scan_ff / k_stuff_write   count 0xFF bytes, scan, copy with 0x00 inserted
//
// Restart intervals (JPEZYB200_OPT_RESTART_INTERVAL = R > 0, the kernels' RST = true instantiations; RST = false compiles to
// the restart-less pipeline): the DC predictors restart at 0 in every interval of R MCUs (T.81 F.1.2.3), and one more
// kernel, k_rst_intervals, runs between E3b and E3c.  It rounds every interval up to whole bytes and scans them into the
// byte base B_i of interval i in the un-stuffed stream (B_nint = its length).  k_scatter writes block b of interval i at
// bit 8 B_i + G(b) - G(first block of i), G being the block's offset without padding, and the last block of every interval
// writes that interval's pad bits.  The RSTn markers are not stored in the un-stuffed stream (the stuffing would put a 00
// behind their FF): k_stuff_write inserts FF D((i-1) mod 8) in front of byte B_i, i >= 1, so un-stuffed byte k lands at
// k + (0xFF bytes before k) + 2 (interval starts in 1..k).
#pragma once
#include "common.cuh"

namespace jz {

constexpr int kEntThreads = 256;   // blocks per tile
constexpr int kStuffThreads = 256;
constexpr int kStuffChunk = kStuffThreads * 16;

constexpr uint32_t kBadTile = 0xffffffffu;   // tile_sum of a tile that holds a coefficient without a baseline code

struct EntParams {
    const int16_t* coefs;
    size_t coef_stride;      // int16 per image
    const uint32_t* bmeta;   // nullptr, or [nimg][nblk] side information of the forward transform (FwdParams::bmeta)
    uint32_t nblk;           // blocks per image (6 * MCUs)
    uint32_t ntile;          // ceil(nblk / kEntThreads)
    uint32_t* blk_off;       // [nimg][nblk]   exclusive bit offset of the block within its tile
    uint32_t* tile_sum;      // [nimg][ntile]
    uint64_t* tile_base;     // [nimg][ntile]  exclusive bit offset of the tile within the image
    uint64_t* img_bits;      // [nimg]         total bits (before padding)
    uint64_t* img_bytes;     // [nimg]         stuffed byte count
    uint8_t* ustream;        // [nimg][uslot]  un-stuffed stream
    size_t uslot;            // bytes per image in ustream (multiple of 16)
    const HuffEncLut* lut;   // [2], or [nimg][2] with lut_stride = 2
    const int32_t* dc_init;  // [nimg][3] predictors of the first blocks (nullptr = 0), shards
    int pad_ones;
    // stuffing
    uint32_t* ff_sum;        // [nimg][nchunk]
    uint64_t* ff_base;       // [nimg][nchunk]
    uint32_t nchunk;         // chunks per image (capacity)
    uint8_t* out;            // [nimg][slot]
    size_t slot;
    uint64_t* out_bytes;     // [nimg] or nullptr
    uint64_t* out_bits;      // [nimg] or nullptr
    uint32_t lut_stride;     // HuffEncLut per image: 0 = every image reads lut[0..1], 2 = per-image tables (enc_huffopt.cuh)
};

// restart intervals: read by the RST = true kernels only (a kernel argument of its own, so that EntParams, and with it the
// layout of ShardParams, stays as the restart-less kernels have it)
struct RstParams {
    uint32_t rst;            // MCUs per interval
    uint32_t nint;           // intervals per image = ceil(MCUs / rst)
    uint64_t* base;          // [nimg][nint + 1]  byte base B_i of each interval in the un-stuffed stream, then its length
};

// index of the previous block of the same component in scan order, or -1; with RST, -1 also for the first block of each
// component in an interval of `rst` MCUs (the predictors restart at 0)
template <bool RST = false>
__device__ __forceinline__ long long prev_same_component(uint32_t b, uint32_t rst = 0)
{
    const uint32_t k = b % 6u;
    if (k >= 1 && k <= 3) return (long long)b - 1;
    if (b < 6) return -1;
    if (RST && (b / 6u) % rst == 0) return -1;
    return (long long)b - (k == 0 ? 3 : 6);
}

// the 64 coefficients of one block: eight 16-byte loads issued back to back (one exposed memory latency, not eight)
struct BlockRegs {
    int4 q[8];
    __device__ __forceinline__ void load(const int16_t* __restrict__ c)
    {
#pragma unroll
        for (int i = 0; i < 8; ++i) q[i] = __ldg(reinterpret_cast<const int4*>(c) + i);
    }
    // with the forward transform's side information: only the groups that hold a non-zero coefficient are fetched
    __device__ __forceinline__ void load(const int16_t* __restrict__ c, uint32_t meta)
    {
        const uint32_t m = meta >> 16;
#pragma unroll
        for (int i = 0; i < 8; ++i) q[i] = (m >> i) & 1u ? __ldg(reinterpret_cast<const int4*>(c) + i) : make_int4(0, 0, 0, 0);
        q[0].x = int((uint32_t(q[0].x) & 0xffff0000u) | (meta & 0xffffu));
    }
    __device__ __forceinline__ int dc() const { return int(short(q[0].x & 0xffff)); }
};
// block b of an image and the predictor of its DC coefficient
__device__ __forceinline__ void load_block(const int16_t* __restrict__ base, const uint32_t* __restrict__ meta, uint32_t b, long long pb,
                                           int init, BlockRegs& blk, int& pred)
{
    if (meta) {
        blk.load(base + size_t(b) * 64, __ldg(meta + b));
        pred = pb >= 0 ? int(short(__ldg(meta + pb) & 0xffffu)) : init;
    } else {
        blk.load(base + size_t(b) * 64);
        pred = pb >= 0 ? int(__ldg(base + size_t(pb) * 64)) : init;
    }
}

// Visit the code words of one block in stream order.  emit(bits, nbits), nbits <= 27.
// Returns false when a coefficient has no code in the baseline tables (DC difference of more than 11 bits, AC value of more
// than 10 bits: the reference throws std::runtime_error there, src/encoder/jpezy_encoder.hpp:186,207); the table indices are
// clamped so that such input -- possible through jpezyb200_entropy_encode_dev only -- never reads outside the tables.
template <class Emit>
__device__ __forceinline__ bool encode_block(const BlockRegs& blk, int dc_pred, const uint32_t* __restrict__ ac,
                                             const uint32_t* __restrict__ dc, Emit&& emit)
{
    bool ok = true;
    // DC (:180-191)
    {
        const int diff = blk.dc() - dc_pred;
        int cat = bit_length(abs(diff));
        if (cat > 11) ok = false, cat = 11;
        const uint32_t e = dc[cat];
        const uint32_t vbits = uint32_t(diff < 0 ? diff - 1 : diff) & ((1u << cat) - 1u);
        emit(((e >> 5) << cat) | vbits, int(e & 31u) + cat);
    }
    // AC (:194-224).  Per 8-coefficient group a mask of the non-zero ones; the loop visits only those, so the code of
    // emit() exists once per group instead of once per coefficient (the fully unrolled version was 78 KiB of code in
    // k_scatter) and sparse blocks cost a few iterations.
    int run = 0;
    const uint32_t zrl = ac[0xf0], eob = ac[0x00];
#pragma unroll
    for (int n8 = 0; n8 < 8; ++n8) {
        const int4 q = blk.q[n8];
        if (n8 && (q.x | q.y | q.z | q.w) == 0) { run += 8; continue; }
        const uint32_t w[4] = {uint32_t(q.x), uint32_t(q.y), uint32_t(q.z), uint32_t(q.w)};
        uint32_t m = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t ne = __vsetne2(w[i], 0u);      // 1 in every non-zero halfword
            m |= ((ne & 1u) | (ne >> 15)) << (2 * i);
        }
        if (n8 == 0) m &= ~1u;                            // the DC coefficient went first
        int next = n8 == 0 ? 1 : 0;                        // first position of the group not yet accounted for (0 of group 0 = DC)
        while (m) {
            const int h = __ffs(int(m)) - 1;
            m &= m - 1u;
            run += h - next;
            next = h + 1;
            const uint32_t ww = (h >> 1) == 0 ? w[0] : ((h >> 1) == 1 ? w[1] : ((h >> 1) == 2 ? w[2] : w[3]));
            const int v = (h & 1) ? (int(ww) >> 16) : int(short(ww & 0xffffu));
            while (run > 15) { emit(zrl >> 5, int(zrl & 31u)); run -= 16; }
            int s = bit_length(abs(v));
            if (s > 10) ok = false, s = 10;
            const uint32_t e = ac[(run << 4) | s];
            const uint32_t vbits = uint32_t(v < 0 ? v - 1 : v) & ((1u << s) - 1u);
            emit(((e >> 5) << s) | vbits, int(e & 31u) + s);
            run = 0;
        }
        run += 8 - next;
    }
    if (run) emit(eob >> 5, int(eob & 31u));   // coefficient 63 is zero <=> a run is pending
    return ok;
}

__device__ __forceinline__ uint32_t block_scan_excl(uint32_t v, uint32_t* s_warp, uint32_t* total)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) s_warp[wid] = x;
    __syncthreads();
    const int nw = blockDim.x >> 5;
    uint32_t base = 0, tot = 0;
    for (int w = 0; w < nw; ++w) {
        const uint32_t s = s_warp[w];
        if (w < wid) base += s;
        tot += s;
    }
    __syncthreads();
    *total = tot;
    return base + x - v;
}

__device__ __forceinline__ void load_lut(const HuffEncLut* __restrict__ g, uint32_t (*s_ac)[256], uint32_t (*s_dc)[16])
{
    for (int i = threadIdx.x; i < 512; i += blockDim.x) s_ac[i >> 8][i & 255] = g[i >> 8].ac[i & 255];
    if (threadIdx.x < 32) s_dc[threadIdx.x >> 4][threadIdx.x & 15] = g[threadIdx.x >> 4].dc[threadIdx.x & 15];
}

__device__ __forceinline__ uint64_t block_scan_excl64(uint64_t v, uint64_t* s_warp, uint64_t* total)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint64_t x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint64_t y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) s_warp[wid] = x;
    __syncthreads();
    const int nw = blockDim.x >> 5;
    uint64_t base = 0, tot = 0;
    for (int w = 0; w < nw; ++w) {
        const uint64_t s = s_warp[w];
        if (w < wid) base += s;
        tot += s;
    }
    __syncthreads();
    *total = tot;
    return base + x - v;
}

// ---- E3a ------------------------------------------------------------------------------------------
template <bool RST>
__global__ void __launch_bounds__(kEntThreads) k_block_bits(const EntParams p, const RstParams r)
{
    pdl_wait();
    __shared__ uint32_t s_ac[2][256];
    __shared__ uint32_t s_dc[2][16];
    __shared__ uint32_t s_warp[kEntThreads / 32];
    load_lut(p.lut + blockIdx.y * p.lut_stride, s_ac, s_dc);
    __syncthreads();
    const size_t img = blockIdx.y;
    const uint32_t b = blockIdx.x * kEntThreads + threadIdx.x;
    uint32_t bits = 0;
    bool bad = false;
    if (b < p.nblk) {
        const int16_t* base = p.coefs + img * p.coef_stride;
        const long long pb = prev_same_component<RST>(b, r.rst);
        const int cls = (b % 6u) >= 4;
        const int comp = (b % 6u) < 4 ? 0 : int(b % 6u) - 3;
        BlockRegs blk;
        int pred;
        load_block(base, p.bmeta ? p.bmeta + img * p.nblk : nullptr, b, pb, p.dc_init ? p.dc_init[img * 3 + comp] : 0, blk, pred);
        bad = !encode_block(blk, pred, s_ac[cls], s_dc[cls], [&](uint32_t, int n) { bits += uint32_t(n); });
    }
    uint32_t total;
    const uint32_t off = block_scan_excl(bits, s_warp, &total);
    if (b < p.nblk) p.blk_off[img * p.nblk + b] = off;
    // a coefficient without a code: the tile reports kBadTile, k_scan_tiles turns that into a bit count no slot can hold, and the
    // image ends like one that does not fit (scan_bytes = UINT64_MAX) instead of as a silently corrupt stream
    const int anybad = __syncthreads_or(bad ? 1 : 0);
    if (threadIdx.x == 0) p.tile_sum[img * p.ntile + blockIdx.x] = anybad ? kBadTile : total;
}

// ---- E3b: one CTA per image, 64-bit running carry ------------------------------------------------------
__global__ void __launch_bounds__(1024) k_scan_tiles(const EntParams p)
{
    pdl_wait();
    __shared__ uint32_t s_warp[32];
    __shared__ uint64_t s_carry;
    const size_t img = blockIdx.x;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t t0 = 0; t0 < p.ntile; t0 += 1024) {
        const uint32_t t = t0 + threadIdx.x;
        uint32_t v = t < p.ntile ? p.tile_sum[img * p.ntile + t] : 0u;
        const int bad = __syncthreads_or(v == kBadTile ? 1 : 0);
        if (bad) {
            if (threadIdx.x == 0) {
                p.img_bits[img] = 1ull << 62;
                if (p.out_bits) p.out_bits[img] = ~0ull;
            }
            return;
        }
        uint32_t total;
        const uint32_t off = block_scan_excl(v, s_warp, &total);   // < 1024 * 256 * 1700 bits: fits 32 bits
        const uint64_t carry = s_carry;
        if (t < p.ntile) p.tile_base[img * p.ntile + t] = carry + off;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        p.img_bits[img] = s_carry;
        if (p.out_bits) p.out_bits[img] = s_carry;
    }
}

// ---- restart intervals: one CTA per image, 64-bit running carry ------------------------------------------
// Interval i covers blocks [6 R i, 6 R (i + 1)); its length is G(first block of i + 1) - G(first block of i) bits, rounded
// up to bytes.  Writes B_i (and B_nint = the padded length) to rst_base and replaces img_bits with 8 B_nint, so the zeroing
// and stuffing kernels size the padded stream; scan_bits (out_bits, written by k_scan_tiles) stays the Huffman bit count.
__device__ __forceinline__ uint64_t block_bit_offset(const EntParams& p, size_t img, uint32_t b)
{
    return p.tile_base[img * p.ntile + b / kEntThreads] + p.blk_off[img * p.nblk + b];
}

__global__ void __launch_bounds__(1024) k_rst_intervals(const EntParams p, const RstParams r)
{
    pdl_wait();
    __shared__ uint64_t s_warp[32];
    const size_t img = blockIdx.x;
    const uint64_t bits = p.img_bits[img];
    if (bits >= (1ull << 62)) return;   // a coefficient without a code (k_scan_tiles): nothing to lay out
    const uint32_t per = 6u * r.rst;     // blocks per interval
    uint64_t* base = r.base + img * (size_t(r.nint) + 1);
    uint64_t carry = 0;
    for (uint32_t i0 = 0; i0 < r.nint; i0 += 1024) {
        const uint32_t i = i0 + threadIdx.x;
        uint64_t len = 0;
        if (i < r.nint) {
            const uint32_t b0 = i * per;
            const uint64_t g0 = block_bit_offset(p, img, b0);
            const uint64_t g1 = p.nblk - b0 > per ? block_bit_offset(p, img, b0 + per) : bits;
            len = (g1 - g0 + 7) / 8;
        }
        uint64_t total;
        const uint64_t off = block_scan_excl64(len, s_warp, &total);
        if (i < r.nint) base[i] = carry + off;
        carry += total;
    }
    // (every thread read img_bits before the first scan's barrier)
    if (threadIdx.x == 0) {
        base[r.nint] = carry;
        p.img_bits[img] = carry * 8;
    }
}

// ---- zero the part of the un-stuffed stream that will be written (grid-stride, data dependent) -----------
__global__ void __launch_bounds__(256) k_zero_ustream(const EntParams p)
{
    pdl_wait();
    const size_t img = blockIdx.y;
    const uint64_t bits = p.img_bits[img];
    uint64_t n16 = ((bits + 7) / 8 + 15) / 16 + 1;   // 16-byte units, one spare for the pad byte
    if (n16 > p.uslot / 16) n16 = p.uslot / 16;
    uint4* dst = reinterpret_cast<uint4*>(p.ustream + img * p.uslot);
    for (uint64_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n16; i += size_t(gridDim.x) * blockDim.x)
        dst[i] = make_uint4(0, 0, 0, 0);
}

// ---- E3c ------------------------------------------------------------------------------------------
template <bool RST>
__global__ void __launch_bounds__(kEntThreads) k_scatter(const EntParams p, const RstParams r)
{
    pdl_wait();
    __shared__ uint32_t s_ac[2][256];
    __shared__ uint32_t s_dc[2][16];
    load_lut(p.lut + blockIdx.y * p.lut_stride, s_ac, s_dc);
    __syncthreads();
    const size_t img = blockIdx.y;
    const uint32_t b = blockIdx.x * kEntThreads + threadIdx.x;
    if (b >= p.nblk) return;
    const uint64_t total = p.img_bits[img];
    if ((total + 7) / 8 + 4 > p.uslot) return;   // does not fit: reported by k_scan_ff
    const int16_t* base = p.coefs + img * p.coef_stride;
    const long long pb = prev_same_component<RST>(b, r.rst);
    const int cls = (b % 6u) >= 4;
    const int comp = (b % 6u) < 4 ? 0 : int(b % 6u) - 3;
    BlockRegs blk;
    int pred;
    load_block(base, p.bmeta ? p.bmeta + img * p.nblk : nullptr, b, pb, p.dc_init ? p.dc_init[img * 3 + comp] : 0, blk, pred);
    uint64_t pos = p.tile_base[img * p.ntile + blockIdx.x] + p.blk_off[img * p.nblk + b];
    if constexpr (RST) {   // from the interval's byte base instead of its unpadded bit offset
        const uint32_t i = b / (6u * r.rst);
        pos += 8 * r.base[img * (size_t(r.nint) + 1) + i] - block_bit_offset(p, img, i * 6u * r.rst);
    }
    uint32_t* out = reinterpret_cast<uint32_t*>(p.ustream + img * p.uslot) + (pos >> 5);
    uint64_t acc = 0;
    int n = int(pos & 31u);     // bits already occupied in the current word (not ours)
    auto flush_word = [&](uint32_t wbe) {
        if (wbe) atomicOr(out, __byte_perm(wbe, 0, 0x0123));
        ++out;
    };
    auto emit = [&](uint32_t bits, int nb) {
        acc = (acc << nb) | bits;
        n += nb;
        if (n >= 32) {
            n -= 32;
            flush_word(uint32_t(acc >> n));
            acc &= (1ull << n) - 1ull;
        }
    };
    encode_block(blk, pred, s_ac[cls], s_dc[cls], emit);
    if constexpr (RST) {
        // the last block of every interval completes the interval's last byte (n = where the block's bits end, modulo 32)
        if (((b + 1) % (6u * r.rst) == 0 || b == p.nblk - 1) && p.pad_ones) {
            const int padn = (8 - (n & 7)) & 7;
            if (padn) emit((1u << padn) - 1u, padn);
        }
    } else if (b == p.nblk - 1 && p.pad_ones) {   // complete the last byte with 1-bits (write_eoi)
        const int padn = int((8u - uint32_t(total & 7u)) & 7u);
        if (padn) emit((1u << padn) - 1u, padn);
    }
    if (n) flush_word(uint32_t(acc << (32 - n)));
}

// ---- E3d ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t count_ff16(const uint4 v, uint64_t first_byte, uint64_t nbytes)
{
    // number of 0xFF bytes among the valid bytes [first_byte, first_byte+16) /\ [0, nbytes)
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const uint32_t byte = (w[i >> 2] >> ((i & 3) * 8)) & 0xffu;
        c += (byte == 0xffu && first_byte + i < nbytes) ? 1u : 0u;
    }
    return c;
}

__global__ void __launch_bounds__(kStuffThreads) k_ff_count(const EntParams p)
{
    pdl_wait();
    __shared__ uint32_t s_warp[kStuffThreads / 32];
    const size_t img = blockIdx.y;
    const uint64_t nbytes = (p.img_bits[img] + 7) / 8;
    if (nbytes + 4 > p.uslot) return;
    const uint32_t nch = uint32_t((nbytes + kStuffChunk - 1) / kStuffChunk);
    const uint4* src = reinterpret_cast<const uint4*>(p.ustream + img * p.uslot);
    for (uint32_t ch = blockIdx.x; ch < nch; ch += gridDim.x) {
        const uint64_t i16 = uint64_t(ch) * kStuffThreads + threadIdx.x;
        uint32_t c = 0;
        if (i16 * 16 < nbytes) c = count_ff16(src[i16], i16 * 16, nbytes);
        uint32_t total;
        block_scan_excl(c, s_warp, &total);
        if (threadIdx.x == 0) p.ff_sum[img * p.nchunk + ch] = total;
    }
}

template <bool RST>
__global__ void __launch_bounds__(1024) k_scan_ff(const EntParams p, const RstParams r)
{
    pdl_wait();
    __shared__ uint32_t s_warp[32];
    __shared__ uint64_t s_carry;
    const size_t img = blockIdx.x;
    const uint64_t nbytes = (p.img_bits[img] + 7) / 8;
    if (nbytes + 4 > p.uslot) {
        if (threadIdx.x == 0 && p.out_bytes) p.out_bytes[img] = ~0ull;
        return;
    }
    const uint32_t nch = uint32_t((nbytes + kStuffChunk - 1) / kStuffChunk);
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t c0 = 0; c0 < nch; c0 += 1024) {
        const uint32_t c = c0 + threadIdx.x;
        const uint32_t v = c < nch ? p.ff_sum[img * p.nchunk + c] : 0u;
        uint32_t total;
        const uint32_t off = block_scan_excl(v, s_warp, &total);
        const uint64_t carry = s_carry;
        if (c < nch) p.ff_base[img * p.nchunk + c] = carry + off;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const uint64_t outb = nbytes + s_carry + (RST ? 2ull * (r.nint - 1) : 0ull);   // (RST: the markers)
        if (p.out_bytes) p.out_bytes[img] = outb <= p.slot ? outb : ~0ull;
        p.img_bytes[img] = outb;
    }
}

template <bool RST>
__global__ void __launch_bounds__(kStuffThreads) k_stuff_write(const EntParams p, const RstParams r)
{
    pdl_wait();
    __shared__ uint32_t s_warp[kStuffThreads / 32];
    const size_t img = blockIdx.y;
    const uint64_t nbytes = (p.img_bits[img] + 7) / 8;
    if (nbytes + 4 > p.uslot) return;
    if (p.img_bytes[img] > p.slot) return;   // stuffed size exceeds the caller's slot
    const uint32_t nch = uint32_t((nbytes + kStuffChunk - 1) / kStuffChunk);
    const uint4* src = reinterpret_cast<const uint4*>(p.ustream + img * p.uslot);
    uint8_t* dst = p.out + img * p.slot;
    for (uint32_t ch = blockIdx.x; ch < nch; ch += gridDim.x) {
        const uint64_t i16 = uint64_t(ch) * kStuffThreads + threadIdx.x;
        uint4 v = make_uint4(0, 0, 0, 0);
        uint32_t c = 0;
        const bool live = i16 * 16 < nbytes;
        if (live) { v = src[i16]; c = count_ff16(v, i16 * 16, nbytes); }
        uint32_t total;
        const uint32_t off = block_scan_excl(c, s_warp, &total);
        if (!live) continue;
        uint64_t o = i16 * 16 + p.ff_base[img * p.nchunk + ch] + off;
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        if constexpr (RST) {
            // the first interval j >= 1 that starts at or after this group (B strictly increasing, B_nint = nbytes), and the
            // markers in front of the group
            const uint64_t* B = r.base + img * (size_t(r.nint) + 1);
            const uint64_t k0 = i16 * 16;
            uint32_t lo = 1, hi = r.nint;
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (B[mid] < k0) lo = mid + 1;
                else hi = mid;
            }
            o += 2ull * (lo - 1);
            uint64_t next = B[lo];
            for (int i = 0; i < 16; ++i) {
                const uint64_t k = k0 + i;
                if (k >= nbytes) break;
                if (k == next) {   // RST((j - 1) mod 8) in front of interval j's first byte
                    dst[o++] = 0xffu;
                    dst[o++] = uint8_t(0xd0u + ((lo - 1) & 7u));
                    next = B[++lo];
                }
                const uint8_t byte = uint8_t(w[i >> 2] >> ((i & 3) * 8));
                dst[o++] = byte;
                if (byte == 0xffu) dst[o++] = 0;
            }
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                if (i16 * 16 + i >= nbytes) break;
                const uint8_t byte = uint8_t(w[i >> 2] >> ((i & 3) * 8));
                dst[o++] = byte;
                if (byte == 0xffu) dst[o++] = 0;
            }
        }
    }
}

}  // namespace jz
