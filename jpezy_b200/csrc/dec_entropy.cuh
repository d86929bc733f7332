// dec_entropy.cuh -- stage D1: byte-stuffed Huffman segment -> quantised coefficients.
//
// Replaces decode_huffman / decode_huffman_impl (src/decoder/jpezy_decoder.hpp:583-642) and the bit
// reader behind them (srook::io::jpeg::bifstream: MSB-first, the 0x00 after 0xFF dropped).  The
// reference decodes one bit at a time, strictly sequentially; jpezy's encoder writes no restart
// markers, so the whole image is ONE entropy-coded segment.  It is decoded in parallel with the
// self-synchronising scheme of Weissenberger & Schmidt: the un-stuffed stream is cut into
// subsequences of `sub_bits` bits, every thread decodes its subsequence from a guessed decoder
// state, then repeatedly re-decodes from its predecessor's end state until all end states are a
// fixed point (Huffman codes re-synchronise after a few code words).  A prefix sum of the
// per-subsequence block counts gives each subsequence its first block index; a last pass decodes
// once more and writes the coefficients; DC differences are turned into absolute values by a
// per-component prefix sum.
//
//   D0  k_unstuff_count / k_scan_u32 / k_unstuff_write     drop stuffed zeros (compaction scan)
//   D1a k_sync_decode (round 0, then rounds until no end state changes)
//   D1b k_scan_u32 over block counts
//   D1c k_write_coefs
//   D1d k_dc_sum / k_scan_dc / k_dc_apply                  DC prediction = prefix sum per component
#pragma once
#include "common.cuh"

namespace jz {

constexpr int kDecThreads = 256;
constexpr int kMaxSyncRounds = 66;   // entries of DecParams::changed
constexpr int kLutBits = 10;

// compact canonical decoder table for one DHT table, built on the host; entry layout:
//   bits 0..4   bits to consume: code length + size of the value field (+ a folded end-of-block code); bits 5..7 are zero
//               (the bit reader adds whole entries to its shift count and relies on that)
//   bits 8..15  advance of the zig-zag index z.  DC tables: 1; AC tables: run + 1; end-of-block: 64, so that z + dz >= 64
//               closes the block in both cases (ZRL = (15, 0) advances by 16 like the generic path of the reference,
//               src/decoder/jpezy_decoder.hpp:611-622).
//               64 + (run + 1): the end-of-block code of the block's AC table follows inside the kLutBits window and is
//               consumed with this symbol -- one table access instead of two for "DC difference, EOB" and
//               "coefficient, EOB" (most blocks of photographic content).  Not valid when the symbol itself fills the
//               block (then z + dz >= 128: the bits that look like EOB belong to the next block); the decoders turn the
//               entry back into the plain one with bits 25..28.
//               255 (kEntryNone, consume = 0): no code of at most kLutBits bits starts here -> HuffSlow.
//   bits 16..20 code length, bits 21..24 size (value extraction in the writing pass)
//   bits 25..28 length of the folded end-of-block code
constexpr uint32_t kEntryNone = 255u << 8;
__host__ __device__ inline uint32_t huff_entry(uint32_t len, uint32_t sym, bool ac)
{
    const uint32_t size = sym & 15u, run = sym >> 4;
    const uint32_t dz = !ac ? 1u : (sym == 0u ? 64u : run + 1u);
    return (len + size) | (dz << 8) | (len << 16) | (size << 21);
}
// the plain entry of a folded one
__host__ __device__ inline uint32_t unfold_entry(uint32_t e) { return e - ((e >> 25) & 15u) - (64u << 8); }
struct HuffSlow {                  // codes longer than kLutBits
    int32_t maxcode[18];           // maxcode[len] (left-aligned compare uses plain codes), -1 = none
    int32_t valptr[17];            // index into vals of the first code of this length minus its code
    int32_t pad_;                  // keeps sizeof(HuffDecTab) a multiple of 16
    uint8_t vals[256];
};
struct HuffDecTab {
    uint32_t fast[1 << kLutBits];  // indexed by the next kLutBits bits
    HuffSlow slow;                 // slow.pad_ = 1 for AC tables
};
static_assert(sizeof(HuffSlow) % 4 == 0 && sizeof(HuffDecTab) % 16 == 0, "copied to shared memory in words / 16-byte chunks");
// the four tables of a scan as the kernels keep them in shared memory
struct DecTabs {
    uint32_t fast[4][1 << kLutBits];
    HuffSlow slow[4];
    // per block position b of the MCU (decode_span): x = shared address of the AC table of block b, y = shared address of the DC table
    // of the block after b, z = shared address of the record of that block, w = b
    uint4 binfo[16];
};

struct DecParams {
    // geometry
    uint32_t nblk;            // blocks per image
    uint32_t nmcu;
    uint32_t nb;              // blocks per MCU (sum of H*V over the components: 1, 3, 4 or 6)
    uint32_t ny;              // of which luma (component 0); the others are one block each and use the class-1 tables
    // stuffed input
    const uint8_t* scan;      // [nimg][slot]
    size_t slot;
    const uint64_t* scan_bytes;   // device copy of the host array [nimg]
    uint64_t inline_bytes[8];     // ninline != 0 (small batches): the sizes travel as kernel arguments and k_unstuff_count
    uint32_t ninline;             // fills scan_bytes itself -- no host-to-device copy in front of the first kernel
    const uint64_t* ext_bytes;    // != nullptr: the lengths are read from this device array (jpezyb200_decode_batch_dev2); k_unstuff_count
                                  // copies them into scan_bytes, refusing (length 0, JPEZYB200_ECAPACITY) what exceeds max_bytes
    uint64_t max_bytes;           // capacity the launch was sized for
    // un-stuffed stream
    uint8_t* ustream;         // [nimg][uslot]  (uslot multiple of 16, 32 bytes of zero slack)
    size_t uslot;
    uint32_t nchunk;          // 4 KiB chunks per image (capacity)
    uint32_t* chunk_cnt;      // [nimg][nchunk] kept bytes per chunk
    uint64_t* chunk_base;     // [nimg][nchunk]
    uint64_t* ubytes;         // [nimg] un-stuffed byte count
    // restart intervals (DRI, src/decoder/jpezy_decoder.hpp:152-163,400-404): 0 = none
    uint32_t dri;             // MCUs per restart interval
    uint32_t nseg;            // restart segments per image = ceil(nmcu / dri)
    uint32_t* chunk_mcnt;     // [nimg][nchunk] RSTn markers per chunk
    uint64_t* chunk_mbase;    // [nimg][nchunk]
    uint64_t* nmarkers;       // [nimg]
    uint64_t* seg_start;      // [nimg][nseg + 1] first un-stuffed byte of every segment (segment 0: 0)
    // synchronisation
    uint32_t sub_bits;        // subsequence length in bits (128, 256 or 512)
    uint32_t cta_own;         // subsequences a CTA of k_sync_decode / k_write_coefs owns: its threads minus kDecWarm (96 or 224)
    uint32_t nsub;            // subsequences per image (capacity)
    uint32_t* sub_state;      // [nimg][nsub] packed end state of every subsequence
    uint32_t* state_a;        // [nimg][ncta] CTA tail states, double buffered across launches
    uint32_t* state_b;
    uint32_t* sub_blk;        // [nimg][nsub] exclusive prefix of block counts
    unsigned long long* changed;   // [rounds + 1] number of end states that changed in launch k (k >= 1); [0]: CTA boundaries at which
                                   // launch 0 found its warm-up result different from the previous CTA's tail; zeroed per call
    uint32_t* cta_flag;            // [nimg][ncta] set when a CTA of launch 0 has published its tail; zeroed per call (k_unstuff_count)
    uint32_t nflag;                // nimg * ncta
    uint32_t rounds;          // launches 1..rounds of k_sync_decode are enqueued after launch 0
    uint32_t rounds_host;     // launches the host-driven loop needed (rounds == 0)
    unsigned long long* rounds_stat;   // receives the number of launches that did work
    unsigned long long* iters_stat;    // [2] max / sum over CTAs of the shared-memory iterations of launch 0
    // tables: [0]=DC sel by comp class 0, [1]=DC class 1, [2]=AC class 0, [3]=AC class 1
    const HuffDecTab* tabs;
    // output
    int16_t* coefs;           // [nimg][nblk*64]
    size_t coef_stride;
    int32_t* status;          // [nimg] or nullptr
    // DC scan: the differences are written to a dense array (2 bytes per block) instead of coefficient 0 of every block,
    // so that the prefix sums read 12 contiguous bytes per MCU and not one 32-byte sector per block
    int16_t* dcd;             // [nimg][nblk] DC differences, then (k_dc_apply, in place) the DC coefficients
    uint32_t dc_dense;        // != 0: the DC coefficients stay in dcd only (the inverse transform reads them from there)
    int32_t* dc_part;         // [nimg][ndc_tiles][3]
    uint32_t ndc_tiles;
};

// packed end state: overshoot(6) | b(3) | z(6) | nblocks(12) | valid(1)
__device__ __forceinline__ uint32_t pack_state(uint32_t over, uint32_t b, uint32_t z, uint32_t n)
{
    return (over & 63u) | (b << 6) | (z << 9) | (min(n, 4095u) << 15);
}
constexpr uint32_t kStateSyncMask = (1u << 15) - 1u;   // (overshoot, b, z)

// ---- bit reader over the CTA's span of the un-stuffed stream, staged in shared memory ---------------------
// The span holds the CTA's kDecThreads subsequences plus kSpanSlack bytes of look-ahead, as raw bytes (big-endian
// bit order); positions are bits relative to the span start.  The word after the buffered ones is always
// pre-loaded, so that a refill costs two shifts and no shared-memory latency on the critical path.
constexpr int kSpanSlack = 64;
struct BitBuf {
    const uint32_t* w;   // next word to pre-load (shared memory)
    uint64_t buf;        // left-aligned
    uint32_t nxt;        // pre-loaded, byte-swapped word that follows the buffered bits
    int n;               // valid bits in buf
    uint32_t pos;        // bit position of the first bit of buf, relative to the span
    __device__ __forceinline__ void init(const uint32_t* span, uint32_t p)
    {
        w = span + (p >> 5);
        const uint32_t a = __byte_perm(w[0], 0, 0x0123), b = __byte_perm(w[1], 0, 0x0123);
        nxt = __byte_perm(w[2], 0, 0x0123);
        w += 3;
        const uint32_t sh = p & 31u;
        buf = ((uint64_t(a) << 32) | b) << sh;
        n = 64 - int(sh);
        pos = p;
    }
    __device__ __forceinline__ void refill()   // guarantees n >= 32
    {
        if (n < 32) {
            buf |= uint64_t(nxt) << (32 - n);
            n += 32;
            nxt = __byte_perm(*w++, 0, 0x0123);
        }
    }
    __device__ __forceinline__ uint32_t peek32() const { return uint32_t(buf >> 32); }
    __device__ __forceinline__ void skip(int k) { buf <<= k; n -= k; pos += k; }
};

__device__ __noinline__ uint32_t huff_lookup_slow(const HuffSlow* __restrict__ t, uint32_t bits32)
{
#pragma unroll 1
    for (int len = kLutBits + 1; len <= 16; ++len) {
        const int32_t code = int32_t(bits32 >> (32 - len));
        if (code <= t->maxcode[len]) return huff_entry(uint32_t(len), t->vals[(code + t->valptr[len]) & 255], t->pad_ != 0);
    }
    return 0;
}

// ---- the reader of the synchronisation / writing passes ------------------------------------------------------
// A thread's decode rate is set by the number of instructions per symbol (one warp per scheduler issues them in order,
// ~4 cycles apart when they depend on each other), so the loop below is written to need few:
//  * the span is staged as byte-swapped words; two of them (hi, lo) are the bit window, a third is pre-loaded; the
//    shift count is a running sum of whole table entries (the funnel shift looks at its low 5 bits only, bit 5 flipping
//    says "one word used up"), the exact position is kept on the side for the loop bound;
//  * shared memory is addressed with 32-bit shared-space addresses (no generic-address arithmetic in the loop);
//  * the next symbol comes from the AC table of the block's class or, if this symbol closes the block, from the DC table
//    of the next block's class: both words are fetched as soon as the window is known, the block-end test selects.
// (lds32: common.cuh)
struct FastBits {
    uint32_t wa;         // shared address of the word after nx
    uint32_t hi, lo, nx; // window words i, i + 1 and the pre-loaded word i + 2
    uint32_t acc;        // low 5 bits: bits of hi already consumed; bit 5 flips when a word is used up; rest: junk
    uint32_t pk;         // the next 32 bits
    uint32_t pos;        // bit position of pk, relative to the span
    __device__ __forceinline__ void init(uint32_t span_saddr, uint32_t p)
    {
        const uint32_t a = span_saddr + ((p >> 5) << 2);
        hi = lds32(a), lo = lds32(a + 4), nx = lds32(a + 8);
        wa = a + 12;
        acc = p & 31u;
        pk = __funnelshift_l(lo, hi, acc);
        pos = p;
    }
    // drop the bits of table entry e (<= 31, bits 5..7 of e are zero)
    __device__ __forceinline__ void consume(uint32_t e)
    {
        const uint32_t a2 = acc + e;
        if ((a2 ^ acc) & 32u) {
            hi = lo, lo = nx;
            nx = lds32(wa);
            wa += 4;
        }
        acc = a2;
        pk = __funnelshift_l(lo, hi, a2);
        pos += e & 31u;
    }
};

// Decode from (br.pos, b, z) until br.pos >= end (or >= limit); positions are relative to the span.  With kWrite the
// coefficients that carry a value field are stored (the buffer is pre-zeroed), block ordinals start at blk.
// Tables: T->fast[0] = DC class 0 (luma), [1] = DC class 1, [2] = AC class 0, [3] = AC class 1 (contiguous).
//
// One thread decodes one symbol after the other (ncu: ~110 cycles per symbol in the first version, the serial chain of the
// synchronisation passes).  What sets the rate is the dependency chain  table word -> shift count -> bit window -> table address
// -> table word,  every branch that must resolve before the next instruction may issue, and the instructions per symbol (one
// warp per scheduler issues them in order).  So:
//  * the symbol is consumed speculatively, as a plain symbol, into temporaries, and the table load of the NEXT symbol is issued
//    before anything is tested; "not a plain symbol" (code longer than kLutBits, folded end-of-block that does not apply) and "end
//    of the span" are tested while that load is in flight; the first commits nothing, corrects the entry and starts over;
//  * both candidate windows (word boundary crossed or not) are shifted in parallel and one select picks, instead of selecting
//    the words first; the table of the next symbol (AC of this block / DC of the next) is chosen from the zig-zag position
//    while the window is being computed, so one load suffices and its result is the next entry without a select;
//  * block bookkeeping (next block, its tables) comes from an 8-byte record per block position in shared memory.
template <bool kWrite>
__device__ __forceinline__ void decode_span(FastBits& br, uint32_t& b, uint32_t& z, uint32_t& nblocks, const uint32_t end,
                                            const uint32_t limit, const DecTabs* __restrict__ T, int16_t* __restrict__ out,
                                            int16_t* __restrict__ dcd, uint64_t blk, const uint64_t nblk, int* corrupt,
                                            const uint32_t nb, const uint32_t ny)
{
    (void)nb, (void)ny;
    const uint32_t stop = end < limit ? end : limit;
    if (!(br.pos < stop)) return;
    uint32_t tab, binfo;       // (opaque to the compiler, which would otherwise re-derive the shared-window addresses per symbol)
    asm volatile("mov.u32 %0, %1;" : "=r"(tab) : "r"(uint32_t(__cvta_generic_to_shared(&T->fast[0][0]))));
    asm volatile("mov.u32 %0, %1;" : "=r"(binfo) : "r"(uint32_t(__cvta_generic_to_shared(&T->binfo[0]))));
    constexpr uint32_t kTab = 4u << kLutBits;                          // bytes per table
    static_assert(kLutBits == 10, "the shift count in the step below");
    uint32_t w0 = br.hi, w1 = br.lo, w2 = br.nx, wa = br.wa, acc = br.acc, pk = br.pk, pos = br.pos;
    // the record of the current block position: AC table of this block, DC table of the next block, record of the next block
    uint32_t pb = binfo + 16u * b, t_cont, t_new, pbn;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%3];\n\tld.shared.u32 %2, [%3+8];" : "=r"(t_cont), "=r"(t_new), "=r"(pbn) : "r"(pb));
    uint32_t e = lds32((z == 0u ? t_cont - 2u * kTab : t_cont) + ((pk >> (32 - kLutBits)) << 2));
    // one symbol; returns 0 = go on, 1 = the span is done, 2 = not a plain symbol (nothing committed)
    auto step = [&]() -> int {
        const uint32_t dz = __byte_perm(e, 0, 0x4441);
        const uint32_t zs = z + dz;
        const uint32_t a2 = acc + e;
        const bool endb = zs >= 64u;
        const uint32_t tsel = endb ? t_new : t_cont;
        // (spelled out: left to itself the compiler puts the word-boundary test in front of the shift and three more
        // instructions on the chain)
        uint32_t pk2, en, crossw;
        asm volatile(
            "{\n\t.reg .pred c;\n\t.reg .b32 x, pa, pb, i, ad;\n\t"
            "xor.b32 x, %3, %4;\n\t"
            "and.b32 %2, x, 32;\n\t"
            "setp.ne.u32 c, %2, 0;\n\t"
            "shf.l.wrap.b32 pa, %6, %5, %3;\n\t"
            "shf.l.wrap.b32 pb, %7, %6, %3;\n\t"
            "selp.b32 %0, pb, pa, c;\n\t"
            "shr.u32 i, %0, 22;\n\t"
            "mad.lo.u32 ad, i, 4, %8;\n\t"
            "ld.shared.u32 %1, [ad];\n\t}"
            : "=r"(pk2), "=r"(en), "=r"(crossw)
            : "r"(a2), "r"(acc), "r"(w0), "r"(w1), "r"(w2), "r"(tsel)
            : "memory");
        const bool cross = crossw != 0u;
        uint32_t w3 = w2;
        if (cross) w3 = lds32(wa);
        if (zs >= 128u) return 2;
        // commit
        const uint32_t w = pk;
        w0 = cross ? w1 : w0, w1 = cross ? w2 : w1, w2 = w3;
        wa += crossw >> 3;
        acc = a2, pk = pk2;
        pos += e & 31u;
        if (kWrite) {
            const uint32_t len = (e >> 16) & 31u, sz = (e >> 21) & 15u;
            const uint32_t k = z + ((dz - 1u) & 63u);          // zig-zag index of this coefficient
            if (k > 63u && dz != 64u) {                        // run past the end of the block (src/decoder/jpezy_decoder.hpp:619)
                if (corrupt) *corrupt = 1;
            } else if (sz && blk < nblk) {
                const uint32_t vbits = (w << len) >> (32 - sz);
                int v = int(vbits);
                if (!(vbits & (1u << (sz - 1)))) v -= (1 << sz) - 1;
                if (z == 0u) dcd[blk] = int16_t(v);                // DC difference: dense side array (k_dc_sum / k_dc_apply)
                else out[blk * 64 + k] = int16_t(v);
            }
        }
        z = endb ? 0u : zs;
        pb = endb ? pbn : pb;
        nblocks += endb ? 1u : 0u;
        blk += endb ? 1u : 0u;
        e = en;
        if (kWrite && blk >= nblk) return 1;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%3];\n\tld.shared.u32 %2, [%3+8];" : "=r"(t_cont), "=r"(t_new), "=r"(pbn) : "r"(pb));
        return pos >= stop ? 1 : 0;
    };
    for (;;) {
        int r;
        for (;;) {             // (two symbols per trip: the compiler renames the loop-carried values instead of copying them)
            if ((r = step())) break;
            if ((r = step())) break;
        }
        if (r == 1) break;
        // not a plain symbol
        const uint32_t t_cur = z == 0u ? t_cont - 2u * kTab : t_cont;
        if ((e & 0xff00u) == 0xff00u) {      // code longer than kLutBits, or none
            e = huff_lookup_slow(T->slow + ((t_cur - tab) / kTab), pk);
            if (e == 0u) {     // no such code: only legal while speculating.  One bit is dropped, the state stays
                if (kWrite && corrupt) *corrupt = 1;
                const uint32_t a1 = acc + 1u;
                if ((a1 ^ acc) & 32u) {
                    w0 = w1, w1 = w2, w2 = lds32(wa);
                    wa += 4u;
                }
                acc = a1;
                pk = __funnelshift_l(w1, w0, a1);
                pos += 1u;
                e = lds32(t_cur + ((pk >> (32 - kLutBits)) << 2));
                if (pos >= stop) break;
            }
        } else {               // the symbol fills the block itself: the bits that look like EOB are the next block's
            e = unfold_entry(e);
        }
    }
    b = lds32(pb + 12u);
    br.hi = w0, br.lo = w1, br.nx = w2, br.wa = wa, br.acc = acc, br.pk = pk, br.pos = pos;
}

__device__ __forceinline__ void load_dec_tabs(const HuffDecTab* __restrict__ tabs, DecTabs* __restrict__ T, uint32_t nb, uint32_t ny)
{
    if (threadIdx.x < 16) {
        const uint32_t b = threadIdx.x, bn = b + 1u >= nb ? 0u : b + 1u;
        const uint32_t base = uint32_t(__cvta_generic_to_shared(&T->fast[0][0]));
        T->binfo[b] = make_uint4(base + (2u + (b >= ny ? 1u : 0u)) * (4u << kLutBits), base + (bn >= ny ? 1u : 0u) * (4u << kLutBits),
                                 uint32_t(__cvta_generic_to_shared(&T->binfo[bn])), b);
    }
    constexpr int kFast16 = (1 << kLutBits) * 4 / 16, kSlowW = int(sizeof(HuffSlow) / 4);
    // eight loads in flight per thread: the tables come out of L2 at its latency, not at eight times that
    for (int i0 = threadIdx.x; i0 < 4 * kFast16; i0 += 8 * blockDim.x) {
        uint4 v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int i = i0 + k * int(blockDim.x);
            if (i < 4 * kFast16) v[k] = __ldg(reinterpret_cast<const uint4*>(tabs[i / kFast16].fast) + i % kFast16);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int i = i0 + k * int(blockDim.x);
            if (i < 4 * kFast16) reinterpret_cast<uint4*>(T->fast[i / kFast16])[i % kFast16] = v[k];
        }
    }
    for (int i = threadIdx.x; i < 4 * kSlowW; i += blockDim.x)
        reinterpret_cast<uint32_t*>(&T->slow[i / kSlowW])[i % kSlowW] = __ldg(reinterpret_cast<const uint32_t*>(&tabs[i / kSlowW].slow) + i % kSlowW);
}

// stage the CTA's span of the un-stuffed stream: bytes [byte0, byte0 + span_bytes + kSpanSlack), 16-byte chunks, as
// byte-swapped words (FastBits)
// (the stream buffer carries >= 128 bytes of zero slack behind the data and its slots are 16-byte aligned)
__device__ __forceinline__ void load_span(const uint8_t* __restrict__ ustream, uint64_t byte0, uint32_t span_bytes, uint64_t uslot, uint32_t* s_span)
{
    const uint4* src = reinterpret_cast<const uint4*>(ustream + byte0);
    uint4* dst = reinterpret_cast<uint4*>(s_span);
    const uint32_t n16 = (span_bytes + kSpanSlack) / 16;
    const uint64_t avail16 = (uslot - byte0) / 16;        // the last CTA's span reaches past the image's slot: zeros there
    for (uint32_t i = threadIdx.x; i < n16; i += blockDim.x) {
        uint4 v = i < avail16 ? __ldg(src + i) : make_uint4(0, 0, 0, 0);
        v.x = __byte_perm(v.x, 0, 0x0123), v.y = __byte_perm(v.y, 0, 0x0123);      // big-endian bit order inside every word
        v.z = __byte_perm(v.z, 0, 0x0123), v.w = __byte_perm(v.w, 0, 0x0123);
        dst[i] = v;
    }
}

// ---- D0: un-stuffing -------------------------------------------------------------------------------
// keep[i] = !(byte[i] == 0x00 && byte[i-1] == 0xFF)
// dri: RSTn markers (FF D0..D7) are dropped as well; bit i of *markers = byte i is the FF of such a marker
__device__ __forceinline__ uint32_t keep_mask16(const uint8_t* __restrict__ src, uint64_t i0, uint64_t n, uint8_t* bytes, bool dri, uint32_t* markers)
{
    uint32_t m = 0, mk = 0;
    uint8_t prev = i0 ? src[i0 - 1] : 0;
    uint8_t c = i0 < n ? src[i0] : 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const uint64_t idx = i0 + i;
        const uint8_t nxt = idx + 1 < n ? src[idx + 1] : 0;
        bytes[i] = c;
        const bool stuffed = c == 0 && prev == 0xff;
        const bool rst_ff = dri && c == 0xff && (nxt & 0xf8) == 0xd0;
        const bool rst_dx = dri && prev == 0xff && (c & 0xf8) == 0xd0;
        if (idx < n && !stuffed && !rst_ff && !rst_dx) m |= 1u << i;
        if (idx < n && rst_ff) mk |= 1u << i;
        prev = c;
        c = nxt;
    }
    *markers = mk;
    return m;
}

__device__ __forceinline__ uint32_t cta_scan_excl(uint32_t v, uint32_t* s_warp, uint32_t* total)
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

__global__ void __launch_bounds__(kDecThreads) k_unstuff_count(const DecParams p)
{
    pdl_wait();
    __shared__ uint32_t s_warp[kDecThreads / 32];
    const size_t img = blockIdx.y;
    // first kernel of a decode: clears the counters of the synchronisation launches (no zero-fill between the kernels,
    // which would break the chain of dependent launches)
    if (blockIdx.x == 0 && blockIdx.y == 0 && p.changed) {
        if (threadIdx.x < kMaxSyncRounds) p.changed[threadIdx.x] = 0;
        if (threadIdx.x < 2) p.iters_stat[threadIdx.x] = 0;
    }
    if (p.cta_flag)
        for (uint32_t i = (blockIdx.y * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x; i < p.nflag; i += gridDim.x * gridDim.y * blockDim.x) p.cta_flag[i] = 0;
    uint64_t n = p.ext_bytes ? p.ext_bytes[img] : (p.ninline ? p.inline_bytes[img & 7] : p.scan_bytes[img]);
    if (p.ext_bytes && n > p.max_bytes) n = 0;       // does not fit what the launch was sized for: nothing is decoded (k_scan_blocks reports it)
    if ((p.ninline || p.ext_bytes) && blockIdx.x == 0 && threadIdx.x == 0) const_cast<uint64_t*>(p.scan_bytes)[img] = n;
    const uint8_t* src = p.scan + img * p.slot;
    const uint32_t nch = uint32_t((n + 4095) / 4096);
    for (uint32_t ch = blockIdx.x; ch < nch; ch += gridDim.x) {
        uint8_t bytes[16];
        const uint64_t i0 = (uint64_t(ch) * kDecThreads + threadIdx.x) * 16;
        uint32_t mk = 0;
        const uint32_t m = i0 < n ? keep_mask16(src, i0, n, bytes, p.dri != 0, &mk) : 0u;
        uint32_t total;
        cta_scan_excl(__popc(m), s_warp, &total);
        if (threadIdx.x == 0) p.chunk_cnt[img * p.nchunk + ch] = total;
        if (p.dri) {
            cta_scan_excl(__popc(mk), s_warp, &total);
            if (threadIdx.x == 0) p.chunk_mcnt[img * p.nchunk + ch] = total;
        }
    }
}

// generic per-image exclusive scan of uint32 counts with a 64-bit carry; one CTA (1024 threads) per image
__global__ void __launch_bounds__(1024) k_scan_chunks(const uint32_t* __restrict__ cnt, uint64_t* __restrict__ base, uint32_t stride,
                                                      const uint64_t* __restrict__ nbytes, uint32_t unit, uint64_t* __restrict__ total_out)
{
    pdl_wait();
    __shared__ uint32_t s_warp[32];
    __shared__ uint64_t s_carry;
    const size_t img = blockIdx.x;
    const uint32_t n = uint32_t((nbytes[img] + unit - 1) / unit);
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t c0 = 0; c0 < n; c0 += 1024) {
        const uint32_t c = c0 + threadIdx.x;
        const uint32_t v = c < n ? cnt[img * stride + c] : 0u;
        uint32_t total;
        const uint32_t off = cta_scan_excl(v, s_warp, &total);
        const uint64_t carry = s_carry;
        if (c < n) base[img * stride + c] = carry + off;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + total;
        __syncthreads();
    }
    if (threadIdx.x == 0 && total_out) total_out[img] = s_carry;
}

__global__ void __launch_bounds__(kDecThreads) k_unstuff_write(const DecParams p)
{
    pdl_wait();
    __shared__ uint32_t s_warp[kDecThreads / 32];
    const size_t img = blockIdx.y;
    const uint64_t n = p.scan_bytes[img];
    const uint8_t* src = p.scan + img * p.slot;
    uint8_t* dst = p.ustream + img * p.uslot;
    const uint32_t nch = uint32_t((n + 4095) / 4096);
    for (uint32_t ch = blockIdx.x; ch < nch; ch += gridDim.x) {
        uint8_t bytes[16];
        const uint64_t i0 = (uint64_t(ch) * kDecThreads + threadIdx.x) * 16;
        uint32_t mk = 0;
        const uint32_t m = i0 < n ? keep_mask16(src, i0, n, bytes, p.dri != 0, &mk) : 0u;
        uint32_t total;
        const uint32_t off = cta_scan_excl(__popc(m), s_warp, &total);
        uint64_t o = p.chunk_base[img * p.nchunk + ch] + off;
        if (p.dri) {
            // the segment after the k-th marker starts at the next kept byte (marker bytes are not kept)
            const uint32_t moff = cta_scan_excl(__popc(mk), s_warp, &total);
            uint64_t k = p.chunk_mbase[img * p.nchunk + ch] + moff;
            for (uint32_t mm = mk; mm; mm &= mm - 1, ++k) {
                const int i = __ffs(int(mm)) - 1;
                if (k + 1 <= p.nseg) p.seg_start[img * (p.nseg + 1) + k + 1] = o + __popc(m & ((1u << i) - 1u));
            }
        }
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (m & (1u << i)) dst[o++] = bytes[i];
    }
    // zero slack after the data so that peeks past the end read zeros
    if (blockIdx.x == 0 && threadIdx.x < 64) {
        const uint64_t u = p.ubytes[img];
        if (u + threadIdx.x < p.uslot) dst[u + threadIdx.x] = 0;
    }
}

// ---- D1a: speculative decode + synchronisation --------------------------------------------------------
// One CTA owns kDecOwn consecutive subsequences and, in launch 0, also decodes the kDecWarm subsequences in front of
// them (which belong to the previous CTA) as a warm-up.  Launch 0: every thread decodes its subsequence from the guessed
// state (b = 0, z = 0); then the CTA iterates in shared memory: a thread whose predecessor's end state changed
// re-decodes from it, until nothing changes inside the CTA.  Huffman codes re-synchronise within a few subsequences, so
// by the end of the warm-up run the states are the true ones and the owned subsequences come out right in launch 0.
// Launch 0 ends with a check across the CTA boundary: the CTA's own (warm-up) end state of the subsequence in front of its
// first owned one against the previous CTA's tail.  If they agree at every boundary, every CTA's owned states follow from its
// predecessor's tail, and by induction from CTA 0 (which starts at the beginning of the stream) all of them are the true ones:
// changed[0] stays 0 and the launches behind return at once.
// Launch k >= 1: the first owned subsequence is re-seeded from the previous CTA's last end state of launch k - 1
// (`tail`); `changed` counts the end states that changed during a launch, 0 = global fixed point.
constexpr int kDecWarm = 32;

__global__ void __launch_bounds__(kDecThreads) k_sync_decode(const DecParams p, const int launch, const int host_poll)
{
    pdl_wait();
    extern __shared__ __align__(16) uint32_t s_span[];      // (kDecThreads * sub_bits / 8 + kSpanSlack) bytes of the stream
    __shared__ __align__(16) DecTabs s_tabs;
    __shared__ uint32_t s_state[kDecThreads];
    __shared__ uint8_t s_chg[2][kDecThreads];
    __shared__ uint16_t s_list[kDecThreads];      // subsequences to re-decode in this iteration
    __shared__ uint32_t s_nlist;
    // launches are enqueued without host round trips: once a launch saw no change (a global fixed point), the
    // later ones return immediately (changed[] stays 0 for them, so the zero propagates to changed[rounds])
    // (host_poll: the host reads changed[1] after every launch instead)
    if (!host_poll && launch >= 1 && p.changed[launch - 1] == 0) return;
    const size_t img = blockIdx.y;
    const uint64_t total_bits = p.ubytes[img] * 8;
    const int t = threadIdx.x;
    const uint32_t nthr = p.cta_own + kDecWarm;                                          // == blockDim.x
    const uint32_t first_own = blockIdx.x * p.cta_own;                                   // first owned subsequence
    const uint32_t first = blockIdx.x == 0 ? 0u : first_own - kDecWarm;                // first subsequence of the span
    const int64_t isub = int64_t(first_own) - kDecWarm + t;                            // this thread's subsequence
    if (uint64_t(first_own) * p.sub_bits >= total_bits) {     // (capacity CTA beyond the data of this image)
        if (t == 0) p.sub_blk[img * gridDim.x + blockIdx.x] = 0;
        return;
    }
    const uint64_t span_start = uint64_t(first) * p.sub_bits;                          // multiple of 128 bits
    const uint32_t span_bits = nthr * p.sub_bits;
    load_dec_tabs(p.tabs, &s_tabs, p.nb, p.ny);
    load_span(p.ustream + img * p.uslot, span_start / 8, span_bits / 8, p.uslot, s_span);
    const uint32_t span_sa = uint32_t(__cvta_generic_to_shared(s_span));
    const uint32_t start = uint32_t(isub - int64_t(first)) * p.sub_bits, end = start + p.sub_bits;   // relative to the span
    const uint32_t limit = uint32_t(min(total_bits - span_start, uint64_t(span_bits) + 256u));
    const bool owner = t >= kDecWarm;
    // warm-up threads only work in launch 0; afterwards the owned states are re-seeded from the previous CTA's tail
    const bool valid = isub >= 0 && isub < int64_t(p.nsub) && start < limit && (owner || launch == 0);
    const size_t si = img * p.nsub + size_t(isub < 0 ? 0 : isub);
    const uint32_t ncta = gridDim.x;
    const uint32_t* tail_in = (launch & 1) ? p.state_b : p.state_a;     // [nimg][ncta] tails of the previous launch
    uint32_t* tail_out = (launch & 1) ? p.state_a : p.state_b;
    __syncthreads();

    uint32_t st = 0;
    bool chg = false;
    if (valid) {
        if (launch == 0) {
            FastBits br;
            br.init(span_sa, start);
            uint32_t b = 0, z = 0, n = 0;
            decode_span<false>(br, b, z, n, end, limit, &s_tabs, nullptr, nullptr, 0, 0, nullptr, p.nb, p.ny);
            st = pack_state(br.pos > end ? br.pos - end : 0u, b, z, n);
            chg = true;
        } else {
            st = p.sub_state[si];
            if (t == kDecWarm && blockIdx.x > 0) {
                const uint32_t ps = tail_in[img * ncta + blockIdx.x - 1];
                FastBits br;
                br.init(span_sa, start + (ps & 63u));
                uint32_t b = (ps >> 6) & 7u, z = (ps >> 9) & 63u, n = 0;
                decode_span<false>(br, b, z, n, end, limit, &s_tabs, nullptr, nullptr, 0, 0, nullptr, p.nb, p.ny);
                const uint32_t ns = pack_state(br.pos > end ? br.pos - end : 0u, b, z, n);
                chg = ((ns ^ st) & kStateSyncMask) != 0;
                st = ns;
            }
        }
    }
    s_state[t] = st;
    s_chg[0][t] = chg ? 1 : 0;
    uint32_t nchanged = (launch > 0 && chg) ? 1u : 0u;
    if (t == 0) s_nlist = 0;
    __syncthreads();
    // The subsequences whose predecessor's end state changed are re-decoded from it.  Their set thins out quickly
    // (a decode re-synchronises within its subsequence more often than not), so it is compacted first: entry j of the
    // list is handled by thread j, and an iteration costs as many warps as there is work, not every warp that holds one
    // such subsequence.
    for (int it = 0; it < 4 * kDecThreads; ++it) {     // (a chain cannot be longer than the CTA)
        // (the very first subsequence of the image has no predecessor: its guessed state is the true one)
        const bool redo = valid && isub > 0 && t > 0 && s_chg[it & 1][t - 1];
        s_chg[(it + 1) & 1][t] = 0;      // (last read two barriers ago)
        const uint32_t bal = __ballot_sync(0xffffffffu, redo);
        uint32_t wbase = 0;
        if ((t & 31) == 0 && bal) wbase = atomicAdd(&s_nlist, uint32_t(__popc(bal)));
        wbase = __shfl_sync(0xffffffffu, wbase, 0);
        if (redo) s_list[wbase + __popc(bal & ((1u << (t & 31)) - 1u))] = uint16_t(t);
        __syncthreads();
        const uint32_t nlist = s_nlist;
        if (nlist == 0) {
            if (t == 0 && launch <= 1) atomicMax(p.iters_stat + launch, (unsigned long long)it);
            break;
        }
        uint32_t tt = 0, ns = 0;
        bool c2 = false;
        if (uint32_t(t) < nlist) {
            tt = s_list[t];
            const uint32_t ps = s_state[tt - 1], old = s_state[tt];
            const uint32_t start_tt = uint32_t(int64_t(tt) + int64_t(first_own) - kDecWarm - int64_t(first)) * p.sub_bits;   // as `start`
            const uint32_t end_tt = start_tt + p.sub_bits;
            FastBits br;
            br.init(span_sa, start_tt + (ps & 63u));
            uint32_t b = (ps >> 6) & 7u, z = (ps >> 9) & 63u, n = 0;
            decode_span<false>(br, b, z, n, end_tt, limit, &s_tabs, nullptr, nullptr, 0, 0, nullptr, p.nb, p.ny);
            ns = pack_state(br.pos > end_tt ? br.pos - end_tt : 0u, b, z, n);
            c2 = ((ns ^ old) & kStateSyncMask) != 0;
        }
        __syncthreads();                 // all reads of s_state and s_list are done
        if (uint32_t(t) < nlist) {
            s_state[tt] = ns;
            s_chg[(it + 1) & 1][tt] = c2 ? 1 : 0;
            if (c2 && tt >= uint32_t(kDecWarm)) ++nchanged;      // an owned subsequence
        }
        if (t == 0) s_nlist = 0;
        __syncthreads();
    }
    st = s_state[t];
    const bool mine = valid && owner;
    if (mine) p.sub_state[si] = st;
    // the CTA's last valid subsequence is the seed of the next CTA
    const bool is_tail = mine && (t == int(nthr) - 1 || end >= limit || isub + 1 >= int64_t(p.nsub));
    if (is_tail) tail_out[img * ncta + blockIdx.x] = st;
    if (launch > 0 && nchanged) atomicAdd(p.changed + (host_poll ? 1 : launch), (unsigned long long)nchanged);
    if (launch == 0 && p.cta_flag) {
        // (a CTA only ever waits for the CTA in front of it, which was scheduled no later: no deadlock)
        volatile uint32_t* flag = p.cta_flag + img * ncta;
        if (is_tail) {
            __threadfence();
            flag[blockIdx.x] = 1u;
        }
        if (t == kDecWarm - 1 && blockIdx.x > 0) {
            uint32_t spins = 0;
            while (flag[blockIdx.x - 1] == 0u) {
                __nanosleep(64);
                if (++spins > (1u << 24)) __trap();      // (a protocol error must not hang the device)
            }
            __threadfence();
            const uint32_t ps = *(volatile uint32_t*)(tail_out + img * ncta + blockIdx.x - 1);
            if ((ps ^ st) & kStateSyncMask) atomicAdd(p.changed, 1ull);
        }
    }
    // blocks completed inside this CTA's own subsequences (input of the block-index scan)
    uint32_t total;
    cta_scan_excl(mine ? (st >> 15) & 4095u : 0u, reinterpret_cast<uint32_t*>(s_state), &total);
    if (t == 0) p.sub_blk[img * ncta + blockIdx.x] = total;
}

// ---- D1a, launch 0 for latency-bound inputs (a single frame): several guesses per subsequence -----------------------------
// How long the chain of dependent re-decodes of k_sync_decode gets is set by the slowest synchronisation anywhere in the
// image: position and zig-zag index of a decoder started from a guess merge with the true parse within a few symbols, but its
// block-in-MCU phase only re-rolls about once per MCU, and the tail of that distribution is long (tools/sync_distance_sim.py on
// a 4K S-photo frame: up to 12+ subsequences of 128 bits for the single guess b = 0, at most 5 -- 99.9 %: at most 3 -- for the
// best of the guesses b = 0..nb-1).  So this kernel runs one chain per guess, nb x as many threads, all at once:
//   round 0       thread (slot, h) decodes its subsequence from the state (block h, start of block);
//   rounds 1..K   ... again from the end state of (slot - 1, h) of the round before, unless that is what it used last time;
//   walk          from an anchor (the start of the image, or the last warm-up slot at which all chains agree) the true state is
//                 carried from slot to slot: E_slot(x) is looked up among the inputs the slot's chains were decoded from, and
//                 decoded only on a miss.
// What comes out are the states k_sync_decode would reach (same arrays, same check against the previous CTA's tail at the end,
// so a wrong anchor is caught and repaired by launch 1): the guesses only decide how fast.
constexpr int kHypRounds = 2;
constexpr int kHypOwn = 64;         // subsequences a CTA owns (DecParams::cta_own on this path)
constexpr int kHypWarm = 16;        // warm-up subsequences in front of them: enough to find a slot at which all chains agree
constexpr int kHypSlots = kHypOwn + kHypWarm;
constexpr int kHypMax = 6;          // blocks per MCU = guesses

__global__ void __launch_bounds__(kHypSlots * kHypMax, 2) k_sync_decode_hyp(const DecParams p)
{
    pdl_wait();
    extern __shared__ __align__(16) uint32_t s_span[];
    __shared__ __align__(16) DecTabs s_tabs;
    __shared__ uint32_t s_v[kHypMax][kHypSlots];       // end state of chain h at the slot
    __shared__ uint32_t s_in[kHypMax][kHypSlots];      // the state it was decoded from (0xffffffff: its guess)
    __shared__ uint32_t s_state[kHypSlots];
    __shared__ uint8_t s_una[kHypSlots];
    __shared__ uint16_t s_work[kHypSlots * kHypMax];   // work list of a round: slot | chain << 8
    __shared__ uint32_t s_nwork;
    __shared__ uint32_t s_scan[32];
    const size_t img = blockIdx.y;
    const uint64_t total_bits = p.ubytes[img] * 8;
    const int t = threadIdx.x;
    constexpr uint32_t slots = uint32_t(kHypSlots);                                      // blockDim.x == slots * p.nb; p.cta_own == kHypOwn
    const uint32_t h = uint32_t(t) / slots, slot = uint32_t(t) - h * slots;
    const uint32_t first_own = blockIdx.x * p.cta_own;
    const uint32_t s0 = blockIdx.x == 0 ? uint32_t(kHypWarm) : 0u;                       // slot of the first subsequence of the span
    const uint32_t first = first_own - (uint32_t(kHypWarm) - s0);
    const int64_t isub = int64_t(first_own) - kHypWarm + slot;
    if (uint64_t(first_own) * p.sub_bits >= total_bits) {     // (capacity CTA beyond the data of this image)
        if (t == 0) p.sub_blk[img * gridDim.x + blockIdx.x] = 0;
        return;
    }
    const uint64_t span_start = uint64_t(first) * p.sub_bits;
    const uint32_t span_bits = slots * p.sub_bits;
    load_dec_tabs(p.tabs, &s_tabs, p.nb, p.ny);
    load_span(p.ustream + img * p.uslot, span_start / 8, span_bits / 8, p.uslot, s_span);
    const uint32_t span_sa = uint32_t(__cvta_generic_to_shared(s_span));
    const uint32_t start = (slot - s0) * p.sub_bits, end = start + p.sub_bits;           // (meaningless for slot < s0: not valid)
    const uint32_t limit = uint32_t(min(total_bits - span_start, uint64_t(span_bits) + 256u));
    const bool owner = slot >= uint32_t(kHypWarm);
    const bool valid = isub >= 0 && isub < int64_t(p.nsub) && start < limit;
    const size_t si = img * p.nsub + size_t(isub < 0 ? 0 : isub);
    const uint32_t ncta = gridDim.x;
    uint32_t* tail_out = p.state_b;                             // (launch 0 of k_sync_decode writes state_b)
    if (t == 0) s_nwork = 0;
    __syncthreads();

    auto decode_from = [&](uint32_t at, uint32_t ps) -> uint32_t {
        FastBits br;
        br.init(span_sa, at + (ps & 63u));
        uint32_t b = (ps >> 6) & 7u, z = (ps >> 9) & 63u, n = 0;
        decode_span<false>(br, b, z, n, at + p.sub_bits, limit, &s_tabs, nullptr, nullptr, 0, 0, nullptr, p.nb, p.ny);
        return pack_state(br.pos > at + p.sub_bits ? br.pos - (at + p.sub_bits) : 0u, b, z, n);
    };

    // ---- round 0: from the guesses (the first subsequence of the image has no guess: block 0, start of block, is the truth) ----
    uint32_t vin = 0xffffffffu;
    s_v[h][slot] = valid ? decode_from(start, isub == 0 ? 0u : (h << 6)) : 0u;
    // ---- rounds 1..K: every chain one subsequence further.  Chains that have merged give their successors the same input: one
    //      thread per distinct (slot, input) decodes -- the work items are compacted so that a round costs as many warps as it has
    //      work -- and the others copy; an input that did not change since the last round needs nothing. ----
    const bool has_pred = valid && isub > 0 && slot > 0;
#pragma unroll 1
    for (int k = 1; k <= kHypRounds; ++k) {
        __syncthreads();
        uint32_t in = 0xffffffffu, rep = h;
        bool work = false;
        if (has_pred) {
            in = s_v[h][slot - 1];
            for (uint32_t a = 0; a < h; ++a)
                if (((s_v[a][slot - 1] ^ in) & kStateSyncMask) == 0u) {
                    rep = a;
                    break;
                }
            work = rep == h && ((in ^ vin) & kStateSyncMask) != 0u;
        }
        {
            const uint32_t bal = __ballot_sync(0xffffffffu, work);
            uint32_t wbase = 0;
            if ((t & 31) == 0 && bal) wbase = atomicAdd(&s_nwork, uint32_t(__popc(bal)));
            wbase = __shfl_sync(0xffffffffu, wbase, 0);
            if (work) s_work[wbase + __popc(bal & ((1u << (t & 31)) - 1u))] = uint16_t(slot | (h << 8));
        }
        __syncthreads();
        const uint32_t nwork = s_nwork;
        uint32_t it_slot = 0, it_h = 0, res = 0;
        if (uint32_t(t) < nwork) {
            const uint32_t item = s_work[t];
            it_slot = item & 255u, it_h = item >> 8;
            res = decode_from((it_slot - s0) * p.sub_bits, s_v[it_h][it_slot - 1]);
        }
        __syncthreads();                 // every read of the previous round's states is done
        if (uint32_t(t) < nwork) s_v[it_h][it_slot] = res;
        if (t == 0) s_nwork = 0;
        __syncthreads();
        if (has_pred) {
            // a follower takes its representative's state (the representative's own, if its input did not change, is still the one
            // that belongs to this input)
            if (rep != h) s_v[h][slot] = s_v[rep][slot];
            vin = in;
        }
    }
    __syncthreads();
    s_in[h][slot] = vin;
    if (h == 0) {
        // all chains in the same state: the true one (a decoder that has merged with another stays merged, and the true parse is one
        // of the decoders; nb chains that agree with each other but not with it would have had to merge without touching it)
        bool una = valid;
        for (uint32_t a = 1; a < p.nb; ++a) una = una && ((s_v[a][slot] ^ s_v[0][slot]) & kStateSyncMask) == 0u;
        s_una[slot] = una ? 1 : 0;
        s_state[slot] = s_v[0][slot];
    }
    __syncthreads();
    // ---- the true chain: from an anchor -- the start of the image, or the last warm-up slot whose chains all agree -- follow
    //      E_slot(x) through the slots; it is looked up among the inputs the slot's chains were decoded from (a hit is a few
    //      shared-memory reads by the lanes of one warp, and supplies the block count that goes with the TRUE input) and decoded
    //      only on a miss.  One warp walks, the others wait: ~40 cycles per slot. ----
    if (t < 32) {
        const uint32_t lane = uint32_t(t);
        int w = int(kHypWarm) - 1;                                                       // anchor slot
        if (blockIdx.x == 0) w = int(kHypWarm);
        else {
            const uint32_t bal = __ballot_sync(0xffffffffu, lane < uint32_t(kHypWarm) && s_una[lane] != 0);
            if (bal) w = 31 - __clz(int(bal));
        }
        uint32_t x = s_state[w];
        uint32_t misses = 0;
        for (uint32_t ts = uint32_t(w) + 1u; ts < slots; ++ts) {
            const uint32_t start_ts = (ts - s0) * p.sub_bits;
            if (start_ts >= limit || int64_t(first_own) - kHypWarm + ts >= int64_t(p.nsub)) break;
            const uint32_t key = lane < p.nb ? s_in[lane][ts] : 0xffffffffu;
            const uint32_t val = lane < p.nb ? s_v[lane][ts] : 0u;
            const uint32_t hit = __ballot_sync(0xffffffffu, key != 0xffffffffu && ((key ^ x) & kStateSyncMask) == 0u);
            if (hit) {
                x = __shfl_sync(0xffffffffu, val, __ffs(int(hit)) - 1);
            } else {
                if (lane == 0) x = decode_from(start_ts, x);
                x = __shfl_sync(0xffffffffu, x, 0);
                ++misses;
            }
            if (lane == 0) s_state[ts] = x;
        }
        if (lane == 0) {
            atomicMax(p.iters_stat, (unsigned long long)(misses + kHypRounds));
            atomicAdd(p.iters_stat + 1, (unsigned long long)misses);
        }
    }
    __syncthreads();
    // ---- results: as k_sync_decode, by the threads of chain 0 ----
    const uint32_t st = h == 0 ? s_state[slot] : 0u;
    const bool mine = h == 0 && valid && owner;
    if (mine) p.sub_state[si] = st;
    const bool is_tail = mine && (slot == slots - 1 || end >= limit || isub + 1 >= int64_t(p.nsub));
    if (is_tail) tail_out[img * ncta + blockIdx.x] = st;
    if (p.cta_flag) {
        volatile uint32_t* flag = p.cta_flag + img * ncta;
        if (is_tail) {
            __threadfence();
            flag[blockIdx.x] = 1u;
        }
        if (h == 0 && slot == uint32_t(kHypWarm) - 1u && blockIdx.x > 0) {
            uint32_t spins = 0;
            while (flag[blockIdx.x - 1] == 0u) {
                __nanosleep(64);
                if (++spins > (1u << 24)) __trap();
            }
            __threadfence();
            const uint32_t ps = *(volatile uint32_t*)(tail_out + img * ncta + blockIdx.x - 1);
            if ((ps ^ st) & kStateSyncMask) atomicAdd(p.changed, 1ull);
        }
    }
    uint32_t total;
    cta_scan_excl(mine ? (st >> 15) & 4095u : 0u, s_scan, &total);
    if (t == 0) p.sub_blk[img * ncta + blockIdx.x] = total;
}

// exclusive scan of the per-CTA block counts (in place) and per-image status
__global__ void __launch_bounds__(1024) k_scan_blocks(const DecParams p, const uint32_t ncta)
{
    pdl_wait();
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_carry;
    const size_t img = blockIdx.x;
    const uint64_t total_bits = p.ubytes[img] * 8;
    const uint32_t nsub = uint32_t(min(uint64_t(p.nsub), (total_bits + p.sub_bits - 1) / p.sub_bits));
    const uint32_t n = (nsub + p.cta_own - 1) / p.cta_own;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t c0 = 0; c0 < n; c0 += 1024) {
        const uint32_t c = c0 + threadIdx.x;
        const uint32_t v = c < n ? p.sub_blk[img * ncta + c] : 0u;
        uint32_t total;
        const uint32_t off = cta_scan_excl(v, s_warp, &total);
        const uint32_t carry = s_carry;
        if (c < n) p.sub_blk[img * ncta + c] = carry + off;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // not a fixed point after the enqueued launches: the caller has to run the host-driven loop (JPEZYB200_EAGAIN)
        const bool converged = p.rounds == 0 || p.changed[p.rounds] == 0;
        if (p.status) {
            p.status[img] = !converged ? JPEZYB200_EAGAIN : (s_carry >= p.nblk ? 0 : JPEZYB200_ECORRUPT);
            if (p.ext_bytes && p.ext_bytes[img] > p.max_bytes) p.status[img] = JPEZYB200_ECAPACITY;
        }
        if (img == 0) {
            unsigned long long n = 1 + p.rounds_host;
            for (uint32_t k = 1; k <= p.rounds; ++k) n += p.changed[k - 1] != 0 ? 1ull : 0ull;
            *p.rounds_stat = n;
        }
    }
}

// ---- D1c: final pass, writes the non-zero coefficients (buffer pre-zeroed) ------------------------------
__global__ void __launch_bounds__(kDecThreads) k_write_coefs(const DecParams p)
{
    pdl_wait();
    extern __shared__ __align__(16) uint32_t s_span[];
    __shared__ __align__(16) DecTabs s_tabs;
    __shared__ uint32_t s_warp[kDecThreads / 32];
    const size_t img = blockIdx.y;
    const uint64_t total_bits = p.ubytes[img] * 8;
    // same ownership as k_sync_decode (p.cta_own subsequences per CTA; the last kDecWarm threads idle)
    const uint64_t cta_start = uint64_t(blockIdx.x) * p.cta_own * p.sub_bits;
    if (cta_start >= total_bits) return;
    const uint32_t span_bits = p.cta_own * p.sub_bits;
    load_dec_tabs(p.tabs, &s_tabs, p.nb, p.ny);
    load_span(p.ustream + img * p.uslot, cta_start / 8, span_bits / 8, p.uslot, s_span);
    const uint32_t span_sa = uint32_t(__cvta_generic_to_shared(s_span));
    const uint32_t i = blockIdx.x * p.cta_own + threadIdx.x;
    const uint32_t start = threadIdx.x * p.sub_bits;
    const uint32_t limit = uint32_t(min(total_bits - cta_start, uint64_t(span_bits) + 256u));
    const bool valid = threadIdx.x < p.cta_own && start < limit && i < p.nsub;
    const size_t si = img * p.nsub + i;
    const uint32_t mine = valid ? p.sub_state[si] : 0u;
    __syncthreads();
    uint32_t total;
    const uint64_t blk = uint64_t(p.sub_blk[img * gridDim.x + blockIdx.x]) + cta_scan_excl((mine >> 15) & 4095u, s_warp, &total);
    if (!valid || blk >= p.nblk) return;
    uint32_t pos = start;
    uint32_t b = 0, z = 0, n = 0;
    if (i) {
        const uint32_t ps = p.sub_state[si - 1];
        pos = start + (ps & 63u), b = (ps >> 6) & 7u, z = (ps >> 9) & 63u;
    }
    FastBits br;
    br.init(span_sa, pos);
    int corrupt = 0;
    decode_span<true>(br, b, z, n, start + p.sub_bits, limit, &s_tabs, p.coefs + img * p.coef_stride, p.dcd + img * p.nblk, blk, p.nblk, &corrupt, p.nb, p.ny);
    // (only over "ok": when the synchronisation did not converge -- JPEZYB200_EAGAIN from k_scan_blocks -- this pass ran from wrong
    // states, and what it saw says nothing about the stream: the caller decodes again)
    if (corrupt && p.status) atomicCAS(p.status + img, 0, int(JPEZYB200_ECORRUPT));
}

// ---- restart intervals: every segment is self-contained (predictors reset, byte aligned), one thread each --------
// restart_interval_check (src/decoder/jpezy_decoder.hpp:152-163): after `dri` MCUs the reference reads the next marker and
// resets pred_dct[]; the segments between the markers were located by the un-stuffing pass (seg_start).
__global__ void __launch_bounds__(128) k_decode_segments(const DecParams p)
{
    pdl_wait();
    __shared__ __align__(16) DecTabs s_tabs;
    load_dec_tabs(p.tabs, &s_tabs, p.nb, p.ny);
    __syncthreads();
    const size_t img = blockIdx.y;
    const uint32_t seg = blockIdx.x * blockDim.x + threadIdx.x;
    if (seg >= p.nseg) return;
    const uint64_t nmark = p.nmarkers[img];
    const uint64_t ubytes = p.ubytes[img];
    if (nmark + 1 < p.nseg) {                       // fewer RSTn markers than the frame needs
        if (seg == 0 && p.status) p.status[img] = JPEZYB200_ECORRUPT;
        return;
    }
    const uint64_t b0 = seg == 0 ? 0 : p.seg_start[img * (p.nseg + 1) + seg];
    const uint64_t b1 = seg + 1 < p.nseg ? p.seg_start[img * (p.nseg + 1) + seg + 1] : ubytes;
    if (b0 > ubytes || b1 > ubytes || b1 < b0 || (b1 - b0) * 8 > 0xfffffff0ull) {
        if (p.status) p.status[img] = JPEZYB200_ECORRUPT;
        return;
    }
    // the bit reader works on 32-bit words: start at the word that holds byte b0
    const uint8_t* base = p.ustream + img * p.uslot;
    const uint64_t w0 = b0 & ~uint64_t(3);
    BitBuf br;
    br.init(reinterpret_cast<const uint32_t*>(base + w0), uint32_t(b0 - w0) * 8u);
    const uint32_t limit = uint32_t((b1 - w0) * 8);
    const uint32_t mcu0 = seg * p.dri, mcu1 = min(p.nmcu, mcu0 + p.dri);
    int16_t* out = p.coefs + img * p.coef_stride;
    int pred[3] = {0, 0, 0};
    int corrupt = 0;
    bool dc_wide = false;     // a DC coefficient outside the int16 range of the coefficient format
    for (uint32_t m = mcu0; m < mcu1 && !corrupt; ++m) {
        for (uint32_t k = 0; k < p.nb; ++k) {
            const uint32_t comp = k < p.ny ? 0u : k - p.ny + 1u;
            const uint32_t cls = comp ? 1u : 0u;
            int16_t* blk = out + (size_t(m) * p.nb + k) * 64;
            uint32_t z = 0;
            while (z < 64u) {
                if (br.pos >= limit) { corrupt = 1; break; }
                br.refill();
                const uint32_t w = br.peek32();
                const uint32_t ti = (z == 0u ? 0u : 2u) + cls;
                uint32_t e = s_tabs.fast[ti][w >> (32 - kLutBits)];
                if (e == kEntryNone) e = huff_lookup_slow(s_tabs.slow + ti, w);
                if (e == 0u) { corrupt = 1; break; }
                if (((e >> 8) & 255u) > 64u && z + ((e >> 8) & 255u) >= 128u) e = unfold_entry(e);   // see huff_entry
                br.skip(int(e & 31u));
                const uint32_t dzf = (e >> 8) & 255u, len = (e >> 16) & 31u, sz = (e >> 21) & 15u;
                const bool fold = dzf > 64u;
                const uint32_t dz = fold ? dzf - 64u : dzf;
                const uint32_t kk = z + dz - 1u;
                if (kk > 63u && dz != 64u) { corrupt = 1; break; }
                if (sz) {
                    const uint32_t vbits = (w << len) >> (32 - sz);
                    int v = int(vbits);
                    if (!(vbits & (1u << (sz - 1)))) v -= (1 << sz) - 1;
                    if (z == 0u) {
                        v = (pred[comp] += v);
                        dc_wide |= v != int(int16_t(v));
                    }
                    blk[kk] = int16_t(v);
                } else if (z == 0u) {
                    blk[0] = int16_t(pred[comp]);
                }
                z = fold ? 64u : z + dz;
            }
            if (corrupt) break;
        }
    }
    if (corrupt && p.status) p.status[img] = JPEZYB200_ECORRUPT;
    else if (dc_wide && p.status) atomicCAS(p.status + img, 0, int(JPEZYB200_EUNSUPPORTED));
}

// ---- D1d: DC differences -> absolute DC (pred_dct[sc] += diff, src/decoder/jpezy_decoder.hpp:596-597) -----
// tile = 256 MCUs; per tile the sums of the Y (ny blocks per MCU), Cb, Cr differences
__global__ void __launch_bounds__(256) k_dc_sum(const DecParams p)
{
    pdl_wait();
    __shared__ int s_red[3][8];
    const size_t img = blockIdx.y;
    const uint32_t m = blockIdx.x * 256 + threadIdx.x;
    int y = 0, cb = 0, cr = 0;
    if (m < p.nmcu) {
        const int16_t* c = p.dcd + img * p.nblk + size_t(m) * p.nb;
        for (uint32_t k = 0; k < p.ny; ++k) y += int(c[k]);
        if (p.nb > p.ny) cb = c[p.ny], cr = c[p.ny + 1];
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        y += __shfl_xor_sync(0xffffffffu, y, d);
        cb += __shfl_xor_sync(0xffffffffu, cb, d);
        cr += __shfl_xor_sync(0xffffffffu, cr, d);
    }
    if ((threadIdx.x & 31) == 0) s_red[0][threadIdx.x >> 5] = y, s_red[1][threadIdx.x >> 5] = cb, s_red[2][threadIdx.x >> 5] = cr;
    __syncthreads();
    if (threadIdx.x < 3) {
        int s = 0;
        for (int w = 0; w < 8; ++w) s += s_red[threadIdx.x][w];
        p.dc_part[(img * p.ndc_tiles + blockIdx.x) * 3 + threadIdx.x] = s;
    }
}

__global__ void __launch_bounds__(32) k_dc_scan_tiles(const DecParams p)
{
    pdl_wait();
    // one warp per (image, component): sequential over tiles in chunks of 32 with a shuffle scan
    const size_t img = blockIdx.x;
    const int comp = blockIdx.y;
    int carry = 0;
    for (uint32_t t0 = 0; t0 < p.ndc_tiles; t0 += 32) {
        const uint32_t t = t0 + threadIdx.x;
        int v = t < p.ndc_tiles ? p.dc_part[(img * p.ndc_tiles + t) * 3 + comp] : 0;
        int x = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, d);
            if (int(threadIdx.x) >= d) x += y;
        }
        if (t < p.ndc_tiles) p.dc_part[(img * p.ndc_tiles + t) * 3 + comp] = carry + x - v;   // exclusive
        carry += __shfl_sync(0xffffffffu, x, 31);
    }
}

__global__ void __launch_bounds__(256) k_dc_apply(const DecParams p)
{
    pdl_wait();
    __shared__ int s_w[3][8];
    const size_t img = blockIdx.y;
    const uint32_t m = blockIdx.x * 256 + threadIdx.x;
    const size_t mc = min(m, p.nmcu - 1);
    int16_t* dd = p.dcd + img * p.nblk + mc * p.nb;
    int16_t* c = p.coefs + img * p.coef_stride + mc * p.nb * 64;
    int d[6] = {0, 0, 0, 0, 0, 0};
    if (m < p.nmcu) {
        for (uint32_t k = 0; k < p.nb; ++k) d[k] = dd[k];
    }
    int v[3] = {0, 0, 0};
    for (uint32_t k = 0; k < p.ny; ++k) v[0] += d[k];
    if (p.nb > p.ny) v[1] = d[p.ny], v[2] = d[p.ny + 1];
    int incl[3];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        int x = v[k];
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, s);
            if (lane >= s) x += y;
        }
        incl[k] = x;
        if (lane == 31) s_w[k][wid] = x;
    }
    __syncthreads();
    if (m >= p.nmcu) return;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        int base = p.dc_part[(img * p.ndc_tiles + blockIdx.x) * 3 + k];
        for (int w = 0; w < wid; ++w) base += s_w[k][w];
        incl[k] += base;   // inclusive prefix up to and including this MCU
    }
    int py = incl[0] - v[0];   // predictor before this MCU
    for (uint32_t k = 0; k < p.ny; ++k) {
        py += d[k];
        d[k] = py;
    }
    if (p.nb > p.ny) d[p.ny] = incl[1], d[p.ny + 1] = incl[2];
    bool dc_wide = false;     // a DC coefficient outside the int16 range of the coefficient format
    for (uint32_t k = 0; k < p.nb; ++k) {
        dd[k] = int16_t(d[k]);
        if (!p.dc_dense) c[k * 64] = int16_t(d[k]);
        dc_wide |= d[k] != int(int16_t(d[k]));
    }
    // (only over "ok": an EAGAIN of the first attempt keeps driving the host's retry)
    if (dc_wide && p.status) atomicCAS(p.status + img, 0, int(JPEZYB200_EUNSUPPORTED));
}

}  // namespace jz
