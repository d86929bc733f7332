// enc_huffopt.cuh -- per-image optimised Huffman tables, built on the device (the encoder's counterpart of libjpeg's
// -optimize).  The reference writes every image with the Annex K tables (src/encoder/huffman_table.hpp); it has no
// counterpart of this stage.
//
//   k_sym_hist     one thread per 8x8 block (tiled like k_block_bits): counts the symbols encode_block would emit, per
//                  image and table class, into counts[img][class][16 DC categories + 256 AC symbols]
//   k_huff_build   one CTA per image, one warp per table: T.81 section K.2 (Figures K.1-K.4) exactly as libjpeg's
//                  jpeg_gen_optimal_table does it; writes the image's HuffEncLut[2] for the entropy kernels, the
//                  jpezyb200_huff records for the caller, and clears the counts it consumed (the buffer is zeroed once,
//                  when it is allocated, so the chain needs neither a memset launch nor a host synchronisation)
#pragma once
#include "enc_entropy.cuh"

namespace jz {

constexpr int kHistBins = 16 + 256;   // per table class: DC categories, then AC symbols (run << 4) | size
// Code lengths before limiting: a Huffman tree whose deepest leaf sits at depth d needs a total count of at least
// Fib(d + 1); an image has fewer than 2^32 blocks of at most 64 symbols, so d < 60.
constexpr int kMaxCodeLen = 64;
constexpr int kHuffSlots = 9;         // ceil(257 / 32): live symbols (256 values + the reserved one) per lane

// The symbol walk of encode_block, counting instead of emitting.  A separate walk: running encode_block's own loop
// through a visitor changed the instruction schedule of k_block_bits and k_scatter.  Categories and sizes are clamped
// the same way, so a block with a coefficient that has no baseline code is counted as encode_block codes it (and the
// image still ends with scan_bytes = UINT64_MAX through k_block_bits).  Returns the DC category and whether EOB ends the
// block; AC symbols and ZRL go straight into the shared histogram s_ac.
__device__ __forceinline__ int count_block(const BlockRegs& blk, int dc_pred, uint32_t* s_ac, bool& eob)
{
    const int diff = blk.dc() - dc_pred;
    const int cat = min(bit_length(abs(diff)), 11);
    int run = 0;
#pragma unroll
    for (int n8 = 0; n8 < 8; ++n8) {
        const int4 q = blk.q[n8];
        if (n8 && (q.x | q.y | q.z | q.w) == 0) { run += 8; continue; }
        const uint32_t w[4] = {uint32_t(q.x), uint32_t(q.y), uint32_t(q.z), uint32_t(q.w)};
        uint32_t m = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t ne = __vsetne2(w[i], 0u);
            m |= ((ne & 1u) | (ne >> 15)) << (2 * i);
        }
        if (n8 == 0) m &= ~1u;
        int next = n8 == 0 ? 1 : 0;
        while (m) {
            const int h = __ffs(int(m)) - 1;
            m &= m - 1u;
            run += h - next;
            next = h + 1;
            const uint32_t ww = (h >> 1) == 0 ? w[0] : ((h >> 1) == 1 ? w[1] : ((h >> 1) == 2 ? w[2] : w[3]));
            const int v = (h & 1) ? (int(ww) >> 16) : int(short(ww & 0xffffu));
            if (run > 15) { atomicAdd(&s_ac[0xf0], uint32_t(run >> 4)); run &= 15; }
            const int s = min(bit_length(abs(v)), 10);
            atomicAdd(&s_ac[(run << 4) | s], 1u);
            run = 0;
        }
        run += 8 - next;
    }
    eob = run != 0;
    return cat;
}

template <bool RST>   // RST: the DC differences of a stream with restart intervals (enc_entropy.cuh)
__global__ void __launch_bounds__(kEntThreads) k_sym_hist(const EntParams p, unsigned long long* __restrict__ counts, const RstParams r)
{
    pdl_wait();
    __shared__ uint32_t s_cnt[2][kHistBins];
    for (int i = threadIdx.x; i < 2 * kHistBins; i += kEntThreads) (&s_cnt[0][0])[i] = 0;
    __syncthreads();
    const size_t img = blockIdx.y;
    const uint32_t b = blockIdx.x * kEntThreads + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int cls = (b % 6u) >= 4;
    int key = -1;   // DC bin of this thread's block, -1 past the last block
    bool eob = false;
    if (b < p.nblk) {
        const int16_t* base = p.coefs + img * p.coef_stride;
        const int comp = (b % 6u) < 4 ? 0 : int(b % 6u) - 3;
        BlockRegs blk;
        int pred;
        load_block(base, p.bmeta ? p.bmeta + img * p.nblk : nullptr, b, prev_same_component<RST>(b, r.rst),
                   p.dc_init ? p.dc_init[img * 3 + comp] : 0, blk, pred);
        key = cls * kHistBins + count_block(blk, pred, &s_cnt[cls][16], eob);
    }
    // DC categories and EOB are in nearly every block: one shared atomic per distinct bin of the warp, not one per block
    const uint32_t same = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && lane == __ffs(int(same)) - 1) atomicAdd(&(&s_cnt[0][0])[key], uint32_t(__popc(same)));
    const uint32_t eob_y = __ballot_sync(0xffffffffu, eob && cls == 0), eob_c = __ballot_sync(0xffffffffu, eob && cls == 1);
    if (lane == 0 && eob_y) atomicAdd(&s_cnt[0][16], uint32_t(__popc(eob_y)));
    if (lane == 1 && eob_c) atomicAdd(&s_cnt[1][16], uint32_t(__popc(eob_c)));
    __syncthreads();
    unsigned long long* g = counts + img * 2 * kHistBins;
    for (int i = threadIdx.x; i < 2 * kHistBins; i += kEntThreads) {
        const uint32_t c = (&s_cnt[0][0])[i];
        if (c) atomicAdd(g + i, (unsigned long long)c);
    }
}

__device__ __forceinline__ void min2_merge(unsigned long long& a1, unsigned long long& a2, unsigned long long b1, unsigned long long b2)
{
    // the two smallest of {a1 <= a2} and {b1 <= b2}
    const unsigned long long lo = a1 < b1 ? a1 : b1, hi = a1 < b1 ? b1 : a1;
    a2 = hi < (a2 < b2 ? a2 : b2) ? hi : (a2 < b2 ? a2 : b2);
    a1 = lo;
}

// Table w of image blockIdx.x: 0 = DC luma, 1 = AC luma, 2 = DC chroma, 3 = AC chroma.
// lut: [nimg][2] (class 0 luma, 1 chroma); ht: [nimg][2 = DC, AC][2 = luma, chroma]
__global__ void __launch_bounds__(128) k_huff_build(unsigned long long* __restrict__ counts, HuffEncLut* __restrict__ lut,
                                                    jpezyb200_huff* __restrict__ ht)
{
    pdl_wait();
    __shared__ unsigned long long s_freq[4][257];
    __shared__ uint16_t s_sym[4][257];
    __shared__ int s_len[4][kMaxCodeLen];    // symbols (without the reserved one) per code length of Figure K.1
    __shared__ int s_bits[4][kMaxCodeLen];   // BITS, Figures K.2 and K.3
    __shared__ int s_cum[4][18];             // codes shorter than L after limiting
    __shared__ int s_first[4][17];           // first code of length L
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cls = w >> 1, is_ac = w & 1;
    const size_t img = blockIdx.x;
    unsigned long long* cnt = counts + (img * 2 + cls) * kHistBins + (is_ac ? 16 : 0);
    const int nsym = is_ac ? 256 : 16;

    // live symbols, ascending, then the reserved symbol 256 with frequency 1 (K.2: no code word of all 1-bits)
    int n = 0;
    for (int c0 = 0; c0 < nsym; c0 += 32) {
        const int i = c0 + lane;
        unsigned long long f = 0;
        if (i < nsym) {
            f = cnt[i];
            cnt[i] = 0;
        }
        const uint32_t live = __ballot_sync(0xffffffffu, f != 0);
        if (f) {
            const int pos = n + __popc(live & ((1u << lane) - 1u));
            s_freq[w][pos] = f;
            s_sym[w][pos] = uint16_t(i);
        }
        n += __popc(live);
    }
    if (lane == 0) s_freq[w][n] = 1, s_sym[w][n] = 256;
    ++n;
    for (int i = lane; i < kMaxCodeLen; i += 32) s_len[w][i] = 0, s_bits[w][i] = 0;
    __syncwarp();

    // Figure K.1.  key = frequency << 9 | (511 - symbol): the smallest key is the smallest frequency, ties going to the
    // larger symbol (jpeg_gen_optimal_table); a merged tree keeps the key of its c1 root.  grp = root of the symbol's tree.
    unsigned long long key[kHuffSlots];
    int grp[kHuffSlots], csz[kHuffSlots];
#pragma unroll
    for (int k = 0; k < kHuffSlots; ++k) {
        const int j = k * 32 + lane;
        key[k] = j < n ? (s_freq[w][j] << 9) | uint64_t(511 - s_sym[w][j]) : ~0ull;
        grp[k] = j < n ? s_sym[w][j] : -1;
        csz[k] = 0;
    }
    for (;;) {
        unsigned long long m1 = ~0ull, m2 = ~0ull;
#pragma unroll
        for (int k = 0; k < kHuffSlots; ++k) min2_merge(m1, m2, key[k], ~0ull);
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const unsigned long long b1 = __shfl_xor_sync(0xffffffffu, m1, o), b2 = __shfl_xor_sync(0xffffffffu, m2, o);
            min2_merge(m1, m2, b1, b2);
        }
        if (m2 == ~0ull) break;   // one tree left
        const int c1 = 511 - int(m1 & 511u), c2 = 511 - int(m2 & 511u);
        const unsigned long long merged = (((m1 >> 9) + (m2 >> 9)) << 9) | (m1 & 511u);
#pragma unroll
        for (int k = 0; k < kHuffSlots; ++k) {
            key[k] = key[k] == m1 ? merged : (key[k] == m2 ? ~0ull : key[k]);
            const bool in = grp[k] == c1 || grp[k] == c2;   // the others[] chains of c1 and c2
            csz[k] += in ? 1 : 0;
            grp[k] = in ? c1 : grp[k];
        }
    }
    // Figure K.2
#pragma unroll
    for (int k = 0; k < kHuffSlots; ++k) {
        const int j = k * 32 + lane;
        if (j < n) {
            atomicAdd(&s_bits[w][csz[k]], 1);
            if (j < n - 1) atomicAdd(&s_len[w][csz[k]], 1);
        }
    }
    __syncwarp();
    if (lane == 0) {
        int* bits = s_bits[w];
        bits[0] = 0;   // a table of the reserved symbol alone (no real symbol): nothing to code
        // Figure K.3: limit the code lengths to 16, then give the reserved symbol's code point up
        for (int i = kMaxCodeLen - 1; i > 16; --i) {
            while (bits[i] > 0) {
                int j = i - 2;
                while (bits[j] == 0) --j;
                bits[i] -= 2;
                bits[i - 1] += 1;
                bits[j + 1] += 2;
                bits[j] -= 1;
            }
        }
        int i = 16;
        while (i > 0 && bits[i] == 0) --i;
        if (i > 0) bits[i] -= 1;
        // canonical codes (Annex C): codes shorter than L, first code of length L
        int code = 0, cum = 0;
        for (int L = 1; L <= 16; ++L) {
            s_cum[w][L] = cum, s_first[w][L] = code;
            cum += bits[L];
            code = (code + bits[L]) << 1;
        }
        s_cum[w][17] = cum;
        // Figure K.4 order: HUFFVAL position of the first symbol of each length before limiting
        int start = 0;
        for (int L = 1; L < kMaxCodeLen; ++L) {
            const int c = s_len[w][L];
            s_len[w][L] = start;
            start += c;
        }
    }
    __syncwarp();
    jpezyb200_huff* rec = ht + img * 4 + is_ac * 2 + cls;
    uint32_t* tab = is_ac ? lut[img * 2 + cls].ac : lut[img * 2 + cls].dc;
    for (int i = lane; i < 256; i += 32) rec->vals[i] = 0;
    for (int i = lane; i < nsym; i += 32) tab[i] = 0;
    if (lane < 16) rec->bits[lane] = uint8_t(s_bits[w][lane + 1]);
    if (lane == 0) rec->present = 1;
    __syncwarp();
    // Figure K.4: HUFFVAL by code length, then symbol value.  The slots of a lane hold ascending symbols k * 32 + lane,
    // so each round of 32 ranks its symbols among the equal lengths of the lower lanes.
#pragma unroll
    for (int k = 0; k < kHuffSlots; ++k) {
        const int j = k * 32 + lane;
        const int L = j < n - 1 ? csz[k] : 0;
        const uint32_t same = __match_any_sync(0xffffffffu, L);
        const int pos = L ? s_len[w][L] + __popc(same & ((1u << lane) - 1u)) : 0;
        __syncwarp();
        if (L && lane == __ffs(int(same)) - 1) s_len[w][L] += __popc(same);
        if (L && pos < s_cum[w][17]) {
            const int sym = s_sym[w][j];
            int len = 1;
            while (len < 16 && s_cum[w][len + 1] <= pos) ++len;
            rec->vals[pos] = uint8_t(sym);
            tab[sym] = (uint32_t(s_first[w][len] + pos - s_cum[w][len]) << 5) | uint32_t(len);
        }
        __syncwarp();
    }
}

}  // namespace jz
