// oracle/jpezy_oracle.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// CPU restatement of falgon/jpezy's baseline-JPEG encoder and decoder, used ONLY as the
// checker for the CUDA path (tests/, __graft_entry__.smoke(), bench.py's cpu_baseline /
// --impl reference legs).  Nothing under jpezy_b200/ may call into this file.
//
// Parity status: the reference cannot be built as shipped (SrookCppLibraries + Boost are
// absent and unpinned, SURVEY.md 8c).  Two pins exist:
//   (1) oracle/_ref (see oracle/Makefile, oracle/shim/): the reference's OWN headers
//       compiled unmodified from /root/reference against a minimal stand-in for the absent
//       third-party headers; tests/test_oracle_vs_ref.py compares this file against it.
//   (2) table / header known answers derived from ITU-T T.81 Annex K (tests/test_oracle_kat.py).
// The behaviour of the absent third-party pieces themselves (cosine table O1, 1/sqrt(2) O2,
// bit-writer padding O4, bit reader O6) is a recorded decision, "parity unpinned" at that
// sub-boundary.  Every function cites the reference file:line it restates.
//
// Build: see oracle/Makefile.  Canonical semantics = strict IEEE double, no FMA contraction
// (-ffp-contract=off, decision O3); the "as shipped" flag set is built beside it.

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>
#include <thread>
#include <chrono>
#include <atomic>

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

namespace orc {

// ---- src/jpezy.hpp:36-45 : zig-zag scan order (index n -> natural position) -------------
static const int kZZ[64] = {
    0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
    41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
    30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// ---- src/jpezy.hpp:131-152 : Annex K.1 / K.2 quantisation tables, natural order ----------
static const int kQY[64] = {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
                            14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
                            18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
                            49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
static const int kQC[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99,
                            24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99,
                            99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                            99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};

// ---- src/encoder/huffman_table.hpp:199-282 : the four DHT payloads (Annex K.3-K.6) -------
// Stored as BITS[16] + HUFFVAL[]; the encoder-side (size,code) LUTs of huffman_table.hpp:26-195
// are *derived* from these (canonical code construction, T.81 Annex C) and the derivation is
// checked against the reference's literal LUT values in tests/test_oracle_kat.py.
static const uint8_t kBitsDcY[16] = {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0};
static const uint8_t kBitsDcC[16] = {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0};
static const uint8_t kValsDc[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
static const uint8_t kBitsAcY[16] = {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d};
static const uint8_t kValsAcY[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71,
    0x14, 0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72,
    0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37,
    0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
    0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83,
    0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3,
    0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
    0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
    0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
static const uint8_t kBitsAcC[16] = {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77};
static const uint8_t kValsAcC[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22,
    0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1,
    0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36,
    0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
    0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a,
    0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a,
    0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
    0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
    0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};

// Encoder LUT in the reference's index space (huffman_table.hpp:26-195):
//   DC: index = category (0..11).   AC: index = run*10 + size + (run==15); EOB = 0, ZRL = 151.
struct EncLut {
    int dc_size[12], dc_code[12];
    int ac_size[162], ac_code[162];
};

static void canonical(const uint8_t* bits, const uint8_t* vals, int nvals, int* size_of_sym, int* code_of_sym)
{
    // T.81 Annex C.2 (Generate_size_table / Generate_code_table); same construction the
    // reference decoder uses in analyze_dht (src/decoder/jpezy_decoder.hpp:223-239).
    for (int i = 0; i < 256; ++i) size_of_sym[i] = 0, code_of_sym[i] = 0;
    int code = 0, k = 0;
    for (int len = 1; len <= 16; ++len) {
        for (int j = 0; j < bits[len - 1]; ++j, ++k) {
            if (k >= nvals) throw std::runtime_error("bad DHT");
            size_of_sym[vals[k]] = len;
            code_of_sym[vals[k]] = code++;
        }
        code <<= 1;
    }
}

static EncLut make_lut(const uint8_t* dcbits, const uint8_t* acbits, const uint8_t* acvals)
{
    EncLut t{};
    int sz[256], cd[256];
    canonical(dcbits, kValsDc, 12, sz, cd);
    for (int c = 0; c < 12; ++c) t.dc_size[c] = sz[c], t.dc_code[c] = cd[c];
    canonical(acbits, acvals, 162, sz, cd);
    t.ac_size[0] = sz[0x00], t.ac_code[0] = cd[0x00];        // EOB
    for (int run = 0; run < 16; ++run)
        for (int s = 1; s <= 10; ++s) {
            int idx = run * 10 + s + (run == 15);
            t.ac_size[idx] = sz[run * 16 + s], t.ac_code[idx] = cd[run * 16 + s];
        }
    t.ac_size[151] = sz[0xf0], t.ac_code[151] = cd[0xf0];    // ZRL
    return t;
}

static const EncLut& lutY() { static const EncLut t = make_lut(kBitsDcY, kBitsAcY, kValsAcY); return t; }
static const EncLut& lutC() { static const EncLut t = make_lut(kBitsDcC, kBitsAcC, kValsAcC); return t; }

// ---- decisions O1 / O2 (SURVEY.md 8c): constants produced by the absent third party ------
// O1: cos_table[u*8+x] = cos((2x+1) u pi / 16) in double (src/encoder/jpezy_encoder.hpp:271,
//     src/decoder/jpezy_decoder.hpp:698).  O2: 1.0 / sqrt(2.0) with IEEE sqrt and division.
struct Consts {
    double cos_table[64];
    double dis_sqrt;
    Consts()
    {
        for (int u = 0; u < 8; ++u)
            for (int x = 0; x < 8; ++x) cos_table[u * 8 + x] = std::cos((2 * x + 1) * u * M_PI / 16);
        volatile double two = 2.0;
        dis_sqrt = 1.0 / std::sqrt(two);
    }
};
static const Consts& K() { static const Consts c; return c; }

// ---- decision O4: MSB-first bit writer with FF->FF00 stuffing on bit writes ---------------
// Call sites: src/encoder/jpezy_encoder.hpp:189-220 (Bits), src/encoder/jpezy_writer.hpp:26-104
// (Byte/Word/Bytes).  pad_ones: value of the fill bits when a byte write follows a partial byte.
struct BitWriter {
    std::vector<uint8_t> buf;
    size_t cap;
    uint32_t acc = 0;
    int nacc = 0;     // bits pending in acc (0..7)
    uint64_t total_bits = 0;   // bits written through bits(), fill bits of align() included
    bool pad_ones;
    explicit BitWriter(size_t capacity, bool pad1) : cap(capacity), pad_ones(pad1) { buf.reserve(capacity < (1u << 20) ? capacity : (1u << 20)); }
    void put_raw(uint8_t b)
    {
        if (buf.size() >= cap) throw std::runtime_error("bofstream overflow");
        buf.push_back(b);
    }
    void bits(int n, int v)
    {
        total_bits += uint64_t(n > 0 ? n : 0);
        for (int i = n - 1; i >= 0; --i) {
            acc = (acc << 1) | ((static_cast<unsigned>(v) >> i) & 1u);
            if (++nacc == 8) {
                put_raw(static_cast<uint8_t>(acc));
                if ((acc & 0xff) == 0xff) put_raw(0x00);
                acc = 0, nacc = 0;
            }
        }
    }
    void align()
    {
        if (nacc) bits(8 - nacc, pad_ones ? 0xff : 0x00);
    }
    void byte(int b) { align(); put_raw(static_cast<uint8_t>(b)); }
    void word(int w) { byte((w >> 8) & 0xff); byte(w & 0xff); }
};

// ---- src/encoder/jpezy_writer.hpp:20-94 : header ----------------------------------------------
static void write_dht(BitWriter& w, int tc_th, const uint8_t* bits, const uint8_t* vals, int nvals)
{
    w.byte(0xff), w.byte(0xc4);
    w.word(2 + 1 + 16 + nvals);
    w.byte(tc_th);
    for (int i = 0; i < 16; ++i) w.byte(bits[i]);
    for (int i = 0; i < nvals; ++i) w.byte(vals[i]);
}

static void write_header(BitWriter& w, int W, int H, const char* comment)
{
    w.byte(0xff), w.byte(0xd8);                                   // SOI            :26
    w.byte(0xff), w.byte(0xe0);                                   // APP0 / JFIF    :29-37
    w.word(16);
    for (const char* p = "JFIF"; ; ++p) { w.byte(*p); if (!*p) break; }
    w.word(0x0102);
    w.byte(1);                                                    // Units::dots_inch (encode_io.hpp:152)
    w.word(96), w.word(96);
    w.byte(0), w.byte(0);
    size_t clen = std::strlen(comment);
    if (clen) {                                                   // COM            :40-44
        w.byte(0xff), w.byte(0xfe);
        w.word(static_cast<int>(clen + 3));
        for (size_t i = 0; i <= clen; ++i) w.byte(comment[i]);    // Byte_n(len+1): includes the NUL
    }
    for (int t = 0; t < 2; ++t) {                                 // DQT x2         :47-58
        w.byte(0xff), w.byte(0xdb);
        w.word(67);
        w.byte(t);
        for (int i = 0; i < 64; ++i) w.byte((t ? kQC : kQY)[kZZ[i]]);
    }
    write_dht(w, 0x00, kBitsDcY, kValsDc, 12);                    // DHT x4         :61-64
    write_dht(w, 0x01, kBitsDcC, kValsDc, 12);
    write_dht(w, 0x10, kBitsAcY, kValsAcY, 162);
    write_dht(w, 0x11, kBitsAcC, kValsAcC, 162);
    w.byte(0xff), w.byte(0xc0);                                   // SOF0           :67-81
    w.word(3 * 3 + 8);
    w.byte(8);
    w.word(H), w.word(W);
    w.byte(3);
    w.byte(0), w.byte(0x22), w.byte(0);
    for (int i = 1; i < 3; ++i) w.byte(i), w.byte(0x11), w.byte(1);
    w.byte(0xff), w.byte(0xda);                                   // SOS            :84-93
    w.word(2 * 3 + 6);
    w.byte(3);
    for (int i = 0; i < 3; ++i) w.byte(i), w.byte(i == 0 ? 0 : 0x11);
    w.byte(0), w.byte(63), w.byte(0);
}

// ---- src/encoder/jpezy_encoder.hpp:244-256 : colour formulas ------------------------------------
static inline int rgbY(int r, int g, int b) { return int((0.2990 * r) + (0.5870 * g) + (0.1140 * b) - 128); }
static inline int rgbCb(int r, int g, int b) { return int(-(0.1687 * r) - (0.3313 * g) + (0.5000 * b)); }
static inline int rgbCr(int r, int g, int b) { return int((0.5000 * r) - (0.4187 * g) - (0.0813 * b)); }

struct Encoder {
    int W, H;
    const uint8_t *r, *g, *b;
    bool gray;
    int Yb[4][64], Cbb[64], Crb[64], F[64];
    double Fraw[64];
    int preDC[3] = {0, 0, 0};

    // src/encoder/jpezy_encoder.hpp:90-144
    void make_ycc(int ux, int uy)
    {
        int cbfull[4][64], crfull[4][64];
        for (int i = 0; i < 4; ++i) {
            int n = 0;
            for (int sy = uy * 16 + ((i > 1) ? 8 : 0), e = sy + 8; sy < e; ++sy) {
                const int ii = sy < H ? sy : H - 1;
                for (int sx = ux * 16 + ((i & 1) ? 8 : 0), ex = sx + 8; sx < ex; ++sx, ++n) {
                    const int jj = sx < W ? sx : W - 1;
                    const size_t idx = static_cast<size_t>(ii) * W + jj;
                    Yb[i][n] = rgbY(r[idx], g[idx], b[idx]);
                    cbfull[i][n] = rgbCb(r[idx], g[idx], b[idx]);
                    crfull[i][n] = rgbCr(r[idx], g[idx], b[idx]);
                }
            }
        }
        static const int base[4] = {0, 4, 32, 36};
        for (int i = 0; i < 4; ++i) {
            int n = base[i];
            for (int y = 0; y < 8; y += 2) {
                for (int x = 0; x < 8; x += 2, ++n) Crb[n] = crfull[i][y * 8 + x], Cbb[n] = cbfull[i][y * 8 + x];
                n += 4;
            }
        }
    }
    // src/encoder/jpezy_encoder.hpp:146-166
    void dct(const int* pic)
    {
        const double* ct = K().cos_table;
        const double ds = K().dis_sqrt;
        for (int i = 0; i < 8; ++i) {
            const double cv = i ? 1.0 : ds;
            for (int j = 0; j < 8; ++j) {
                const double cu = j ? 1.0 : ds;
                double sum = 0;
                for (int y = 0; y < 8; ++y)
                    for (int x = 0; x < 8; ++x) sum += pic[y * 8 + x] * ct[j * 8 + x] * ct[i * 8 + y];
                const double v = sum * cu * cv / 4;
                Fraw[i * 8 + j] = v;
                F[i * 8 + j] = int(v);
            }
        }
    }
    // src/encoder/jpezy_encoder.hpp:168-172
    void quant(int cs)
    {
        const int* q = cs ? kQC : kQY;
        for (int i = 0; i < 64; ++i) F[i] /= q[i];
    }
    // src/encoder/jpezy_encoder.hpp:174-225
    void huff(int cs, BitWriter& w, const EncLut& t)
    {
        const int diff = F[0] - preDC[cs];
        preDC[cs] = F[0];
        int di = 0;
        for (int a = std::abs(diff); a > 0; a >>= 1) ++di;
        if (di > 12) throw std::runtime_error("encode_huffman");
        w.bits(t.dc_size[di], t.dc_code[di]);
        if (di) w.bits(di, diff < 0 ? diff - 1 : diff);
        int run = 0;
        for (int n = 1; n < 64; ++n) {
            int a = std::abs(F[kZZ[n]]);
            if (a) {
                while (run > 15) w.bits(t.ac_size[151], t.ac_code[151]), run -= 16;
                int s = 0;
                for (; a > 0; a >>= 1) ++s;
                const int idx = run * 10 + s + (run == 15);
                if (idx >= 162) throw std::runtime_error("encode_huffman");
                w.bits(t.ac_size[idx], t.ac_code[idx]);
                int v = F[kZZ[n]];
                if (v < 0) --v;
                w.bits(s, v);
                run = 0;
            } else if (n == 63) {
                w.bits(t.ac_size[0], t.ac_code[0]);
            } else {
                ++run;
            }
        }
    }
};

// coefficient sink: zig-zag int16, MCU-major, block order Y0 Y1 Y2 Y3 Cb Cr
static inline void store_zz(const int* F, int16_t* out)
{
    for (int n = 0; n < 64; ++n) out[n] = static_cast<int16_t>(F[kZZ[n]]);
}

// src/encoder/jpezy_encoder.hpp:38-77 (+227-242).  If coefs != nullptr the quantised
// coefficients are emitted; if raw != nullptr the pre-truncation DCT values (natural order)
// are emitted; if w != nullptr the entropy-coded segment is produced.
static void encode_core(Encoder& e, BitWriter* w, int16_t* coefs, double* raw)
{
    const int VU = e.H / 16 + ((e.H % 16) ? 1 : 0);
    const int HU = e.W / 16 + ((e.W % 16) ? 1 : 0);
    size_t blk = 0;
    for (int y = 0; y < VU; ++y)
        for (int x = 0; x < HU; ++x) {
            e.make_ycc(x, y);
            if (e.gray) std::memset(e.Cbb, 0, sizeof e.Cbb), std::memset(e.Crb, 0, sizeof e.Crb);
            for (int k = 0; k < 6; ++k, ++blk) {
                const int cs = k < 4 ? 0 : k - 3;
                e.dct(k < 4 ? e.Yb[k] : (k == 4 ? e.Cbb : e.Crb));
                if (raw) std::memcpy(raw + blk * 64, e.Fraw, sizeof e.Fraw);
                e.quant(cs);
                if (coefs) store_zz(e.F, coefs + blk * 64);
                if (w) e.huff(cs, *w, cs ? lutC() : lutY());
            }
        }
}

// entropy-code a given coefficient array (zig-zag, scan order) -- lets the tests check
// "given identical coefficients the stream is byte-identical" independently of the DCT.
// restart_interval > 0: after every restart_interval MCUs but the last, the predictors are reset, the
// segment is padded to a byte and RSTn is written (T.81 F.1.2.3 / E.1.4; the decoder side is :152-163).
template <typename T>
static void encode_from_coefs(const T* coefs, size_t nmcu, BitWriter& w, int restart_interval = 0)
{
    Encoder e{};
    for (size_t m = 0; m < nmcu; ++m) {
        if (restart_interval > 0 && m > 0 && m % size_t(restart_interval) == 0) {
            w.align();
            w.byte(0xff), w.byte(0xd0 + int((m / size_t(restart_interval) - 1) & 7));
            e.preDC[0] = e.preDC[1] = e.preDC[2] = 0;
        }
        for (int k = 0; k < 6; ++k) {
            const int cs = k < 4 ? 0 : k - 3;
            const T* c = coefs + (m * 6 + k) * 64;
            for (int n = 0; n < 64; ++n) e.F[kZZ[n]] = int(c[n]);
            e.huff(cs, w, cs ? lutC() : lutY());
        }
    }
}

// ================================= decoder =====================================================

// decision O6: MSB-first bit reader, drops the 00 that follows FF inside entropy data,
// returns <0 on exhaustion (src/decoder/jpezy_decoder.hpp:634-635).
struct BitReader {
    const uint8_t* p;
    size_t n, pos = 0;
    uint32_t cur = 0;
    int left = 0;
    BitReader(const uint8_t* d, size_t len) : p(d), n(len) {}
    int byte()
    {
        left = 0;
        if (pos >= n) return -1;
        return p[pos++];
    }
    int word()
    {
        int a = byte(), b = byte();
        if (a < 0 || b < 0) return -1;
        return (a << 8) | b;
    }
    int bit()
    {
        if (!left) {
            if (pos >= n) return -1;
            cur = p[pos++];
            if (cur == 0xff && pos < n && p[pos] == 0x00) ++pos;
            left = 8;
        }
        --left;
        return (cur >> left) & 1;
    }
    int bits(int k)
    {
        int v = 0;
        for (int i = 0; i < k; ++i) {
            int b = bit();
            if (b < 0) return -1;
            v = (v << 1) | b;
        }
        return v;
    }
    void skip(long k) { left = 0; pos = (k < 0 && size_t(-k) > pos) ? 0 : pos + k; if (pos > n) pos = n; }
};

struct HuffDec {
    std::vector<int> size, code, value;
};

struct Decoder {
    BitReader br;
    int W = 0, H = 0, ncomp = 0, prec = 0;
    int restart_interval = 0;
    int hmax = 0, vmax = 0;
    struct { int C, Hs, Vs, Tq; } fc[3]{};
    struct { int Cs, Td, Ta; } sc[3]{};
    HuffDec ht[2][4];
    int qt[4][64]{};
    int pred[3] = {0, 0, 0};
    int dctc[64], block[64];
    bool have_ht = false, have_qt = false, have_sos = false;
    std::string comment;
    Decoder(const uint8_t* d, size_t n) : br(d, n) {}

    // src/decoder/jpezy_decoder.hpp:486-502
    int get_marker()
    {
        for (;;) {
            int c = br.byte();
            if (c < 0) throw std::runtime_error("eof");
            if (c == 0xff) {
                c = br.byte();
                if (c < 0) throw std::runtime_error("eof");
                if (c) {
                    if (c > 0x02 && c < 0xc0) return 0xff;
                    return c;
                }
            }
        }
    }
    // :190-256
    void dht(int size)
    {
        const size_t end = br.pos + size;
        do {
            int uc = br.byte();
            int tc = uc >> 4, th = uc & 15;
            if (tc > 1 || th > 3) throw std::runtime_error("DHT format error");
            HuffDec& h = ht[tc][th];
            int cc[16], n = 0;
            for (int i = 0; i < 16; ++i) cc[i] = br.byte(), n += cc[i];
            h.size.assign(n, 0), h.code.assign(n, 0), h.value.assign(n, 0);
            for (int i = 1, k = 0; i <= 16; ++i)
                for (int j = 1; j <= cc[i - 1]; ++j, ++k) h.size[k] = i;
            int code = 0, k = 0;
            for (int len = 1; len <= 16 && k < n; ++len) {
                while (k < n && h.size[k] == len) h.code[k++] = code++;
                code <<= 1;
            }
            for (int i = 0; i < n; ++i) h.value[i] = br.byte();
        } while (br.pos < end);
    }
    // :258-277
    void dqt(int size)
    {
        const size_t end = br.pos + size;
        do {
            int c = br.byte();
            int* q = qt[c & 3];
            if (!(c >> 4)) for (int i = 0; i < 64; ++i) q[kZZ[i]] = br.byte();
            else for (int i = 0; i < 64; ++i) q[kZZ[i]] = br.word();
        } while (br.pos < end);
    }
    // :279-305
    void frame()
    {
        prec = br.byte();
        H = br.word();
        W = br.word();
        ncomp = br.byte();
        if (ncomp != 3 && ncomp != 1) throw std::runtime_error("dimension");
        for (int i = 0; i < ncomp; ++i) {
            fc[i].C = br.byte();
            int c = br.byte();
            fc[i].Hs = c >> 4, fc[i].Vs = c & 15;
            if (fc[i].Hs > hmax) hmax = fc[i].Hs;
            if (fc[i].Vs > vmax) vmax = fc[i].Vs;
            fc[i].Tq = br.byte();
        }
    }
    // :307-334
    void scan()
    {
        int ns = br.byte();
        for (int i = 0; i < ns && i < 3; ++i) {
            sc[i].Cs = br.byte();
            int c = br.byte();
            sc[i].Td = c >> 4, sc[i].Ta = c & 15;
            if (sc[i].Td > 2 || sc[i].Ta > 2) throw std::runtime_error("scan");
        }
        br.byte(), br.byte(), br.byte();
    }
    // :360-484 ; returns true when SOS has been consumed
    bool marker()
    {
        const int m = get_marker();
        int len;
        switch (m) {
        case 0xc0: len = br.word(); (void)len; frame(); return false;
        case 0xc4: len = br.word() - 2; dht(len); have_ht = true; return false;
        case 0xdc: br.word(); H = br.word(); return false;
        case 0xdb: len = br.word() - 2; dqt(len); have_qt = true; return false;
        case 0xd9: throw std::runtime_error("EOI before SOS");
        case 0xda: br.word(); scan(); have_sos = true; return true;
        case 0xdd: br.word(); restart_interval = br.word(); return false;
        case 0xfe: {
            len = br.word() - 2;
            comment.clear();
            for (int i = 0; i < len; ++i) comment.push_back(static_cast<char>(br.byte()));
            return false;
        }
        case 0xe0: {
            len = br.word() - 2;
            if (len >= 4) {
                char id[5];
                for (int i = 0; i < 5; ++i) id[i] = static_cast<char>(br.byte());
                if (!std::memcmp(id, "JFIF", 4)) { for (int i = 0; i < 9; ++i) br.byte(); br.skip(len - 14); }
                else if (!std::memcmp(id, "JFXX", 4)) { br.byte(); br.skip(len - 1); }
                else br.skip(len - 4);
            } else br.skip(len);
            return false;
        }
        default:
            if (m >= 0xe1 && m <= 0xef) { len = br.word() - 2; br.skip(len); return false; }
            if ((m >= 0xc1 && m <= 0xcf && m != 0xc8) || m == 0xde || m == 0xdf) return false;  // "Not supported": exception object built but never thrown (:412-421)
            throw std::runtime_error("Marker error");
        }
    }
    void header()
    {
        while (get_marker() != 0xd8) {}
        while (!marker()) {}
    }
    // :626-642 (table selector quirk: Td used for both DC and AC)
    int sym(int is_ac, int s)
    {
        const HuffDec& h = ht[is_ac][sc[s].Td];
        int code = 0;
        size_t k = 0;
        for (int length = 0; k < h.size.size() && length < 16;) {
            ++length;
            code <<= 1;
            int nx = br.bit();
            if (nx < 0) return nx;
            code |= nx;
            for (; k < h.size.size() && h.size[k] == length; ++k)
                if (h.code[k] == code) return h.value[k];
        }
        throw std::runtime_error("decode_huffman_impl");
    }
    // :583-624
    void huff(int s)
    {
        int diff = 0;
        int cat = sym(0, s);
        if (cat > 0) {
            diff = br.bits(cat);
            if ((diff & (1 << (cat - 1))) == 0) diff -= (1 << cat) - 1;
        } else if (cat < 0) throw std::runtime_error("decode_huffman");
        pred[s] += diff;
        dctc[0] = pred[s];
        for (int k = 1; k < 64;) {
            cat = sym(1, s);
            if (!cat) { for (; k < 64; ++k) dctc[kZZ[k]] = 0; break; }
            if (cat < 0) throw std::runtime_error("decode_huffman");
            int run = cat >> 4, acv = 0;
            cat &= 15;
            if (cat) {
                acv = br.bits(cat);
                if (!(acv & (1 << (cat - 1)))) acv -= (1 << cat) - 1;
            }
            if (run + k > 63) throw std::runtime_error("decode_huffman");
            for (; run-- > 0; ++k) dctc[kZZ[k]] = 0;
            dctc[kZZ[k++]] = acv;
        }
    }
    // :645-650
    void dequant(int s) { const int* q = qt[fc[s].Tq]; for (int i = 0; i < 64; ++i) dctc[i] *= q[i]; }
    // :652-670
    void idct()
    {
        const int sl = prec == 8 ? 128 : 2048;
        const double* ct = K().cos_table;
        const double ds = K().dis_sqrt;
        for (int y = 0; y < 8; ++y)
            for (int x = 0; x < 8; ++x) {
                double sum = 0;
                for (int v = 0; v < 8; ++v) {
                    const double cv = (!v) ? ds : 1.0;
                    for (int u = 0; u < 8; ++u) {
                        const double cu = (!u) ? ds : 1.0;
                        sum += cu * cv * dctc[v * 8 + u] * ct[u * 8 + x] * ct[v * 8 + y];
                    }
                }
                block[y * 8 + x] = int(sum / 4 + sl);
            }
    }
    static inline uint8_t revise(double v) { return v < 0.0 ? 0 : (v > 255.0 ? 255 : static_cast<uint8_t>(v)); }
};

// MCU geometry (src/decoder/jpezy_decoder.hpp:94-101): hu x vu MCUs, planes of plane_len bytes
struct Geom {
    size_t hu, vu, plane_len;
};
static Geom geometry(const Decoder& d)
{
    const size_t Vb = (d.H >> 3) + ((d.H & 7) > 0), Hb = (d.W >> 3) + ((d.W & 7) > 0);
    Geom g;
    g.hu = Hb / d.hmax + ((Hb % d.hmax) ? 1 : 0), g.vu = Vb / d.vmax + ((Vb % d.vmax) ? 1 : 0);
    g.plane_len = (g.vu * d.vmax) * 8 * (g.hu * d.hmax) * 8;
    return g;
}

// The pixel stage of one MCU, shared by the file decoder and orc_pixels_from_coefs: the component tiles
// (value-initialised as at :105) and make_rgb (:531-565).
struct PixelStage {
    std::vector<int> comp[3];
    size_t vstep;
    explicit PixelStage(const Decoder& d)
    {
        const size_t unit = size_t(d.hmax) * d.vmax * 64;
        comp[0].assign(unit, 0), comp[1].assign(unit, 0x80), comp[2].assign(unit, 0x80);
        vstep = size_t(d.hmax) * 8;
    }
    // block (ky, kx) of component s, quantised coefficients in d.dctc (natural order): dequant, idct and the pixel
    // replication of decode_mcu (:519-524)
    void block(Decoder& d, int s, int ky, int kx)
    {
        const int dy = d.vmax / d.fc[s].Vs, dx = d.hmax / d.fc[s].Hs;
        d.dequant(s);
        d.idct();
        int* tp = comp[s].data() + ky * vstep * 8 + kx * 8;
        for (int yu = 0; yu < 8 * dy; ++yu)
            for (int xu = 0; xu < 8 * dx; ++xu) tp[yu * vstep + xu] = d.block[(yu / dy) * 8 + (xu / dx)];
    }
    // make_rgb :531-565
    void rgb(const Decoder& d, size_t ux, size_t uy, bool gray, std::vector<uint8_t>* planes) const
    {
        const int *yp = comp[0].data(), *up = comp[1].data(), *vp = comp[2].data();
        const size_t off_h = ux * d.hmax * 8;
        const size_t off = uy * d.vmax * 8 * size_t(d.W) + off_h;
        const size_t ex = size_t(d.hmax) * 8, ey = size_t(d.vmax) * 8;
        for (size_t py = 0; py < ey; ++py)
            for (size_t px = 0; px < ex; ++px) {
                if (px + off_h >= size_t(d.W)) { yp += ex - px, up += ex - px, vp += ex - px; break; }
                const size_t idx = off + py * d.W + px;
                if (!gray) {
                    const double Y = *yp, U = *up, V = *vp;
                    planes[0][idx] = Decoder::revise(Y + (V - 0x80) * 1.4020);
                    planes[1][idx] = Decoder::revise(Y - (U - 0x80) * 0.3441 - (V - 0x80) * 0.7139);
                    planes[2][idx] = Decoder::revise(Y + (U - 0x80) * 1.7718);
                    ++yp, ++up, ++vp;
                } else {
                    planes[0][idx] = planes[1][idx] = planes[2][idx] = Decoder::revise(*yp++);
                }
            }
    }
};

// src/decoder/jpezy_decoder.hpp:76-134 + 504-565.  Outputs: planes of plane_len bytes (zero
// filled beyond what the MCU loop writes), optional coefficient dump (zig-zag int16, scan order,
// DC already de-predicted = absolute).
static int decode_core(const uint8_t* file, size_t n, bool gray, std::vector<uint8_t>* planes, int* Wout, int* Hout,
                       std::vector<int16_t>* coefs)
{
    Decoder d(file, n);
    try { d.header(); } catch (const std::exception&) { return 1; }
    // :89 only requires one of is_htable|is_qtable|is_start_data; SOS is always set here.
    if (d.hmax <= 0 || d.vmax <= 0) return 1;   // the reference would divide by zero (no SOF0 seen)
    const Geom g = geometry(d);
    *Wout = d.W, *Hout = d.H;
    if (planes) for (int c = 0; c < 3; ++c) planes[c].assign(g.plane_len, 0);
    PixelStage px(d);
    size_t restart_counter = 0;
    try {
        for (size_t uy = 0; uy < g.vu; ++uy)
            for (size_t ux = 0; ux < g.hu; ++ux) {
                for (int s = 0; s < d.ncomp; ++s) {                      // decode_mcu :504-528
                    const int nv = d.fc[s].Vs, nh = d.fc[s].Hs;
                    if (nv <= 0 || nh <= 0) return 2;
                    for (int ky = 0; ky < nv; ++ky)
                        for (int kx = 0; kx < nh; ++kx) {
                            d.huff(s);
                            if (coefs) { for (int k = 0; k < 64; ++k) coefs->push_back(static_cast<int16_t>(d.dctc[kZZ[k]])); }
                            px.block(d, s, ky, kx);
                        }
                }
                if (planes) px.rgb(d, ux, uy, gray, planes);
                if (d.restart_interval && ++restart_counter >= size_t(d.restart_interval)) {   // :152-163
                    restart_counter = 0;
                    try {
                        const int m = d.get_marker();
                        if (m >= 0xd0 && m <= 0xd7) d.pred[0] = d.pred[1] = d.pred[2] = 0;
                    } catch (const std::exception&) {}
                }
            }
    } catch (const std::exception&) { return 2; }
    return 0;
}

} // namespace orc

// ======================================= C ABI for ctypes =======================================
extern "C" {

// number of MCUs / blocks for a WxH image (16x16 MCUs, 6 blocks each)
size_t orc_num_mcus(int W, int H) { return size_t((W + 15) / 16) * size_t((H + 15) / 16); }

// planar RGB -> quantised zig-zag int16 coefficients (+ optional raw FP64 DCT values, natural order)
int orc_coefs(const uint8_t* r, const uint8_t* g, const uint8_t* b, int W, int H, int gray, int16_t* coefs, double* raw)
{
    orc::Encoder e{};
    e.W = W, e.H = H, e.r = r, e.g = g, e.b = b, e.gray = gray != 0;
    try { orc::encode_core(e, nullptr, coefs, raw); } catch (const std::exception&) { return 1; }
    return 0;
}

// planar RGB -> complete JPEG file (header + scan + EOI), as jpezy::encoder::encode would write it.
// mode: 0 file, 1 scan segment only (stuffed, padded).  Returns 0 ok, 1 error/overflow.
int orc_encode(const uint8_t* r, const uint8_t* g, const uint8_t* b, int W, int H, int gray, int pad_ones, int scan_only,
               uint8_t* out, size_t cap, size_t* out_len)
{
    try {
        size_t size = size_t(W) * size_t(H) * 3;                  // decision O5: size_t, not int
        if (size < 10240) size = 10240;
        orc::BitWriter w(size, pad_ones != 0);
        if (!scan_only) orc::write_header(w, W, H, gray ? "Encoded by JPEZY" : "Encoded by jpezy");
        orc::Encoder e{};
        e.W = W, e.H = H, e.r = r, e.g = g, e.b = b, e.gray = gray != 0;
        orc::encode_core(e, &w, nullptr, nullptr);
        if (scan_only) w.align();
        else w.byte(0xff), w.byte(0xd9);                           // write_eoi, jpezy_writer.hpp:101-105
        *out_len = w.buf.size();
        if (w.buf.size() > cap) return 1;
        std::memcpy(out, w.buf.data(), w.buf.size());
    } catch (const std::exception&) { return 1; }
    return 0;
}

int orc_header(int W, int H, int gray, uint8_t* out, size_t cap, size_t* out_len)
{
    orc::BitWriter w(4096, true);
    orc::write_header(w, W, H, gray ? "Encoded by JPEZY" : "Encoded by jpezy");
    *out_len = w.buf.size();
    if (w.buf.size() > cap) return 1;
    std::memcpy(out, w.buf.data(), w.buf.size());
    return 0;
}

// coefficients (zig-zag int16, scan order) -> stuffed + padded entropy segment
int orc_scan_from_coefs(const int16_t* coefs, size_t nmcu, int pad_ones, uint8_t* out, size_t cap, size_t* out_len, uint64_t* nbits)
{
    try {
        orc::BitWriter w(cap, pad_ones != 0);
        orc::encode_from_coefs(coefs, nmcu, w);
        if (nbits) *nbits = w.total_bits;   // before the fill bits
        w.align();
        *out_len = w.buf.size();
        std::memcpy(out, w.buf.data(), w.buf.size());
    } catch (const std::exception&) { return 1; }
    return 0;
}

// coefficients (zig-zag int32, scan order, 4:2:0 MCUs) -> stuffed + padded entropy segment, with RSTn markers every
// restart_interval MCUs when it is > 0
int orc_scan_from_coefs32(const int32_t* coefs, size_t nmcu, int pad_ones, int restart_interval, uint8_t* out, size_t cap, size_t* out_len,
                          uint64_t* nbits)
{
    try {
        orc::BitWriter w(cap, pad_ones != 0);
        orc::encode_from_coefs(coefs, nmcu, w, restart_interval);
        if (nbits) *nbits = w.total_bits;   // before the fill bits
        w.align();
        *out_len = w.buf.size();
        std::memcpy(out, w.buf.data(), w.buf.size());
    } catch (const std::exception&) { return 1; }
    return 0;
}

// JPEG file -> geometry (W, H, padded plane length as in jpezy_decoder.hpp:94-101); ncomp / hs / vs / nblocks may be null
int orc_probe(const uint8_t* file, size_t n, int* W, int* H, size_t* plane_len, int* ncomp, int* hs, int* vs, size_t* nblocks)
{
    orc::Decoder d(file, n);
    try { d.header(); } catch (const std::exception&) { return 1; }
    if (d.hmax <= 0 || d.vmax <= 0) return 1;
    const orc::Geom g = orc::geometry(d);
    *W = d.W, *H = d.H, *plane_len = g.plane_len;
    size_t nb = 0;
    for (int i = 0; i < d.ncomp; ++i) {
        if (hs) hs[i] = d.fc[i].Hs;
        if (vs) vs[i] = d.fc[i].Vs;
        nb += size_t(d.fc[i].Hs) * d.fc[i].Vs;
    }
    if (ncomp) *ncomp = d.ncomp;
    if (nblocks) *nblocks = nb * g.hu * g.vu;
    return 0;
}

// quantised coefficients (zig-zag int32, scan order, absolute DC, the blocks of every MCU in decode_mcu's order) ->
// planar RGB of plane_len bytes each, through the file decoder's own dequant / idct / replication / make_rgb.
// qt: one table per component, natural order.  Returns 0 ok, 1 bad layout, 3 planes too small.
int orc_pixels_from_coefs(const int32_t* coefs, size_t ncoefs, int W, int H, int ncomp, const int* hs, const int* vs, const uint16_t* qt,
                          int gray, uint8_t* r, uint8_t* g, uint8_t* b, size_t plane_len)
{
    if ((ncomp != 1 && ncomp != 3) || W <= 0 || H <= 0) return 1;
    orc::Decoder d(nullptr, 0);
    d.W = W, d.H = H, d.ncomp = ncomp, d.prec = 8;
    size_t nb = 0;
    for (int i = 0; i < ncomp; ++i) {
        if (hs[i] <= 0 || vs[i] <= 0) return 1;
        d.fc[i].Hs = hs[i], d.fc[i].Vs = vs[i], d.fc[i].Tq = i;
        d.hmax = std::max(d.hmax, hs[i]), d.vmax = std::max(d.vmax, vs[i]);
        for (int k = 0; k < 64; ++k) d.qt[i][k] = qt[i * 64 + k];
        nb += size_t(hs[i]) * vs[i];
    }
    for (int i = 0; i < ncomp; ++i)
        if (d.hmax % hs[i] || d.vmax % vs[i]) return 1;
    const orc::Geom geo = orc::geometry(d);
    if (ncoefs != geo.hu * geo.vu * nb * 64) return 1;
    if (geo.plane_len > plane_len) return 3;
    std::vector<uint8_t> planes[3];
    for (int c = 0; c < 3; ++c) planes[c].assign(geo.plane_len, 0);
    orc::PixelStage px(d);
    const int32_t* c = coefs;
    for (size_t uy = 0; uy < geo.vu; ++uy)
        for (size_t ux = 0; ux < geo.hu; ++ux) {
            for (int s = 0; s < ncomp; ++s)
                for (int ky = 0; ky < vs[s]; ++ky)
                    for (int kx = 0; kx < hs[s]; ++kx, c += 64) {
                        for (int k = 0; k < 64; ++k) d.dctc[orc::kZZ[k]] = c[k];
                        px.block(d, s, ky, kx);
                    }
            px.rgb(d, ux, uy, gray != 0, planes);
        }
    std::memcpy(r, planes[0].data(), geo.plane_len);
    std::memcpy(g, planes[1].data(), geo.plane_len);
    std::memcpy(b, planes[2].data(), geo.plane_len);
    return 0;
}

// JPEG file -> planar RGB (each plane plane_len bytes, stride W)
int orc_decode(const uint8_t* file, size_t n, int gray, uint8_t* r, uint8_t* g, uint8_t* b, size_t plane_len)
{
    std::vector<uint8_t> planes[3];
    int W, H;
    int rc = orc::decode_core(file, n, gray != 0, planes, &W, &H, nullptr);
    if (rc) return rc;
    if (planes[0].size() > plane_len) return 3;
    std::memcpy(r, planes[0].data(), planes[0].size());
    std::memcpy(g, planes[1].data(), planes[1].size());
    std::memcpy(b, planes[2].data(), planes[2].size());
    return 0;
}

// JPEG file -> entropy-decoded coefficients (zig-zag int16, scan order, absolute DC)
int orc_decode_coefs(const uint8_t* file, size_t n, int16_t* coefs, size_t cap_coefs, size_t* ncoefs)
{
    std::vector<int16_t> c;
    int W, H;
    int rc = orc::decode_core(file, n, false, nullptr, &W, &H, &c);
    if (rc) return rc;
    *ncoefs = c.size();
    if (c.size() > cap_coefs) return 3;
    std::memcpy(coefs, c.data(), c.size() * sizeof(int16_t));
    return 0;
}

// encoder LUTs in the reference's index space, for the table known-answer tests
void orc_enc_lut(int chroma, int* dc_size, int* dc_code, int* ac_size, int* ac_code)
{
    const orc::EncLut& t = chroma ? orc::lutC() : orc::lutY();
    std::memcpy(dc_size, t.dc_size, sizeof t.dc_size), std::memcpy(dc_code, t.dc_code, sizeof t.dc_code);
    std::memcpy(ac_size, t.ac_size, sizeof t.ac_size), std::memcpy(ac_code, t.ac_code, sizeof t.ac_code);
}
void orc_tables(int* zz, int* qy, int* qc, double* cos_table, double* dis_sqrt)
{
    std::memcpy(zz, orc::kZZ, sizeof orc::kZZ), std::memcpy(qy, orc::kQY, sizeof orc::kQY), std::memcpy(qc, orc::kQC, sizeof orc::kQC);
    std::memcpy(cos_table, orc::K().cos_table, 64 * sizeof(double));
    *dis_sqrt = orc::K().dis_sqrt;
}

// ---- CPU baseline timing (bench.py cpu_baseline / --impl reference) -----------------------------
// Runs `reps` encode (+decode) round trips of one WxH image on `nthreads` threads (each thread its
// own copy of the work = "one instance per core"); returns wall seconds for the slowest thread.
// Timed region = encoder::encode() to memory + decoder::decode() from memory (PPM I/O excluded).
double orc_time_roundtrip(const uint8_t* r, const uint8_t* g, const uint8_t* b, int W, int H, int gray, int reps, int nthreads,
                          double* enc_seconds, double* dec_seconds)
{
    std::vector<double> te(nthreads, 0.0), td(nthreads, 0.0);
    auto work = [&](int t) {
        const size_t cap = std::max<size_t>(size_t(W) * H * 3, 10240);
        std::vector<uint8_t> file(cap);
        for (int i = 0; i < reps; ++i) {
            size_t len = 0;
            auto t0 = std::chrono::steady_clock::now();
            orc_encode(r, g, b, W, H, gray, 1, 0, file.data(), cap, &len);
            auto t1 = std::chrono::steady_clock::now();
            std::vector<uint8_t> planes[3];
            int w2, h2;
            orc::decode_core(file.data(), len, gray != 0, planes, &w2, &h2, nullptr);
            auto t2 = std::chrono::steady_clock::now();
            te[t] += std::chrono::duration<double>(t1 - t0).count();
            td[t] += std::chrono::duration<double>(t2 - t1).count();
        }
    };
    auto T0 = std::chrono::steady_clock::now();
    std::vector<std::thread> th;
    for (int t = 1; t < nthreads; ++t) th.emplace_back(work, t);
    work(0);
    for (auto& x : th) x.join();
    auto T1 = std::chrono::steady_clock::now();
    double me = 0, md = 0;
    for (int t = 0; t < nthreads; ++t) me = std::max(me, te[t]), md = std::max(md, td[t]);
    if (enc_seconds) *enc_seconds = me;
    if (dec_seconds) *dec_seconds = md;
    return std::chrono::duration<double>(T1 - T0).count();
}

} // extern "C"
