// include/jpezy/jpezy_writer.hpp -- host side of the encoder: JPEG header / trailer bytes and the output file.
// Mirrors jpezy::jpezy_writer (src/encoder/jpezy_writer.hpp:14-116): same constructor, write_header(), write_eoi(),
// output_file(); get_stream() hands out the byte buffer the entropy-coded segment is appended to (the reference hands out
// its bofstream; here the bit-level writing happens on the device, so the stream is the byte vector itself).
#ifndef JPEZY_B200_JPEZY_WRITER_HPP
#define JPEZY_B200_JPEZY_WRITER_HPP

#include <cstdio>
#include <initializer_list>
#include <stdexcept>
#include <string>
#include <vector>

#include "../jpezy_b200.h"
#include "jpezy.hpp"

namespace jpezy {

namespace tables {
// src/jpezy.hpp:36-45
inline constexpr int ZZ[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                               41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                               30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
// src/jpezy.hpp:131-152 (ITU-T T.81 tables K.1, K.2, natural order)
inline constexpr int YQuantumTb[64] = {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
                                       14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
                                       18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
                                       49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
inline constexpr int CQuantumTb[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99,
                                       99, 99, 47, 66, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                                       99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};
// DHT payloads: BITS (16) + HUFFVAL, ITU-T T.81 tables K.3-K.6 (src/encoder/huffman_table.hpp:205-282 carries them as
// complete marker segments)
struct dht_spec {
    unsigned char tc_th;
    unsigned char bits[16];
    int nvals;
    const unsigned char* vals;
};
inline constexpr unsigned char dc_vals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
inline constexpr unsigned char ac_y_vals[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81,
    0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18,
    0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48,
    0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75,
    0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99,
    0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
    0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5,
    0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
inline constexpr unsigned char ac_c_vals[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08,
    0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25,
    0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47,
    0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74,
    0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97,
    0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
    0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4,
    0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
inline constexpr dht_spec YDcDht{0x00, {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0}, 12, dc_vals};
inline constexpr dht_spec CDcDht{0x01, {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0}, 12, dc_vals};
inline constexpr dht_spec YAcDht{0x10, {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d}, 162, ac_y_vals};
inline constexpr dht_spec CAcDht{0x11, {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}, 162, ac_c_vals};
}  // namespace tables

struct jpezy_writer {
    using stream_type = std::vector<byte>;

    // src/encoder/jpezy_writer.hpp:15-18: buffer of `buffer_size` bytes, file opened (truncated) at construction
    jpezy_writer(const std::size_t buffer_size, const property& pr_, const char* output_name) : cap(buffer_size), pr(pr_)
    {
        fp = output_name ? std::fopen(output_name, "wb") : nullptr;
        buf.reserve(buffer_size < (std::size_t(1) << 26) ? buffer_size : (std::size_t(1) << 26));
    }
    jpezy_writer(const jpezy_writer&) = delete;
    ~jpezy_writer()
    {
        if (fp) std::fclose(fp);
    }

    // src/encoder/jpezy_writer.hpp:20-94, byte for byte (644 bytes for the 16-character comments jpezy uses).  A non-zero
    // restart_interval (MCUs, JPEZYB200_OPT_RESTART_INTERVAL of the encode) adds a DRI segment in front of SOS, where libjpeg
    // writes it.
    void write_header(unsigned restart_interval = 0)
    {
        write_header_with({&tables::YDcDht, &tables::CDcDht, &tables::YAcDht, &tables::CAcDht}, restart_interval);
    }

    // the same header with the four DHT segments carrying the tables of an optimised encode ([0=DC,1=AC][0=luma,1=chroma],
    // jpezyb200_encode_optimized) instead of the Annex K tables: same segments in the same order, lengths from the tables
    void write_header(const jpezyb200_huff (&ht)[2][2], unsigned restart_interval = 0)
    {
        tables::dht_spec d[4];
        const unsigned char tc_th[4] = {0x00, 0x01, 0x10, 0x11};
        for (int k = 0; k < 4; ++k) {
            const jpezyb200_huff& h = ht[tc_th[k] >> 4][tc_th[k] & 1];
            d[k].tc_th = tc_th[k];
            d[k].nvals = 0;
            for (int i = 0; i < 16; ++i) d[k].bits[i] = h.bits[i], d[k].nvals += h.bits[i];
            d[k].vals = h.vals;
        }
        write_header_with({&d[0], &d[1], &d[2], &d[3]}, restart_interval);
    }

    stream_type& get_stream() noexcept { return buf; }
    std::size_t capacity() const noexcept { return cap; }

    // src/encoder/jpezy_writer.hpp:101-105 (the segment handed over by the device is already padded to a byte boundary)
    void write_eoi() { marker(MARKER::EOI); }

    // src/encoder/jpezy_writer.hpp:107-110: one write of the whole buffer
    void output_file()
    {
        if (!fp) throw std::runtime_error(__func__);
        if (!buf.empty() && std::fwrite(buf.data(), 1, buf.size(), fp) != buf.size()) throw std::runtime_error(__func__);
        std::fflush(fp);
    }
    std::size_t wrote_size() const noexcept { return buf.size(); }
    explicit operator bool() const noexcept { return fp != nullptr; }

private:
    void write_header_with(std::initializer_list<const tables::dht_spec*> dhts, unsigned restart_interval)
    {
        if (!fp) throw std::runtime_error(__func__);
        if (restart_interval > 65535u) throw std::runtime_error("jpezy_writer: restart interval above 65535 MCUs");
        marker(MARKER::SOI);
        marker(MARKER::APP0), word(16), bytes("JFIF", 5), word(0x0102), put(static_cast<int>(pr.get<property::At::Units>()));
        word(pr.get<property::At::HDensity>()), word(pr.get<property::At::VDensity>());
        put(pr.get<property::At::HThumbnail>()), put(pr.get<property::At::VThumbnail>());
        if (const std::string& c = pr.get<property::At::Comment>(); !c.empty()) {
            marker(MARKER::COM), word(static_cast<unsigned>(c.size() + 3)), bytes(c.c_str(), c.size() + 1);
        }
        marker(MARKER::DQT), word(67), put(0);
        for (int i = 0; i < 64; ++i) put(tables::YQuantumTb[tables::ZZ[i]]);
        marker(MARKER::DQT), word(67), put(1);
        for (int i = 0; i < 64; ++i) put(tables::CQuantumTb[tables::ZZ[i]]);
        for (const tables::dht_spec* d : dhts) {
            marker(MARKER::DHT), word(2 + 1 + 16 + d->nvals), put(d->tc_th);
            for (unsigned char b : d->bits) put(b);
            for (int i = 0; i < d->nvals; ++i) put(d->vals[i]);
        }
        const int dim = pr.get<property::At::Dimension>();
        marker(MARKER::SOF0), word(3 * dim + 8), put(pr.get<property::At::SamplePrecision>());
        word(static_cast<unsigned>(pr.get<property::At::VSize>())), word(static_cast<unsigned>(pr.get<property::At::HSize>())), put(dim);
        put(0), put(0x22), put(0);
        for (int i = 1; i < 3; ++i) put(i), put(0x11), put(1);
        if (restart_interval) marker(MARKER::DRI), word(4), word(restart_interval);   // T.81 B.2.4.4
        marker(MARKER::SOS), word(2 * dim + 6), put(dim);
        for (int i = 0; i < dim; ++i) put(i), put(i == 0 ? 0 : 0x11);
        put(0), put(63), put(0);
    }

    void put(int v)
    {
        if (buf.size() >= cap) throw std::runtime_error("jpezy_writer: buffer overflow");
        buf.push_back(static_cast<byte>(v));
    }
    void word(unsigned v) { put(int(v >> 8) & 0xff), put(int(v) & 0xff); }
    void marker(MARKER m) { put(0xff), put(static_cast<int>(m)); }
    void bytes(const char* p, std::size_t n)
    {
        for (std::size_t i = 0; i < n; ++i) put(static_cast<unsigned char>(p[i]));
    }

    std::size_t cap;
    const property& pr;
    std::FILE* fp = nullptr;
    stream_type buf;
};

}  // namespace jpezy
#endif
