// include/jpezy/jpezy_encoder.hpp -- drop-in for jpezy::encoder<T> (src/encoder/jpezy_encoder.hpp:22-39,84,277-278).
// Same constructor, same encode<MODE_TAG>(output_file) -> bytes written, same console lines.  The MCU loop
// (src/encoder/jpezy_encoder.hpp:55-67: make_YCC, DCT, quantization, encode_huffman) runs on the B200 behind
// jpezyb200_encode; header, EOI and the file stay here.
#ifndef JPEZY_B200_JPEZY_ENCODER_HPP
#define JPEZY_B200_JPEZY_ENCODER_HPP

#include <stdexcept>
#include <type_traits>
#include <vector>

#include "jpezy.hpp"
#include "jpezy_writer.hpp"
#include "runtime.hpp"

namespace jpezy {

// encode<MODE>(file, optimize_huffman): Huffman tables fitted to the image instead of the Annex K tables
struct optimize_huffman_t {};
inline constexpr optimize_huffman_t optimize_huffman{};

// encode<MODE>(file[, optimize_huffman], restart_interval{n}): restart markers every n MCUs and a DRI segment (0 = none)
struct restart_interval {
    unsigned mcus = 0;
};

namespace b200 {
// JPEZYB200_OPT_RESTART_INTERVAL of the shared context for the lifetime of one encode, back to 0 afterwards
struct restart_scope {
    explicit restart_scope(unsigned mcus)
    {
        if (mcus > 65535u) throw std::runtime_error("encode: restart interval above 65535 MCUs");
        const int rc = jpezyb200_set_option(runtime::ctx(), JPEZYB200_OPT_RESTART_INTERVAL, mcus);
        if (rc != JPEZYB200_OK) throw runtime::error("encode", rc);
    }
    ~restart_scope() { jpezyb200_set_option(runtime::ctx(), JPEZYB200_OPT_RESTART_INTERVAL, 0); }
    restart_scope(const restart_scope&) = delete;
    restart_scope& operator=(const restart_scope&) = delete;
};
}  // namespace b200

template <class T>
struct encoder {
    static_assert(sizeof(T) == 1, "8-bit samples");
    // copies the three planes, keeps a reference to the property (src/encoder/jpezy_encoder.hpp:24-36,265-266)
    encoder(const property& pr_, const std::vector<T>& r_, const std::vector<T>& g_, const std::vector<T>& b_) : pr(pr_), r(r_), g(g_), b(b_) {}

    template <class MODE_TAG = COLOR_MODE>
    std::size_t encode(const char* output_file, restart_interval rst = {})
    {
        const std::size_t W = pr.get<property::At::HSize>(), H = pr.get<property::At::VSize>();
        // src/encoder/jpezy_encoder.hpp:41-43 computes this in `int` (overflows above 715 Mpixel); size_t here (decision O5)
        std::size_t size = W * H * 3;
        if (size < 10240) size = 10240;
        jpezy_writer jpeg(size, pr, output_file);
        {
            raii_messenger mes("Write JPEG Header ...");
            jpeg.write_header(rst.mcus);
        }
        {
            raii_messenger mes("Encoding ...");
            if (r.size() < W * H || g.size() < W * H || b.size() < W * H) throw std::runtime_error("encode: planes smaller than width*height");
            jpezy_writer::stream_type& s = jpeg.get_stream();
            const std::size_t head = s.size();
            const std::size_t room = jpeg.capacity() > head + 2 ? jpeg.capacity() - head - 2 : 0;
            s.resize(head + room);
            std::size_t nbytes = 0;
            const b200::restart_scope scope(rst.mcus);
            const int rc = jpezyb200_encode(b200::runtime::ctx(), reinterpret_cast<const std::uint8_t*>(r.data()),
                                            reinterpret_cast<const std::uint8_t*>(g.data()), reinterpret_cast<const std::uint8_t*>(b.data()),
                                            static_cast<std::uint32_t>(W), static_cast<std::uint32_t>(H), std::is_same_v<MODE_TAG, GRAY_MODE> ? 1 : 0,
                                            s.data() + head, room, &nbytes, nullptr);
            if (rc != JPEZYB200_OK) {
                s.resize(head);
                throw b200::runtime::error("encode", rc);   // std::runtime_error, as the reference's encode_huffman / bofstream throw
            }
            s.resize(head + nbytes);
        }
        {
            raii_messenger mes("Write EOI ...");
            jpeg.write_eoi();
        }
        jpeg.output_file();
        return jpeg.wrote_size();
    }

    // The same file with optimised Huffman tables (jpezyb200_encode_optimized): the tables exist only after the encode, so the
    // segment is encoded first, then the header with the tables' DHT segments, the segment and EOI are written.
    template <class MODE_TAG = COLOR_MODE>
    std::size_t encode(const char* output_file, optimize_huffman_t, restart_interval rst = {})
    {
        const std::size_t W = pr.get<property::At::HSize>(), H = pr.get<property::At::VSize>();
        std::size_t size = W * H * 3;
        if (size < 10240) size = 10240;
        jpezy_writer jpeg(size, pr, output_file);
        if (!jpeg) throw std::runtime_error(__func__);
        std::vector<byte> scan(size);
        std::size_t nbytes = 0;
        jpezyb200_huff ht[2][2];
        {
            raii_messenger mes("Encoding ...");
            if (r.size() < W * H || g.size() < W * H || b.size() < W * H) throw std::runtime_error("encode: planes smaller than width*height");
            const b200::restart_scope scope(rst.mcus);
            const int rc = jpezyb200_encode_optimized(b200::runtime::ctx(), reinterpret_cast<const std::uint8_t*>(r.data()),
                                                      reinterpret_cast<const std::uint8_t*>(g.data()), reinterpret_cast<const std::uint8_t*>(b.data()),
                                                      static_cast<std::uint32_t>(W), static_cast<std::uint32_t>(H),
                                                      std::is_same_v<MODE_TAG, GRAY_MODE> ? 1 : 0, scan.data(), scan.size(), &nbytes, nullptr, ht);
            if (rc != JPEZYB200_OK) throw b200::runtime::error("encode", rc);
        }
        {
            raii_messenger mes("Write JPEG Header ...");
            jpeg.write_header(ht, rst.mcus);
        }
        jpezy_writer::stream_type& s = jpeg.get_stream();
        if (s.size() + nbytes + 2 > jpeg.capacity()) throw std::runtime_error("jpezy_writer: buffer overflow");
        s.insert(s.end(), scan.begin(), scan.begin() + std::ptrdiff_t(nbytes));
        {
            raii_messenger mes("Write EOI ...");
            jpeg.write_eoi();
        }
        jpeg.output_file();
        return jpeg.wrote_size();
    }

    static constexpr int block_size = 8;

private:
    const property& pr;
    const std::vector<T> r, g, b;
};

template <class T>
encoder(const property&, const std::vector<T>&, const std::vector<T>&, const std::vector<T>&) -> encoder<T>;

}  // namespace jpezy
#endif
