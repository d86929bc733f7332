// include/jpezy/encode_io.hpp -- drop-in for jpezy::encode_io, to_jpeg, gray_scale (src/encoder/encode_io.hpp:33-209):
//   jpezy::encode_io pnm("in.ppm");  ofs << (pnm | jpezy::to_jpeg("out.jpg"));  ofs << (pnm | to_jpeg(f) | jpezy::gray_scale);
//   ofs << (pnm | jpezy::to_jpeg(f, jpezy::optimize_huffman)) writes the file with Huffman tables fitted to the image,
//   jpezy::to_jpeg(f, jpezy::restart_interval{n}) (or to_jpeg(f, optimize_huffman, restart_interval{n})) one with restart
//   markers every n MCUs.
// The P3 grammar is the reference's, quirks included (SURVEY.md appendix A.1): lines containing '#' are dropped wherever
// they appear, the size line must split into exactly two tokens, maxval is parsed and ignored, a final line without a
// newline is dropped, an interior empty token makes std::stoi throw std::invalid_argument.  One pass over the file
// instead of std::list<std::string> per token (the reference spends 0.52 of 0.57 s here, README.md:48-56).
#ifndef JPEZY_B200_ENCODE_IO_HPP
#define JPEZY_B200_ENCODE_IO_HPP

#include <algorithm>
#include <cctype>
#include <cstring>
#include <fstream>
#include <iostream>
#include <string>
#include <string_view>
#include <tuple>
#include <utility>
#include <vector>

#include "jpezy.hpp"
#include "jpezy_encoder.hpp"
#include "pnm_stream.hpp"

namespace jpezy {

struct to_jpeg {
    explicit constexpr to_jpeg(const char* file_) : file(file_) {}
    // to_jpeg(f, optimize_huffman): the file carries Huffman tables fitted to the image instead of the Annex K tables
    constexpr to_jpeg(const char* file_, optimize_huffman_t) : file(file_), optimize(true) {}
    // restart markers every rst.mcus MCUs (0 = none), with or without optimised tables
    constexpr to_jpeg(const char* file_, restart_interval rst_) : file(file_), rst(rst_) {}
    constexpr to_jpeg(const char* file_, optimize_huffman_t, restart_interval rst_) : file(file_), optimize(true), rst(rst_) {}
    const char* file;
    bool optimize = false;
    restart_interval rst{};
};
struct gray_scale_t {};
inline constexpr gray_scale_t gray_scale{};

struct encode_io : pnm_stream {
    encode_io(const char* file_name) : pnm_stream(true, 0, 0, 0)
    {
        // the whole file mapped; lines are cut out of it with std::getline's rules
        const pnm_detail::file_view fv(file_name);
        if (!fv.ok) {
            initializing_succeed = false;
            return;
        }
        const struct {
            const char* p;
            std::size_t n;
            const char* data() const { return p; }
            std::size_t size() const { return n; }
        } buf{fv.data ? fv.data : "", fv.size};
        std::size_t pos = 0;
        bool eof = false;
        // std::getline: a line ends at '\n'; reaching the end of the data while reading sets eof (and the text read so far
        // is still a line); a call that extracts nothing fails and leaves an empty string
        const auto getline = [&](std::string_view& out) {
            if (pos >= buf.size()) {
                eof = true;
                out = std::string_view();
                return false;
            }
            const void* nl = std::memchr(buf.data() + pos, '\n', buf.size() - pos);
            if (nl) {
                const std::size_t e = std::size_t(static_cast<const char*>(nl) - buf.data());
                out = std::string_view(buf.data() + pos, e - pos);
                pos = e + 1;
            } else {
                out = std::string_view(buf.data() + pos, buf.size() - pos);
                pos = buf.size();
                eof = true;
            }
            return true;
        };
        // src/encoder/encode_io.hpp:50-56: read lines until one without '#' (or until getline fails; the last string read is returned)
        const auto jump_comment = [&]() {
            std::string_view str;
            while (getline(str) && str.find('#') != std::string_view::npos) {}
            return str;
        };
        const auto is_space = [](char c) { return std::isspace(static_cast<unsigned char>(c)) != 0; };
        // std::stoi on one token; all-digit tokens (every token of a well-formed file) take a short cut
        const auto to_int = [](std::string_view tok) -> int {
            if (!tok.empty() && tok.size() <= 9) {
                int v = 0;
                std::size_t i = 0;
                for (; i < tok.size() && tok[i] >= '0' && tok[i] <= '9'; ++i) v = v * 10 + (tok[i] - '0');
                if (i == tok.size()) return v;
            }
            return std::stoi(std::string(tok));       // "" -> std::invalid_argument, "12x" -> 12, as in the reference
        };
        // boost::split(is_space()) with token_compress_off: every separator ends a token
        const auto for_each_token = [&](std::string_view line, auto&& f) {
            std::size_t i = 0;
            for (;;) {
                std::size_t j = i;
                while (j < line.size() && !is_space(line[j])) ++j;
                const bool last = j >= line.size();
                f(line.substr(i, j - i), last);
                if (last) break;
                i = j + 1;
            }
        };
        std::string_view format = jump_comment();
        if (format != "P3") {
            initializing_succeed = false;
            return;
        }
        format = jump_comment();
        std::vector<std::string_view> wh;
        for_each_token(format, [&](std::string_view t, bool) { wh.push_back(t); });
        if (wh.size() != 2) {
            initializing_succeed = false;
        } else {
            width = std::size_t(to_int(wh[0])), height = std::size_t(to_int(wh[1]));
            format = jump_comment();
            max_color = std::size_t(std::stoi(std::string(format)));      // whole line through stoi (leading blanks allowed)
            // The pixel lines.  Only lines that end in '\n' are data (the reference's loop tests eof after reading a line,
            // :80), lines containing '#' are dropped whole.  The body is cut at line starts into one range per host
            // thread; a token std::stoi rejects throws exactly as in a sequential pass (first one in file order).
            const char* const body = buf.data() + pos;
            const std::size_t blen = buf.size() - pos;
            const unsigned parts = pnm_detail::host_threads(blen);
            std::vector<std::size_t> cut(parts + 1, blen);
            cut[0] = 0;
            for (unsigned k = 1; k < parts; ++k) {
                const std::size_t from = std::max(cut[k - 1], blen * k / parts);
                const void* nl = from < blen ? std::memchr(body + from, '\n', blen - from) : nullptr;
                cut[k] = nl ? std::size_t(static_cast<const char*>(nl) - body) + 1 : blen;
            }
            std::vector<std::vector<value_type>> part(parts);
            pnm_detail::parallel_parts(parts, [&](unsigned k) {
                std::vector<value_type> img;      // (local: the vector headers in `part` share cache lines)
                img.reserve((cut[k + 1] - cut[k]) / 2);
                const char* p = body + cut[k];
                const char* const e = body + cut[k + 1];
                while (p < e) {
                    const void* nl = std::memchr(p, '\n', std::size_t(e - p));
                    if (!nl) break;                                  // unterminated last line of the file: dropped
                    const std::string_view line(p, std::size_t(static_cast<const char*>(nl) - p));
                    p = static_cast<const char*>(nl) + 1;
                    if (line.find('#') != std::string_view::npos) continue;
                    // exactly one trailing empty token is forgiven (:83-84), every other one reaches stoi
                    for_each_token(line, [&](std::string_view t, bool last) {
                        if (!(last && t.empty())) img.push_back(value_type(to_int(t)));
                    });
                }
                part[k] = std::move(img);
            });
            std::size_t total = 0;
            for (const auto& v : part) total += v.size();
            rgb_img.resize(total / 3);
            // std::array<byte, 3> is three contiguous bytes: the parts are laid end to end, the incomplete last triple is cut
            {
                unsigned char* dst = reinterpret_cast<unsigned char*>(rgb_img.data());
                std::size_t room = rgb_img.size() * 3;
                for (const auto& v : part) {
                    const std::size_t n = std::min(room, v.size());
                    if (n) std::memcpy(dst, v.data(), n);
                    dst += n, room -= n;
                }
            }
        }
        std::cout << "width: " << width << " height: " << height << std::endl;
    }

private:
    // P3 echo (:104-119)
    friend std::ostream& operator<<(std::ostream& os, const encode_io& pnm)
    {
        pnm.report_error(__func__);
        const std::string head = "P3\n" + std::to_string(pnm.width) + " " + std::to_string(pnm.height) + "\n" + std::to_string(pnm.max_color) + "\n";
        os.write(head.data(), std::streamsize(head.size()));
        const std::size_t n = pnm.rgb_img.size();
        const unsigned parts = pnm_detail::host_threads(n * 12);
        std::vector<std::string> chunk(parts);
        struct plane {      // view of one channel of the interleaved image
            const std::array<rgb_type, 3>* px;
            int c;
            unsigned operator[](std::size_t i) const { return unsigned(px[i][c]); }
        };
        const plane r{pnm.rgb_img.data(), 0}, g{pnm.rgb_img.data(), 1}, b{pnm.rgb_img.data(), 2};
        pnm_detail::parallel_parts(parts, [&](unsigned k) { pnm_detail::format_triples(r, g, b, n * k / parts, n * (k + 1) / parts, chunk[k]); });
        for (const std::string& c : chunk) os.write(c.data(), std::streamsize(c.size()));
        return os;
    }

    // :121-133
    std::tuple<std::vector<rgb_type>, std::vector<rgb_type>, std::vector<rgb_type>> split_rgb() const
    {
        std::vector<rgb_type> r(rgb_img.size()), g(rgb_img.size()), b(rgb_img.size());
        for (std::size_t i = 0; i < rgb_img.size(); ++i) r[i] = rgb_img[i][0], g[i] = rgb_img[i][1], b[i] = rgb_img[i][2];
        return {std::move(r), std::move(g), std::move(b)};
    }

    // :135-169
    friend std::ofstream& operator<<(std::ofstream& ofs, const std::pair<const to_jpeg, const encode_io&>& pnm)
    {
        ofs.close();
        pnm.second.report_error(__func__);
        const property pr = make_property({.width = pnm.second.width, .height = pnm.second.height, .dimension = 3, .sample_precision = 8,
                                           .comment = "Encoded by jpezy", .format = property::Format::JFIF, .major_rev = 1, .minor_rev = 2,
                                           .units = property::Units::dots_inch, .width_density = 96, .height_density = 96,
                                           .width_thumbnail = 0, .height_thumbnail = 0,
                                           .extension_code = property::ExtensionCodes::undefined, .decodable = property::Yet});
        auto [r, g, b] = pnm.second.split_rgb();
        encoder enc(pr, r, g, b);
        const std::size_t size = pnm.first.optimize ? enc.encode<COLOR_MODE>(pnm.first.file, optimize_huffman, pnm.first.rst)
                                                    : enc.encode<COLOR_MODE>(pnm.first.file, pnm.first.rst);
        std::cout << "Output size: " << size << " byte" << std::endl;
        return ofs;
    }
    // :171-196
    friend std::ofstream& operator<<(std::ofstream& ofs, const std::pair<gray_scale_t, std::pair<const to_jpeg, const encode_io&>>& pnm)
    {
        ofs.close();
        pnm.second.second.report_error(__func__);
        const property pr{pnm.second.second.width, pnm.second.second.height, 3, 8, "Encoded by JPEZY", property::Format::JFIF, byte(1), byte(2),
                          property::Units::dots_inch, 96, 96, 0, 0, property::ExtensionCodes::undefined};
        auto [r, g, b] = pnm.second.second.split_rgb();
        encoder enc(pr, r, g, b);
        const std::size_t size = pnm.second.first.optimize ? enc.encode<GRAY_MODE>(pnm.second.first.file, optimize_huffman, pnm.second.first.rst)
                                                            : enc.encode<GRAY_MODE>(pnm.second.first.file, pnm.second.first.rst);
        std::cout << "Output size: " << size << " srook::byte" << std::endl;   // sic (:193)
        return ofs;
    }
    friend std::pair<gray_scale_t, std::pair<const to_jpeg, const encode_io&>> operator|(const std::pair<const to_jpeg, const encode_io&>& pnm, const gray_scale_t& gr)
    {
        return {gr, pnm};
    }
    friend std::pair<const to_jpeg, const encode_io&> operator|(const encode_io& pnm, const to_jpeg& jpeg_tag) noexcept
    {
        return {jpeg_tag, pnm};
    }
};

}  // namespace jpezy
#endif
