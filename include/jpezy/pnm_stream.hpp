// include/jpezy/pnm_stream.hpp -- base of the two PNM adaptors (src/pnm_stream.hpp:11-43)
#ifndef JPEZY_B200_PNM_STREAM_HPP
#define JPEZY_B200_PNM_STREAM_HPP

#include <algorithm>
#include <array>
#include <cstddef>
#include <exception>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "jpezy.hpp"

namespace jpezy {

// Host-side helper of the two PNM adaptors: run f(part, begin, end) for `parts` contiguous ranges of [0, n) on up to
// `parts` threads.  The first exception in range order is re-thrown on the calling thread once all parts have finished,
// which is the exception a sequential pass over [0, n) would have raised.
namespace pnm_detail {
inline unsigned host_threads(std::size_t work_bytes)
{
    if (work_bytes < (std::size_t(1) << 20)) return 1;
    const unsigned hc = std::thread::hardware_concurrency();
    return std::max(1u, std::min(hc ? hc : 1u, 16u));
}
template <class F>
void parallel_parts(unsigned parts, F&& f)
{
    if (parts <= 1) {
        f(0u);
        return;
    }
    std::vector<std::exception_ptr> err(parts);
    std::vector<std::thread> th;
    th.reserve(parts - 1);
    const auto run = [&](unsigned k) {
        try {
            f(k);
        } catch (...) {
            err[k] = std::current_exception();
        }
    };
    for (unsigned k = 1; k < parts; ++k) th.emplace_back(run, k);
    run(0);
    for (auto& t : th) t.join();
    for (unsigned k = 0; k < parts; ++k)
        if (err[k]) std::rethrow_exception(err[k]);
}
// the bytes of a file, mapped read-only (no copy, no zero-filled buffer; the pages are touched by whoever parses them)
struct file_view {
    const char* data = nullptr;
    std::size_t size = 0;
    bool ok = false;
    explicit file_view(const char* name)
    {
        const int fd = ::open(name, O_RDONLY);
        if (fd < 0) return;
        struct stat st;
        if (::fstat(fd, &st) == 0 && S_ISREG(st.st_mode)) {
            ok = true;
            size = std::size_t(st.st_size);
            if (size) {
                void* m = ::mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
                if (m == MAP_FAILED) ok = false, size = 0;
                else data = static_cast<const char*>(m);
            }
        } else if (::fstat(fd, &st) == 0) {       // a pipe or device: read it
            ok = true;
            char tmp[65536];
            for (ssize_t n; (n = ::read(fd, tmp, sizeof tmp)) > 0;) owned_.append(tmp, std::size_t(n));
            data = owned_.data(), size = owned_.size();
        }
        ::close(fd);
    }
    ~file_view()
    {
        if (data && owned_.empty() && size) ::munmap(const_cast<char*>(data), size);
    }
    file_view(const file_view&) = delete;
    file_view& operator=(const file_view&) = delete;

private:
    std::string owned_;
};
// "r g b\n" for samples [i0, i1) of three planes, appended to out
template <class R>
void format_triples(const R& r, const R& g, const R& b, std::size_t i0, std::size_t i1, std::string& out)
{
    std::string loc;      // (local: the string headers of neighbouring parts share cache lines)
    loc.resize((i1 - i0) * 12);
    char* w = &loc[0];
    const auto put = [&w](unsigned v, char sep) {
        if (v >= 100) *w++ = char('0' + v / 100 % 10);
        if (v >= 10) *w++ = char('0' + v / 10 % 10);
        *w++ = char('0' + v % 10);
        *w++ = sep;
    };
    for (std::size_t i = i0; i < i1; ++i) put(unsigned(r[i]) & 255u, ' '), put(unsigned(g[i]) & 255u, ' '), put(unsigned(b[i]) & 255u, '\n');
    loc.resize(std::size_t(w - loc.data()));
    if (out.empty()) out = std::move(loc);
    else out += loc;
}
}  // namespace pnm_detail

struct pnm_stream {
    pnm_stream() : initializing_succeed(true), width(0), height(0), max_color(0) {}
    pnm_stream(bool b, std::size_t w, std::size_t h, std::size_t max) : initializing_succeed(b), width(w), height(h), max_color(max) {}
    explicit operator bool() const noexcept { return initializing_succeed; }
    std::size_t get_width() const noexcept { return width; }

protected:
    typedef byte value_type;
    typedef byte rgb_type;
    bool initializing_succeed;
    std::size_t width, height, max_color;
    std::vector<std::array<rgb_type, 3>> rgb_img;

    void report_error(const char* funcName) const
    {
        if (initializing_succeed) return;
        throw std::runtime_error(std::string("Initializing was failed: ") + funcName);
    }
};

}  // namespace jpezy
#endif
