// jpezy_encode -- drop-in for the reference's encoder CLI (src/encoder/main.cpp:56-116):
//   jpezy_encode <input.ppm> ( <output.(jpeg | jpg)> [--optimize] [--gray] [--restart N[B]] | <output.ppm> | --debug )
// Same argv sniffing (substring search after the first '.'), same console lines, same exit codes; the MCU loop runs on the
// B200 through libjpezy_b200.so.  Unlike the reference, argv[3] is only looked at when it exists (:67-69 reads argv[argc]).
// --optimize (not in the reference) writes Huffman tables fitted to the image instead of the Annex K tables.
// --restart N (not in the reference) writes restart markers every N MCU rows, --restart NB every N MCUs, as cjpeg's -restart
// does; 0 = none.  It may stand anywhere after the output name; the other arguments are read as if it were not there.
#include <cstdint>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <optional>
#include <stdexcept>
#include <string_view>
#include <vector>

#include "jpezy/encode_io.hpp"

namespace {

int disp_error()
{
    std::cerr << "Usage: jpezy_encode <input.ppm> ( <ouput.(jpeg | jpg) [OPT: --optimize] [OPT: --gray] [OPT: --restart N[B]]> | <output.ppm> | --debug )"
              << std::endl;
    return EXIT_FAILURE;
}

enum class Mode { JPEG, GRAY, PPM, DEBUG, UD };

// --restart's value: N MCU rows or NB MCUs (decimal, at most 65535 either way)
struct restart_arg {
    unsigned long value = 0;
    bool in_mcus = false;
};

bool parse_restart(std::string_view s, restart_arg& out)
{
    if (!s.empty() && (s.back() == 'B' || s.back() == 'b')) out.in_mcus = true, s.remove_suffix(1);
    if (s.empty() || s.size() > 5) return false;
    out.value = 0;
    for (char c : s) {
        if (c < '0' || c > '9') return false;
        out.value = out.value * 10 + unsigned(c - '0');
    }
    return out.value <= 65535;
}

void exec(const jpezy::encode_io& pnm, const char* ofile, Mode m1, Mode m2, bool optimize, unsigned restart)
{
    const jpezy::restart_interval rst{restart};
    const jpezy::to_jpeg jpeg = optimize ? jpezy::to_jpeg(ofile, jpezy::optimize_huffman, rst) : jpezy::to_jpeg(ofile, rst);
    if (m2 == Mode::GRAY) {
        if (m1 != Mode::JPEG) throw std::invalid_argument("2nd Mode parameter must be GRAY");
        std::ofstream ofs(ofile, std::ios::binary);
        ofs << (pnm | jpeg | jpezy::gray_scale);
        return;
    }
    switch (m1) {
    case Mode::JPEG: {
        std::ofstream ofs(ofile, std::ios::binary);
        ofs << (pnm | jpeg);
        break;
    }
    case Mode::PPM: {
        std::ofstream ofs(ofile);
        ofs << pnm;
        break;
    }
    case Mode::DEBUG: std::cout << pnm << std::endl; break;
    default: throw std::runtime_error("Maybe broken memory");
    }
}

}  // namespace

int main(int argc, const char* argv[])
{
    // take --restart <value> out of the arguments; the rest is read exactly as without it
    std::vector<const char*> args(argv, argv + argc);
    std::optional<restart_arg> restart;
    for (std::size_t i = 3; i < args.size(); ++i) {
        if (std::string_view(args[i]) != "--restart") continue;
        restart_arg ra;
        if (restart || i + 1 >= args.size() || !parse_restart(args[i + 1], ra)) return disp_error();
        restart = ra;
        args.erase(args.begin() + std::ptrdiff_t(i), args.begin() + std::ptrdiff_t(i) + 2);
        --i;
    }
    argc = int(args.size());
    args.push_back(nullptr);
    argv = args.data();
    if (argc < 3) return disp_error();
    Mode m1 = Mode::UD, m2 = Mode::UD;
    bool optimize = false;
    const std::string_view sv1 = argv[2];
    std::optional<std::string_view> sv2;
    if (argc > 3) sv2 = argv[3];

    if (sv1.find("jpeg", sv1.find_first_of('.')) != std::string_view::npos || sv1.find("jpg", sv1.find_first_of('.')) != std::string_view::npos) {
        m1 = Mode::JPEG;
        if (sv2 && *sv2 == "--optimize") {   // --optimize [--gray]
            optimize = true;
            sv2.reset();
            if (argc > 4) sv2 = argv[4];
        } else if (argc > 4 && std::string_view(argv[4]) == "--optimize") {   // --gray --optimize
            optimize = true;
        }
        if (sv2 && sv2->find("--gray") != std::string_view::npos) m2 = Mode::GRAY;
    } else if (sv1.find("ppm", sv1.find_first_of('.')) != std::string_view::npos) {
        m1 = Mode::PPM;
    } else if (!sv1.compare("--debug")) {
        m1 = Mode::DEBUG;
    } else {
        return disp_error();
    }

    jpezy::disp_logo();
    jpezy::raii_messenger section("Reading the input file...");
    jpezy::encode_io pnm(argv[1]);
    if (!pnm) {
        std::cerr << "The file is not found or the formatting error" << std::endl;
        return disp_error();
    }
    // the interval in MCUs: N rows are N * ceil(width / 16) MCUs
    unsigned rst_mcus = 0;
    if (restart) {
        const std::uint64_t mcus = restart->in_mcus ? restart->value : restart->value * ((std::uint64_t(pnm.get_width()) + 15) / 16);
        if (mcus > 65535) return disp_error();
        rst_mcus = unsigned(mcus);
    }
    auto t1 = section.stop();
    section.restart("Start encoding and writing ...");
    try {
        exec(pnm, argv[2], m1, m2, optimize, rst_mcus);
    } catch (const std::runtime_error& e) {
        std::cerr << e.what() << std::endl;
        return EXIT_FAILURE;
    }
    auto t2 = section.stop();
    if (t1 && t2) std::cout << "Total processing time: " << t1.value() + t2.value() << std::endl;
    else throw std::runtime_error("Timer error");
}
