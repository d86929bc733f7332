// jpezy_encode -- drop-in for the reference's encoder CLI (src/encoder/main.cpp:56-116):
//   jpezy_encode <input.ppm> ( <output.(jpeg | jpg)> [--optimize] [--gray] | <output.ppm> | --debug )
// Same argv sniffing (substring search after the first '.'), same console lines, same exit codes; the MCU loop runs on the
// B200 through libjpezy_b200.so.  Unlike the reference, argv[3] is only looked at when it exists (:67-69 reads argv[argc]).
// --optimize (not in the reference) writes Huffman tables fitted to the image instead of the Annex K tables.
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <optional>
#include <stdexcept>
#include <string_view>

#include "jpezy/encode_io.hpp"

namespace {

int disp_error()
{
    std::cerr << "Usage: jpezy_encode <input.ppm> ( <ouput.(jpeg | jpg) [OPT: --optimize] [OPT: --gray]> | <output.ppm> | --debug )" << std::endl;
    return EXIT_FAILURE;
}

enum class Mode { JPEG, GRAY, PPM, DEBUG, UD };

void exec(const jpezy::encode_io& pnm, const char* ofile, Mode m1, Mode m2, bool optimize)
{
    const jpezy::to_jpeg jpeg = optimize ? jpezy::to_jpeg(ofile, jpezy::optimize_huffman) : jpezy::to_jpeg(ofile);
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

int main(const int argc, const char* argv[])
{
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
    auto t1 = section.stop();
    section.restart("Start encoding and writing ...");
    try {
        exec(pnm, argv[2], m1, m2, optimize);
    } catch (const std::runtime_error& e) {
        std::cerr << e.what() << std::endl;
        return EXIT_FAILURE;
    }
    auto t2 = section.stop();
    if (t1 && t2) std::cout << "Total processing time: " << t1.value() + t2.value() << std::endl;
    else throw std::runtime_error("Timer error");
}
