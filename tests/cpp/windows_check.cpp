// C++ consumer of include/BICOS/windows.hpp, built with plain g++ like api_check.cpp and driven by
// tests/test_windows.py: a full-row BICOS::match gives the prior, BICOS::windows_from_disparity turns it into windows
// (prior +- margin, the whole row where the prior is invalid) and BICOS::match_windows matches again inside them.
//
//   windows_check <in.bin> <out.bin> <margin>
//
// in.bin / out.bin: as for api_check (out.bin holds the windowed match). Before matching, checks that windows together
// with Config::disparity_range throw BICOS::Exception.
#include <BICOS/windows.hpp>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

using namespace BICOS;

int main(int argc, char** argv) {
    if (argc < 4) {
        std::fprintf(stderr, "usage: windows_check <in.bin> <out.bin> <margin>\n");
        return 2;
    }
    FILE* f = std::fopen(argv[1], "rb");
    if (!f) {
        std::perror(argv[1]);
        return 2;
    }
    std::fseek(f, 0, SEEK_END);
    std::vector<char> in((size_t)std::ftell(f));
    std::fseek(f, 0, SEEK_SET);
    if (std::fread(in.data(), 1, in.size(), f) != in.size())
        return 2;
    std::fclose(f);
    int32_t hdr[9];
    float opt[3];
    std::memcpy(hdr, in.data(), sizeof hdr);
    std::memcpy(opt, in.data() + sizeof hdr, sizeof opt);
    const int n = hdr[0], rows = hdr[1], cols = hdr[2], depth = hdr[3];
    const size_t plane = (size_t)rows * cols * (depth == IMG_16U ? 2 : 1);
    const char* base = in.data() + sizeof hdr + sizeof opt;

    Config cfg;
    cfg.nxcorr_threshold = opt[0] >= 0 ? std::optional<float>(opt[0]) : std::nullopt;
    cfg.subpixel_step = opt[1] >= 0 ? std::optional<float>(opt[1]) : std::nullopt;
    cfg.min_variance = opt[2] >= 0 ? std::optional<float>(opt[2]) : std::nullopt;
    cfg.mode = (hdr[4] & 1) ? TransformMode::FULL : TransformMode::LIMITED;
    cfg.precision = hdr[5] ? Precision::DOUBLE : Precision::SINGLE;
    if (hdr[6])
        cfg.variant = Variant::Consistency { hdr[7], hdr[8] != 0 };

    try {
        std::vector<Image> s0, s1;
        for (int i = 0; i < n; ++i) {
            s0.emplace_back(HostImage(rows, cols, depth, const_cast<char*>(base) + plane * i));
            s1.emplace_back(HostImage(rows, cols, depth, const_cast<char*>(base) + plane * (n + i)));
        }
        Image prior, disp, corr;
        match(s0, s1, prior, cfg);
        DisparityWindows windows;
        windows_from_disparity(prior, std::atoi(argv[3]), std::nullopt, windows);
        Config ranged = cfg;
        ranged.disparity_range = DisparityRange { 0, 10 };
        try {
            match_windows(s0, s1, windows, disp, ranged);
            std::fprintf(stderr, "windows with a disparity range were accepted\n");
            return 1;
        } catch (const Exception&) {
        }
        match_windows(s0, s1, windows, disp, cfg, &corr);
        std::vector<char> dbuf((size_t)rows * cols * disp.elemSize());
        disp.download(HostImage(rows, cols, disp.type(), dbuf.data()));
        std::vector<char> cbuf;
        if (!corr.empty()) {
            cbuf.resize((size_t)rows * cols * corr.elemSize());
            corr.download(HostImage(rows, cols, corr.type(), cbuf.data()));
        }
        FILE* o = std::fopen(argv[2], "wb");
        if (!o)
            return 2;
        const int32_t oh[4] = { disp.type(), corr.empty() ? 0 : corr.type(), rows, cols };
        std::fwrite(oh, sizeof oh, 1, o);
        std::fwrite(dbuf.data(), 1, dbuf.size(), o);
        std::fwrite(cbuf.data(), 1, cbuf.size(), o);
        std::fclose(o);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "exception: %s\n", e.what());
        return 1;
    }
    return 0;
}
