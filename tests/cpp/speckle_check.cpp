// C++ consumer of include/BICOS/speckles.hpp, built with plain g++ like api_check.cpp and driven by
// tests/test_speckles.py: BICOS::filter_speckles on an uploaded disparity, once with counts and once without.
//
//   speckle_check <in.bin> <out.bin>
//
// in.bin: int32 rows, cols, type (3 = CV_16SC1, 5 = CV_32FC1), max_speckle_size; float64 new_value, max_diff; the
// disparity, dense. out.bin: uint64 pixels set, speckles removed; the filtered disparity, dense. Exit code 1 when
// the two calls disagree or a wrong image type is accepted.
#include <BICOS/speckles.hpp>

#include <cstdio>
#include <cstring>
#include <vector>

using namespace BICOS;

static std::vector<char> slurp(const char* path) {
    std::vector<char> buf;
    FILE* f = std::fopen(path, "rb");
    if (!f)
        return buf;
    std::fseek(f, 0, SEEK_END);
    buf.resize((size_t)std::ftell(f));
    std::fseek(f, 0, SEEK_SET);
    if (std::fread(buf.data(), 1, buf.size(), f) != buf.size())
        buf.clear();
    std::fclose(f);
    return buf;
}

int main(int argc, char** argv) {
    if (argc < 3) {
        std::fprintf(stderr, "usage: speckle_check <in.bin> <out.bin>\n");
        return 2;
    }
    std::vector<char> in = slurp(argv[1]);
    if (in.size() < 32) {
        std::fprintf(stderr, "cannot read the input\n");
        return 2;
    }
    int32_t hdr[4];
    double prm[2];
    std::memcpy(hdr, in.data(), sizeof hdr);
    std::memcpy(prm, in.data() + sizeof hdr, sizeof prm);
    const int rows = hdr[0], cols = hdr[1], type = hdr[2], max_size = hdr[3];
    char* disp = in.data() + sizeof hdr + sizeof prm;
    const size_t bytes = (size_t)rows * cols * (type == IMG_16S ? 2 : 4);
    if (in.size() < sizeof hdr + sizeof prm + bytes) {
        std::fprintf(stderr, "short input\n");
        return 2;
    }

    try {
        Image a(HostImage(rows, cols, type, disp)), b(HostImage(rows, cols, type, disp));
        SpeckleCounts n {};
        filter_speckles(a, prm[0], max_size, prm[1], &n);
        filter_speckles(b, prm[0], max_size, prm[1]); // enqueued only; download() below synchronises
        std::vector<char> got_a(bytes), got_b(bytes);
        a.download(HostImage(rows, cols, type, got_a.data()));
        b.download(HostImage(rows, cols, type, got_b.data()));
        if (got_a != got_b) {
            std::fprintf(stderr, "the calls with and without counts disagree\n");
            return 1;
        }
        Image wrong(rows, cols, IMG_64F);
        try {
            filter_speckles(wrong, 0.0, max_size, prm[1]);
            std::fprintf(stderr, "a CV_64FC1 disparity was accepted\n");
            return 1;
        } catch (const Exception&) {
        }
        FILE* o = std::fopen(argv[2], "wb");
        if (!o)
            return 2;
        const unsigned long long counts[2] = { n.pixels, n.speckles };
        std::fwrite(counts, sizeof counts, 1, o);
        std::fwrite(got_a.data(), 1, bytes, o);
        std::fclose(o);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "exception: %s\n", e.what());
        return 1;
    }
    return 0;
}
