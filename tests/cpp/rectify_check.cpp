// C++ consumer of include/BICOS/rectify.hpp, built with plain g++ like api_check.cpp and driven by
// tests/test_rectify.py: BICOS::match_rectified on raw stacks, and BICOS::remap of stack0 through camera 0's maps.
//
//   rectify_check <in.bin> <maps.bin> <out.bin>
//
// in.bin: api_check's input format (the raw stacks, of the source size). maps.bin: int32 rows, cols, then the four
// float32 maps map_x0, map_y0, map_x1, map_y1 of rows x cols, dense. out.bin: api_check's output format (the match),
// followed by the n remapped planes of stack0, dense. Before matching, checks that maps of the wrong type throw.
#include <BICOS/rectify.hpp>

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
    if (argc < 4) {
        std::fprintf(stderr, "usage: rectify_check <in.bin> <maps.bin> <out.bin>\n");
        return 2;
    }
    std::vector<char> in = slurp(argv[1]), mp = slurp(argv[2]);
    if (in.empty() || mp.size() < 8) {
        std::fprintf(stderr, "cannot read the inputs\n");
        return 2;
    }
    int32_t hdr[9];
    float opt[3];
    std::memcpy(hdr, in.data(), sizeof hdr);
    std::memcpy(opt, in.data() + sizeof hdr, sizeof opt);
    const int n = hdr[0], src_rows = hdr[1], src_cols = hdr[2], depth = hdr[3];
    const size_t es = depth == IMG_16U ? 2 : 1;
    const size_t plane = (size_t)src_rows * src_cols * es;
    const char* base = in.data() + sizeof hdr + sizeof opt;
    int32_t msize[2];
    std::memcpy(msize, mp.data(), sizeof msize);
    const int rows = msize[0], cols = msize[1];
    float* maps = reinterpret_cast<float*>(mp.data() + sizeof msize);
    const size_t map_elems = (size_t)rows * cols;

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
            s0.emplace_back(HostImage(src_rows, src_cols, depth, const_cast<char*>(base) + plane * i));
            s1.emplace_back(HostImage(src_rows, src_cols, depth, const_cast<char*>(base) + plane * (n + i)));
        }
        RectifyMaps m;
        Image* dev[4] = { &m.map_x0, &m.map_y0, &m.map_x1, &m.map_y1 };
        for (int k = 0; k < 4; ++k)
            dev[k]->upload(HostImage(rows, cols, IMG_32F, maps + map_elems * k));
        Image disp, corr;
        RectifyMaps wrong = m;
        wrong.map_y1 = s0.front(); // an 8U image where a CV_32FC1 map belongs
        try {
            match_rectified(s0, s1, wrong, disp, cfg, &corr);
            std::fprintf(stderr, "an 8U map was accepted\n");
            return 1;
        } catch (const Exception&) {
        }
        match_rectified(s0, s1, m, disp, cfg, &corr);
        std::vector<Image> rect;
        remap(s0, m.map_x0, m.map_y0, rect);
        std::vector<char> dbuf((size_t)rows * cols * disp.elemSize());
        disp.download(HostImage(rows, cols, disp.type(), dbuf.data()));
        std::vector<char> cbuf;
        if (!corr.empty()) {
            cbuf.resize((size_t)rows * cols * corr.elemSize());
            corr.download(HostImage(rows, cols, corr.type(), cbuf.data()));
        }
        std::vector<char> rbuf((size_t)n * rows * cols * es);
        for (int i = 0; i < n; ++i)
            rect[(size_t)i].download(HostImage(rows, cols, depth, rbuf.data() + (size_t)rows * cols * es * i));
        FILE* o = std::fopen(argv[3], "wb");
        if (!o)
            return 2;
        const int32_t oh[4] = { disp.type(), corr.empty() ? 0 : corr.type(), rows, cols };
        std::fwrite(oh, sizeof oh, 1, o);
        std::fwrite(dbuf.data(), 1, dbuf.size(), o);
        std::fwrite(cbuf.data(), 1, cbuf.size(), o);
        std::fwrite(rbuf.data(), 1, rbuf.size(), o);
        std::fclose(o);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "exception: %s\n", e.what());
        return 1;
    }
    return 0;
}
