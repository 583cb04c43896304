// C++ consumer of include/BICOS/reproject.hpp, built with plain g++ like api_check.cpp and driven by
// tests/test_reproject.py: BICOS::reproject and BICOS::reproject_points on an uploaded disparity, checked against
// this file's own copy of the scalar loop bicos-cli used to run on the host.
//
//   reproject_check <in.bin> <out.bin>
//
// in.bin: int32 rows, cols, type (3 = CV_16SC1, 5 = CV_32FC1), allow_negative_z; 16 float64 Q (row-major); the
// disparity, dense. out.bin: uint64 kept, invalid, non-finite, negative Z; the dense map (rows * cols * 3 float32);
// the kept points (kept * 3 float32); their pixel indices (kept int32). Exit code 1 on any disagreement with the loop.
#include <BICOS/reproject.hpp>

#include <cmath>
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

static bool same_bits(float a, float b) {
    return std::memcmp(&a, &b, sizeof a) == 0;
}

int main(int argc, char** argv) {
    if (argc < 3) {
        std::fprintf(stderr, "usage: reproject_check <in.bin> <out.bin>\n");
        return 2;
    }
    std::vector<char> in = slurp(argv[1]);
    if (in.size() < 16 + 128) {
        std::fprintf(stderr, "cannot read the input\n");
        return 2;
    }
    int32_t hdr[4];
    std::array<double, 16> q;
    std::memcpy(hdr, in.data(), sizeof hdr);
    std::memcpy(q.data(), in.data() + sizeof hdr, sizeof(double) * 16);
    const int rows = hdr[0], cols = hdr[1], type = hdr[2];
    const bool allow_negative_z = hdr[3] != 0;
    char* disp = in.data() + sizeof hdr + sizeof(double) * 16;
    const size_t px = (size_t)rows * cols;

    // the loop, as bicos-cli ran it on the host
    std::vector<float> want_dense(3 * px, std::nanf("")), want_points;
    std::vector<int32_t> want_index;
    unsigned long long want_counts[4] = { 0, 0, 0, 0 };
    for (int r = 0; r < rows; ++r)
        for (int c = 0; c < cols; ++c) {
            const size_t i = (size_t)r * cols + c;
            double d;
            if (type == IMG_16S) {
                int16_t v;
                std::memcpy(&v, disp + 2 * i, 2);
                if (v == -32768) {
                    want_counts[1]++;
                    continue;
                }
                d = v;
            } else {
                float v;
                std::memcpy(&v, disp + 4 * i, 4);
                if (std::isnan(v) || v == -32768.0f) {
                    want_counts[1]++;
                    continue;
                }
                d = v;
            }
            const double in4[4] = { (double)c, (double)r, d, 1.0 };
            double o[4];
            for (int k = 0; k < 4; ++k)
                o[k] = q[4 * k] * in4[0] + q[4 * k + 1] * in4[1] + q[4 * k + 2] * in4[2] + q[4 * k + 3] * in4[3];
            const float x = (float)(o[0] / o[3]), y = (float)(o[1] / o[3]), z = (float)(o[2] / o[3]);
            if (!std::isfinite(x) || !std::isfinite(y) || !std::isfinite(z)) {
                want_counts[2]++;
                continue;
            }
            if (!allow_negative_z && z < 0.0f) {
                want_counts[3]++;
                continue;
            }
            want_counts[0]++;
            want_dense[3 * i] = x;
            want_dense[3 * i + 1] = y;
            want_dense[3 * i + 2] = z;
            want_points.insert(want_points.end(), { x, y, z });
            want_index.push_back((int32_t)i);
        }

    try {
        Image d(HostImage(rows, cols, type, disp));
        Image xyz, points, index;
        reproject(d, q, xyz, allow_negative_z);
        if (xyz.type() != IMG_32FC3 || xyz.channels() != 3 || xyz.elemSize() != 12 || xyz.rows != rows || xyz.cols != cols) {
            std::fprintf(stderr, "reproject: xyz is not a rows x cols CV_32FC3 image\n");
            return 1;
        }
        std::vector<float> dense(3 * px);
        xyz.download(HostImage(rows, cols, IMG_32FC3, dense.data()));
        const ReprojectCounts n = reproject_points(d, q, points, &index, allow_negative_z);
        if (points.type() != IMG_32FC3 || points.rows != 1 || (size_t)points.cols != px || index.type() != IMG_32S ||
            (size_t)index.cols != px) {
            std::fprintf(stderr, "reproject_points: outputs are not 1 x rows*cols CV_32FC3 / CV_32SC1 images\n");
            return 1;
        }
        std::vector<float> pts(3 * px);
        std::vector<int32_t> idx(px);
        points.download(HostImage(1, (int)px, IMG_32FC3, pts.data()));
        index.download(HostImage(1, (int)px, IMG_32S, idx.data()));
        const unsigned long long got_counts[4] = { n.points, n.invalid_disparity, n.non_finite, n.negative_z };
        if (std::memcmp(got_counts, want_counts, sizeof got_counts) != 0) {
            std::fprintf(stderr, "counts %llu %llu %llu %llu, the loop: %llu %llu %llu %llu\n", got_counts[0], got_counts[1],
                         got_counts[2], got_counts[3], want_counts[0], want_counts[1], want_counts[2], want_counts[3]);
            return 1;
        }
        for (size_t i = 0; i < 3 * px; ++i)
            if (!(std::isnan(dense[i]) && std::isnan(want_dense[i])) && !same_bits(dense[i], want_dense[i])) {
                std::fprintf(stderr, "dense value %zu differs\n", i);
                return 1;
            }
        for (size_t i = 0; i < n.points; ++i)
            if (idx[i] != want_index[i] || !same_bits(pts[3 * i], want_points[3 * i]) ||
                !same_bits(pts[3 * i + 1], want_points[3 * i + 1]) || !same_bits(pts[3 * i + 2], want_points[3 * i + 2])) {
                std::fprintf(stderr, "point %zu differs\n", i);
                return 1;
            }
        Image wrong(rows, cols, IMG_64F);
        try {
            reproject(wrong, q, xyz);
            std::fprintf(stderr, "a CV_64FC1 disparity was accepted\n");
            return 1;
        } catch (const Exception&) {
        }
        FILE* o = std::fopen(argv[2], "wb");
        if (!o)
            return 2;
        std::fwrite(got_counts, sizeof got_counts, 1, o);
        std::fwrite(dense.data(), sizeof(float), dense.size(), o);
        std::fwrite(pts.data(), sizeof(float), 3 * n.points, o);
        std::fwrite(idx.data(), sizeof(int32_t), n.points, o);
        std::fclose(o);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "exception: %s\n", e.what());
        return 1;
    }
    return 0;
}
