// bicos-cli on the B200 path: same options, defaults and outputs as the reference CLI
// (reference src/cli.cpp:55-253), without its dependencies (cxxopts, fmt, OpenCV): the argument
// parser and the image I/O (imageio.cpp) are self-contained, the matching is BICOS::match from
// include/BICOS/match.hpp, the point cloud of -q is BICOS::reproject_points from include/BICOS/reproject.hpp,
// --speckles is BICOS::filter_speckles from include/BICOS/speckles.hpp and --disparity-prior is
// BICOS::windows_from_disparity + BICOS::match_windows from include/BICOS/windows.hpp.
//
//   bicos-cli folder0 [folder1] [-t thr] [-v var] [-s step] [-o out.png] [-n N] [-q Q.yaml]
//             [--allow-negative-z] [-m lr-maxdiff] [--double] [--limited] [--corrmap] [--no-dupes] [--wide-descriptors]
//             [--disparity-range MIN:MAX] [--disparity-prior FILE:MARGIN] [--speckles SIZE:DIFF]
//
// Differences, on purpose: --allow-negative-z is honoured (the reference reads a non-existent
// "allow-behind" option, cli.cpp:231); integer-mode disparities with a threshold are float32
// with -32768.0 as the invalid marker (the reference CPU backend's convention, which this
// library follows) and are masked as invalid in the outputs.
#include <BICOS/match.hpp>
#include <BICOS/reproject.hpp>
#include <BICOS/speckles.hpp>
#include <BICOS/windows.hpp>

#include "imageio.hpp"

#include <unistd.h>

#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <iostream>
#include <map>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

namespace fs = std::filesystem;
using namespace BICOS;
using namespace bicos_cli;

namespace {

const char* LICENSE_HEADER =
    "bicos-cli (B200 path): drop-in for libBICOS' bicos-cli, LGPL-3.0-or-later interface.\n";

struct Option {
    const char* name; // long name
    char shortname; // 0 = none
    bool takes_value;
    const char* help;
};

const Option OPTIONS[] = {
    { "threshold", 't', true, "Minimum normalized cross corellation for a match to be accepted. Set to 0.0 to disable. (default: 0.75)" },
    { "variance", 'v', true, "Minimum intensity variance. Only active with --threshold. (default: 1.0)" },
    { "step", 's', true, "Stepsize for subpixel interpolation. Only effective when threshold is set." },
    { "out", 'o', true, "Output file for disparity image. (default: bicosdisp.png)" },
    { "stacksize", 'n', true, "Number of images to process. Defaults to all found in the input folders." },
    { "qmatrix", 'q', true, "Path to cv::FileStorage with single matrix \"Q\" for reconstructing a pointcloud." },
    { "allow-negative-z", 0, false, "Allow for points with negative Z values in the pointcloud output. Only effective with a given qmatrix." },
    { "lr-maxdiff", 'm', true, "Maximum disparity difference between left and right image. Enabling this disables duplicate filtering." },
    { "double", 0, false, "Set double instead of single precision" },
    { "limited", 0, false, "Limit transformation mode. Allows for more images to be used." },
    { "corrmap", 0, false, "Output map of normalized cross correlation values." },
    { "no-dupes", 0, false, "Default BICOS variant when --lr-maxdiff is not specified. Can be set together with --lr-maxdiff to activate both." },
    { "wide-descriptors", 0, false, "Extension: accept 17..23 images without --limited (384 / 512-bit descriptors; the reference stops at 16)." },
    { "disparity-range", 0, true, "Extension: search only disparities MIN..MAX (inclusive, may be negative), e.g. 0:127. (default: the whole row)" },
    { "disparity-prior", 0, true, "Extension: search only within MARGIN px of the disparity in FILE, an int16 or float32 .tiff this tool wrote for the same image size, e.g. last.tiff:4. Pixels without a valid prior search --disparity-range, else the whole row. (default: off)" },
    { "speckles", 0, true, "Extension: after the match, mark connected blobs of at most SIZE pixels whose neighbours differ by at most DIFF as invalid, e.g. 100:1. (default: off)" },
    { "help", 'h', false, "Display this message." },
};

struct Args {
    std::map<std::string, std::string> values;
    std::vector<std::string> positional;
    bool has(const std::string& k) const {
        return values.count(k) != 0;
    }
    const std::string& get(const std::string& k) const {
        return values.at(k);
    }
};

const Option* find_option(const std::string& name, char shortname) {
    for (const Option& o: OPTIONS)
        if ((!name.empty() && name == o.name) || (shortname && shortname == o.shortname))
            return &o;
    return nullptr;
}

Args parse(int argc, char const* const* argv) {
    Args a;
    for (int i = 1; i < argc; ++i) {
        const std::string arg = argv[i];
        const Option* opt = nullptr;
        std::optional<std::string> inline_value;
        if (arg.rfind("--", 0) == 0) {
            const size_t eq = arg.find('=');
            opt = find_option(arg.substr(2, eq == std::string::npos ? std::string::npos : eq - 2), 0);
            if (eq != std::string::npos)
                inline_value = arg.substr(eq + 1);
        } else if (arg.size() >= 2 && arg[0] == '-' && !std::isdigit((unsigned char)arg[1]) && arg[1] != '.') {
            opt = find_option("", arg[1]);
            if (arg.size() > 2)
                inline_value = arg.substr(2);
        } else {
            a.positional.push_back(arg);
            continue;
        }
        if (!opt)
            throw std::invalid_argument("Option '" + arg + "' does not exist");
        if (!opt->takes_value) {
            a.values[opt->name] = "1";
        } else if (inline_value) {
            a.values[opt->name] = *inline_value;
        } else {
            if (i + 1 >= argc)
                throw std::invalid_argument(std::string("Option '") + opt->name + "' is missing an argument");
            a.values[opt->name] = argv[++i];
        }
    }
    return a;
}

void print_help(const char* prog) {
    std::printf("cli to process images with BICOS\nUsage:\n  %s [OPTION...] folder0 [folder1]\n\n", prog);
    std::printf("  folder0  First folder containing input images with numbered names.\n");
    std::printf("  folder1  Optional second folder with input images. If specified, file names need to be 0.png, 1.png... "
                "Else, folder0 needs to contain 0_left.png, 0_right.png, 1_left.png...\n\n");
    for (const Option& o: OPTIONS) {
        std::string left = o.shortname ? std::string("-") + o.shortname + ", --" + o.name : std::string("    --") + o.name;
        if (o.takes_value)
            left += " arg";
        std::printf("  %-26s %s\n", left.c_str(), o.help);
    }
}

float to_float(const Args& a, const char* key, float fallback) {
    if (!a.has(key))
        return fallback;
    size_t used = 0;
    const float v = std::stof(a.get(key), &used);
    if (used != a.get(key).size())
        throw std::invalid_argument(std::string("Argument '") + a.get(key) + "' failed to parse");
    return v;
}

unsigned to_uint(const Args& a, const char* key) {
    size_t used = 0;
    const long v = std::stol(a.get(key), &used);
    if (used != a.get(key).size() || v < 0)
        throw std::invalid_argument(std::string("Argument '") + a.get(key) + "' failed to parse");
    return (unsigned)v;
}

struct Entry {
    size_t idx;
    GrayImage img;
    bool operator<(const Entry& o) const {
        return idx < o.idx;
    }
};

// reference read_sequence / read_single_dir (fileutils.cpp:60-131): numbered file names, either
// two folders with N.png or one folder with N_left.png / N_right.png
void read_dir(const fs::path& dir, bool paired, std::vector<Entry>& left, std::vector<Entry>& right) {
    static const char* ERR_SINGLE = "Expecting numbered files with names NN.png; e.g 0.png, 1.png...";
    static const char* ERR_PAIRED =
        "Expecting numbered files with names NN_{left,right}.png; e.g.: 5_left.png, 10_right.png...";
    for (const auto& e: fs::directory_iterator(dir)) {
        const std::string fname = e.path().filename().string();
        if (paired && fname.find('_') == std::string::npos)
            throw std::invalid_argument(ERR_PAIRED);
        size_t used = 0;
        size_t idx = 0;
        try {
            idx = std::stoul(fname, &used);
        } catch (const std::exception&) {
            used = 0;
        }
        if (used == 0)
            throw std::invalid_argument(paired ? ERR_PAIRED : ERR_SINGLE);
        bool colour = false;
        GrayImage img = read_image(e.path().string(), colour);
        auto& seq = (!paired || fname.find("_left") != std::string::npos) ? left : right;
        seq.push_back(Entry { idx, std::move(img) });
    }
}

std::vector<Image> upload(const std::vector<Entry>& seq) {
    std::vector<Image> out;
    out.reserve(seq.size());
    for (const Entry& e: seq)
        out.emplace_back(HostImage(e.img.rows, e.img.cols, e.img.bits == 16 ? IMG_16U : IMG_8U,
                                   const_cast<uint8_t*>(e.img.data.data())));
    return out;
}

double ms_since(std::chrono::high_resolution_clock::time_point tick) {
    return std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::high_resolution_clock::now() - tick).count() / 1000.0;
}

// reference save_image (fileutils.cpp:30-58): colourised PNG + raw TIFF next to it
void save_image(const std::vector<uint8_t>& image, int type, int rows, int cols, fs::path outfile, Colormap map) {
    // float disparities of the integer path carry -32768.0 as the invalid marker: mask them like NaN
    std::vector<uint8_t> masked;
    const void* data = image.data();
    if (type == IMG_32F) {
        masked = image;
        float* p = reinterpret_cast<float*>(masked.data());
        for (size_t i = 0; i < (size_t)rows * cols; ++i)
            if (p[i] == -32768.0f)
                p[i] = std::nanf("");
        data = masked.data();
    }
    try {
        outfile.replace_extension("png");
        write_png_rgb(outfile.string(), rows, cols, colorize(data, type, rows, cols, map));
        std::cout << "Saved colorized disparity to\t\t" << outfile << std::endl;
    } catch (const std::exception&) {
        std::cerr << "Could not save to\t" << outfile << std::endl;
    }
    try {
        outfile.replace_extension("tiff");
        const int bits = type == IMG_16S ? 16 : type == IMG_32F ? 32 : 64;
        write_tiff(outfile.string(), rows, cols, bits, type == IMG_16S ? 2 : 3, data);
        std::cout << "Saved floating-point disparity to\t" << outfile << std::endl;
    } catch (const std::exception&) {
        std::cerr << "Could not save to\t" << outfile << std::endl;
    }
}

// reference cli.cpp:228-250 + fileutils.hpp:43-89: [X Y Z W] = Q [x y d 1], point = XYZ / W, reprojected on the
// device (BICOS::reproject_points, include/BICOS/reproject.hpp); only the kept points are downloaded
void save_pointcloud(const Image& disp_gpu, const std::array<double, 16>& q, bool allow_negative_z, fs::path outfile) {
    outfile.replace_extension("xyz");
    std::ofstream xyz(outfile);
    Image points;
    const ReprojectCounts n = reproject_points(disp_gpu, q, points, nullptr, allow_negative_z);
    std::vector<float> host(3 * n.points);
    if (n.points > 0)
        Image(1, (int)n.points, IMG_32FC3, points.data, points.step).download(HostImage(1, (int)n.points, IMG_32FC3, host.data()));
    for (size_t i = 0; i < n.points; ++i)
        xyz << host[3 * i] << ' ' << host[3 * i + 1] << ' ' << host[3 * i + 2] << '\n';
    xyz.close();
    std::cout << "Saved pointcloud in ascii-format to\t" << outfile << std::endl;
    if (n.non_finite > 0)
        std::cerr << "Skipped " << n.non_finite << " points with non-finite fp values" << std::endl;
    if (n.negative_z > 0)
        std::cerr << "Skipped " << n.negative_z << " points with negative Z values" << std::endl;
}

std::vector<uint8_t> download(const Image& img) {
    std::vector<uint8_t> host((size_t)img.rows * img.cols * img.elemSize());
    img.download(HostImage(img.rows, img.cols, img.type(), host.data()));
    return host;
}

int run(int argc, char const* const* argv) {
    const Args args = parse(argc, argv);
    if (args.has("help")) {
        print_help(argv[0]);
        return 0;
    }
    std::printf("%s\n", LICENSE_HEADER);
    if (!isatty(STDOUT_FILENO))
        std::cerr << "Danger: bicos-cli does not have a stable CLI interface\n";
    if (args.has("no-dupes") && !args.has("lr-maxdiff"))
        std::cerr << "'no-dupes' is the default when 'lr-maxdiff' is not set.\n";
    if (args.positional.empty())
        throw std::invalid_argument("Option 'folder0' not present");

    const fs::path folder0 = args.positional[0];
    const fs::path outfile = args.has("out") ? args.get("out") : "bicosdisp.png";
    std::optional<fs::path> folder1, q_store;
    if (args.positional.size() > 1)
        folder1 = args.positional[1];
    if (args.has("qmatrix")) {
        q_store = args.get("qmatrix");
        if (!fs::exists(*q_store))
            throw std::invalid_argument("'" + q_store->string() + "' does not exist");
    }

    std::vector<Entry> lseq, rseq;
    if (folder1) {
        std::vector<Entry> unused;
        read_dir(folder0, false, lseq, unused);
        read_dir(*folder1, false, rseq, unused);
    } else {
        read_dir(folder0, true, lseq, rseq);
    }
    if (lseq.size() != rseq.size())
        throw std::invalid_argument("Unequal number of images; left: " + std::to_string(lseq.size())
                                    + ", right: " + std::to_string(rseq.size()));
    std::sort(lseq.begin(), lseq.end());
    std::sort(rseq.begin(), rseq.end());
    if (args.has("stacksize")) {
        const unsigned n = to_uint(args, "stacksize");
        if (n < lseq.size()) {
            lseq.resize(n);
            rseq.resize(n);
        }
    }
    if (lseq.empty())
        throw std::invalid_argument("no images found");
    std::printf("Loaded %zu %d-bit images in total\n", lseq.size() + rseq.size(), lseq.front().img.bits);

    Config c;
    c.nxcorr_threshold = to_float(args, "threshold", 0.75f);
    c.mode = TransformMode::FULL;
    if (c.nxcorr_threshold.value() <= 0.0f)
        c.nxcorr_threshold = std::nullopt;
    const bool need_corrmap = args.has("corrmap");
    if (need_corrmap && !c.nxcorr_threshold.has_value()) {
        c.nxcorr_threshold = -1.0f;
        std::cerr << "Computing with nxcorr-threshold of " << c.nxcorr_threshold.value() << " because 'corrmap' is set\n";
    }
    if (args.has("step"))
        c.subpixel_step = to_float(args, "step", 0.f);
    if (args.has("limited"))
        c.mode = TransformMode::LIMITED;
    if (const float minvar = to_float(args, "variance", 1.0f); minvar > 0.0f)
        c.min_variance = minvar;
    if (args.has("double"))
        c.precision = Precision::DOUBLE;
    if (args.has("wide-descriptors"))
        c.wide_descriptors = true;
    if (args.has("disparity-range")) {
        const std::string& v = args.get("disparity-range");
        const size_t colon = v.find(':', 1); // a leading '-' is the sign of MIN
        size_t used0 = 0, used1 = 0;
        int lo = 0, hi = 0;
        try {
            if (colon == std::string::npos)
                throw std::invalid_argument("no colon");
            lo = std::stoi(v.substr(0, colon), &used0);
            hi = std::stoi(v.substr(colon + 1), &used1);
        } catch (const std::exception&) {
            used0 = 0;
        }
        if (used0 == 0 || used0 != colon || used1 != v.size() - colon - 1)
            throw std::invalid_argument("Option 'disparity-range' expects MIN:MAX, got '" + v + "'");
        c.disparity_range = DisparityRange { lo, hi };
    }
    if (args.has("lr-maxdiff"))
        c.variant = Variant::Consistency { (int)to_uint(args, "lr-maxdiff"), args.has("no-dupes") };
    std::optional<std::pair<std::string, int>> prior;
    if (args.has("disparity-prior")) {
        const std::string& v = args.get("disparity-prior");
        const size_t colon = v.rfind(':');
        size_t used = 0;
        int margin = -1;
        try {
            if (colon != std::string::npos && colon > 0)
                margin = std::stoi(v.substr(colon + 1), &used);
        } catch (const std::exception&) {
            used = 0;
        }
        if (used == 0 || used != v.size() - colon - 1 || margin < 0 || margin > 32767)
            throw std::invalid_argument("Option 'disparity-prior' expects FILE:MARGIN with MARGIN in 0..32767, got '" + v + "'");
        prior = std::make_pair(v.substr(0, colon), margin);
    }
    std::optional<std::pair<int, double>> speckles;
    if (args.has("speckles")) {
        const std::string& v = args.get("speckles");
        const size_t colon = v.find(':');
        size_t used0 = 0, used1 = 0;
        int size = 0;
        double diff = 0.0;
        try {
            if (colon == std::string::npos)
                throw std::invalid_argument("no colon");
            size = std::stoi(v.substr(0, colon), &used0);
            diff = std::stod(v.substr(colon + 1), &used1);
        } catch (const std::exception&) {
            used0 = 0;
        }
        if (used0 == 0 || used0 != colon || used1 == 0 || used1 != v.size() - colon - 1 || std::isnan(diff))
            throw std::invalid_argument("Option 'speckles' expects SIZE:DIFF, got '" + v + "'");
        speckles = std::make_pair(size, diff);
    }

    auto tick = std::chrono::high_resolution_clock::now();
    std::vector<Image> lstack = upload(lseq), rstack = upload(rseq);
    std::printf("Latency:\t %gms (upload)\t", ms_since(tick));
    std::fflush(stdout);

    DisparityWindows windows;
    if (prior) {
        const DisparityImage p = read_disparity_tiff(prior->first);
        if (p.rows != lstack.front().rows || p.cols != lstack.front().cols)
            throw std::invalid_argument("disparity prior " + prior->first + " is " + std::to_string(p.cols) + "x" + std::to_string(p.rows) +
                                        ", the images " + std::to_string(lstack.front().cols) + "x" + std::to_string(lstack.front().rows));
        const Image prior_gpu(HostImage(p.rows, p.cols, p.type, const_cast<uint8_t*>(p.data.data())));
        windows_from_disparity(prior_gpu, prior->second, c.disparity_range, windows);
        c.disparity_range = std::nullopt; // now the fallback of the windows
    }

    Image disp_gpu, corr_gpu;
    tick = std::chrono::high_resolution_clock::now();
    if (prior)
        match_windows(lstack, rstack, windows, disp_gpu, c, need_corrmap ? &corr_gpu : nullptr);
    else
        BICOS::match(lstack, rstack, disp_gpu, c, need_corrmap ? &corr_gpu : nullptr);
    SpeckleCounts removed {};
    if (speckles) {
        // speckles become the type's invalid marker, so the masking below applies unchanged: int16 -32768; float32 NaN
        // in subpixel mode and -32768.0f in integer mode; the corrmap is left as the match wrote it
        const double marker = disp_gpu.type() == IMG_32F && c.subpixel_step.value_or(-1.f) >= 0.f ? std::nan("") : -32768.0;
        filter_speckles(disp_gpu, marker, speckles->first, speckles->second, &removed);
    }
    // the reference's match() returns after its work is done (its destructors synchronise):
    // download() below synchronises the default stream, so time that part with the match
    std::vector<uint8_t> disp = download(disp_gpu);
    std::printf("%gms (match%s + disparity download)\t", ms_since(tick), speckles ? " + speckles" : "");
    std::fflush(stdout);

    tick = std::chrono::high_resolution_clock::now();
    std::vector<uint8_t> corrmap;
    if (need_corrmap && !corr_gpu.empty())
        corrmap = download(corr_gpu);
    std::printf("%gms (download)\n", ms_since(tick));

    if (speckles)
        std::printf("Removed %zu speckles (%zu pixels)\n", removed.speckles, removed.pixels);
    const int rows = disp_gpu.rows, cols = disp_gpu.cols;
    save_image(disp, disp_gpu.type(), rows, cols, outfile, Colormap::TURBO);
    if (need_corrmap && !corrmap.empty())
        save_image(corrmap, corr_gpu.type(), rows, cols,
                   outfile.parent_path() / (outfile.stem().string() + "-corrmap" + outfile.extension().string()),
                   Colormap::VIRIDIS);

    if (q_store) {
        std::array<double, 16> q {};
        std::string error;
        if (!read_q_matrix(q_store->string(), q.data(), error))
            throw std::runtime_error(error);
        save_pointcloud(disp_gpu, q, args.has("allow-negative-z"), outfile);
    }
    return 0;
}

} // namespace

int main(int argc, char const* const* argv) {
    try {
        return run(argc, argv);
    } catch (const std::exception& e) {
        std::cerr << "bicos-cli: " << e.what() << std::endl;
        return 1;
    }
}
