// Dependency-free image I/O for bicos-cli: what the reference CLI gets from OpenCV's imgcodecs,
// imgproc (normalize + applyColorMap) and calib3d (reprojectImageTo3D).
//   reference src/fileutils.cpp:30-154 (save_image, read_sequence, sort_sequence_to_stack)
//   reference include/fileutils.hpp:43-89 (save_pointcloud)
//   reference src/cli.cpp:228-250 (Q matrix, reprojection)
// Readers: PNG (8/16-bit gray, gray+alpha, RGB, RGBA, palette; non-interlaced), binary PGM
// (P5, 8/16 bit) and strip TIFF (8/16-bit gray or RGB[A]; uncompressed, LZW, Deflate, PackBits; both
// byte orders) -- the formats multi-shot camera rigs dump -- and the int16 / float32 disparity TIFFs of write_tiff. Writers: 8-bit RGB PNG, single-strip uncompressed TIFF (int16 / float32 /
// float64), ASCII .xyz. zlib is the only library used.
#pragma once

#include <cstdint>
#include <string>
#include <vector>

namespace bicos_cli {

struct GrayImage {
    int rows = 0, cols = 0;
    int bits = 8; // 8 or 16
    std::vector<uint8_t> data; // dense rows, native-endian uint8 / uint16
};

// throws std::runtime_error with the file name on any failure
GrayImage read_image(const std::string& path, bool& was_colour);

enum class Colormap { TURBO, VIRIDIS };

// 256-entry RGB table (colormaps.inc: OpenCV's COLORMAP_TURBO / COLORMAP_VIRIDIS, tabulated)
void colormap_lut(Colormap map, uint8_t lut[256][3]);

void write_png_rgb(const std::string& path, int rows, int cols, const std::vector<uint8_t>& rgb);

struct DisparityImage {
    int rows = 0, cols = 0;
    int type = 3; // 3 = int16, 5 = float32
    std::vector<uint8_t> data; // dense rows, native-endian
};

// the single-channel disparity TIFFs write_tiff writes: uncompressed strips of int16 (SampleFormat 2, 16 bits) or
// float32 (SampleFormat 3, 32 bits); anything else throws std::runtime_error with the file name
DisparityImage read_disparity_tiff(const std::string& path);

// sample_format: 1 = unsigned int, 2 = signed int, 3 = IEEE float
void write_tiff(const std::string& path, int rows, int cols, int bits, int sample_format, const void* data);

// min-max normalisation of the valid pixels to 0..255 + colormap, invalid pixels black:
// reference save_image (fileutils.cpp:30-45). `type`: 3 = int16 (invalid -32768), 5 = float32,
// 6 = float64 (invalid NaN).
std::vector<uint8_t> colorize(const void* image, int type, int rows, int cols, Colormap map);

// "Q" from an OpenCV FileStorage file (YAML or XML), row-major 4x4
bool read_q_matrix(const std::string& path, double q[16], std::string& error);

} // namespace bicos_cli
