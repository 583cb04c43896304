#include "imageio.hpp"

#include <zlib.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <limits>
#include <sstream>
#include <stdexcept>

namespace bicos_cli {
namespace {

std::vector<uint8_t> slurp(const std::string& path) {
    std::ifstream f(path, std::ios::binary);
    if (!f)
        throw std::runtime_error("cannot open " + path);
    return std::vector<uint8_t>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}

uint32_t be32(const uint8_t* p) {
    return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3];
}

int paeth(int a, int b, int c) {
    const int p = a + b - c, pa = std::abs(p - a), pb = std::abs(p - b), pc = std::abs(p - c);
    return (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
}

// ITU-R BT.601 luma with the 14-bit fixed-point weights OpenCV uses for 8-bit BGR2GRAY
inline uint32_t luma(uint32_t r, uint32_t g, uint32_t b) {
    return (r * 4899u + g * 9617u + b * 1868u + 8192u) >> 14;
}

GrayImage read_png(const std::vector<uint8_t>& file, const std::string& path, bool& was_colour) {
    static const uint8_t sig[8] = { 0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A };
    if (file.size() < 8 + 25 || std::memcmp(file.data(), sig, 8) != 0)
        throw std::runtime_error(path + ": not a PNG file");
    size_t pos = 8;
    uint32_t width = 0, height = 0;
    int depth = 0, ctype = 0, interlace = 0;
    std::vector<uint8_t> idat, palette;
    bool have_ihdr = false;
    while (pos + 12 <= file.size()) {
        const uint32_t len = be32(&file[pos]);
        const uint8_t* type = &file[pos + 4];
        if (pos + 12 + (size_t)len > file.size())
            throw std::runtime_error(path + ": truncated PNG chunk");
        const uint8_t* body = &file[pos + 8];
        if (!std::memcmp(type, "IHDR", 4)) {
            if (len != 13)
                throw std::runtime_error(path + ": bad PNG IHDR length");
            width = be32(body);
            height = be32(body + 4);
            depth = body[8];
            ctype = body[9];
            interlace = body[12];
            have_ihdr = true;
        } else if (!std::memcmp(type, "PLTE", 4)) {
            palette.assign(body, body + len);
        } else if (!std::memcmp(type, "IDAT", 4)) {
            idat.insert(idat.end(), body, body + len);
        } else if (!std::memcmp(type, "IEND", 4)) {
            break;
        }
        pos += 12 + (size_t)len;
    }
    if (!have_ihdr || width == 0 || height == 0)
        throw std::runtime_error(path + ": PNG without IHDR");
    // the library's own limits (include/bicos_b200.h: 32767 columns, 65535 rows): nothing larger is allocated
    if (width > 32767u || height > 65535u)
        throw std::runtime_error(path + ": PNG larger than 32767 x 65535");
    if (interlace != 0)
        throw std::runtime_error(path + ": interlaced PNG is not supported");
    int channels;
    switch (ctype) {
        case 0: channels = 1; break;
        case 2: channels = 3; break;
        case 3: channels = 1; break;
        case 4: channels = 2; break;
        case 6: channels = 4; break;
        default: throw std::runtime_error(path + ": bad PNG colour type");
    }
    if (ctype == 3 && depth == 16)
        throw std::runtime_error(path + ": palette PNG with 16-bit indices");
    if (!(depth == 8 || depth == 16 || (ctype == 0 && (depth == 1 || depth == 2 || depth == 4))
          || (ctype == 3 && (depth == 1 || depth == 2 || depth == 4))))
        throw std::runtime_error(path + ": unsupported PNG bit depth");
    const size_t bpp_bits = (size_t)channels * depth;
    const size_t stride = (width * bpp_bits + 7) / 8;
    const size_t bpp = bpp_bits >= 8 ? bpp_bits / 8 : 1;
    std::vector<uint8_t> raw((stride + 1) * height);
    uLongf out_len = raw.size();
    if (uncompress(raw.data(), &out_len, idat.data(), idat.size()) != Z_OK || out_len != raw.size())
        throw std::runtime_error(path + ": PNG data does not inflate");
    // undo the scanline filters in place
    std::vector<uint8_t> prev(stride, 0);
    for (uint32_t y = 0; y < height; ++y) {
        uint8_t* line = &raw[(stride + 1) * y];
        const int filter = line[0];
        uint8_t* cur = line + 1;
        for (size_t i = 0; i < stride; ++i) {
            const int a = i >= bpp ? cur[i - bpp] : 0, b = prev[i], c = i >= bpp ? prev[i - bpp] : 0;
            int v = cur[i];
            switch (filter) {
                case 0: break;
                case 1: v += a; break;
                case 2: v += b; break;
                case 3: v += (a + b) / 2; break;
                case 4: v += paeth(a, b, c); break;
                default: throw std::runtime_error(path + ": bad PNG filter");
            }
            cur[i] = (uint8_t)v;
        }
        std::memcpy(prev.data(), cur, stride);
    }
    GrayImage img;
    img.rows = (int)height;
    img.cols = (int)width;
    img.bits = depth == 16 ? 16 : 8;
    img.data.resize((size_t)width * height * (img.bits / 8));
    was_colour = ctype == 2 || ctype == 6 || ctype == 3;
    for (uint32_t y = 0; y < height; ++y) {
        const uint8_t* cur = &raw[(stride + 1) * y + 1];
        for (uint32_t x = 0; x < width; ++x) {
            uint32_t v;
            if (depth < 8) {
                const int per = 8 / depth;
                const int shift = (per - 1 - (int)(x % per)) * depth;
                const uint32_t idx = (cur[x / per] >> shift) & ((1u << depth) - 1);
                if (ctype == 3) {
                    if (3 * idx + 2 >= palette.size())
                        throw std::runtime_error(path + ": palette index out of range");
                    v = luma(palette[3 * idx], palette[3 * idx + 1], palette[3 * idx + 2]);
                } else {
                    v = idx * 255u / ((1u << depth) - 1);
                }
            } else if (depth == 8) {
                const uint8_t* p = cur + (size_t)x * channels;
                if (ctype == 3) {
                    if (3u * p[0] + 2 >= palette.size())
                        throw std::runtime_error(path + ": palette index out of range");
                    v = luma(palette[3 * p[0]], palette[3 * p[0] + 1], palette[3 * p[0] + 2]);
                } else {
                    v = channels >= 3 ? luma(p[0], p[1], p[2]) : p[0];
                }
            } else {
                const uint8_t* p = cur + (size_t)x * channels * 2;
                auto s = [&](int c) { return ((uint32_t)p[2 * c] << 8) | p[2 * c + 1]; };
                v = channels >= 3 ? (uint32_t)std::lround(0.299 * s(0) + 0.587 * s(1) + 0.114 * s(2)) : s(0);
            }
            if (img.bits == 16) {
                const uint16_t w = (uint16_t)v;
                std::memcpy(&img.data[((size_t)y * width + x) * 2], &w, 2);
            } else {
                img.data[(size_t)y * width + x] = (uint8_t)v;
            }
        }
    }
    return img;
}

GrayImage read_pgm(const std::vector<uint8_t>& file, const std::string& path) {
    size_t pos = 2;
    auto next_int = [&]() -> int {
        for (;;) {
            while (pos < file.size() && std::isspace(file[pos]))
                ++pos;
            if (pos < file.size() && file[pos] == '#') {
                while (pos < file.size() && file[pos] != '\n')
                    ++pos;
                continue;
            }
            break;
        }
        int v = 0;
        bool any = false;
        while (pos < file.size() && std::isdigit(file[pos])) {
            v = v * 10 + (file[pos++] - '0');
            any = true;
        }
        if (!any)
            throw std::runtime_error(path + ": bad PGM header");
        return v;
    };
    const int width = next_int(), height = next_int(), maxval = next_int();
    ++pos; // single whitespace after maxval
    if (width <= 0 || height <= 0 || maxval <= 0 || maxval > 65535)
        throw std::runtime_error(path + ": bad PGM header");
    GrayImage img;
    img.rows = height;
    img.cols = width;
    img.bits = maxval > 255 ? 16 : 8;
    const size_t bytes = (size_t)width * height * (img.bits / 8);
    if (pos + bytes > file.size())
        throw std::runtime_error(path + ": truncated PGM");
    img.data.assign(file.begin() + pos, file.begin() + pos + bytes);
    if (img.bits == 16) // PGM samples are big-endian
        for (size_t i = 0; i + 1 < img.data.size(); i += 2)
            std::swap(img.data[i], img.data[i + 1]);
    return img;
}

// ---- TIFF input: what camera tools write (the reference reads it through cv::imread, src/fileutils.cpp:72-75,116).
// Baseline TIFF 6.0, strips: 8 / 16-bit grey (either photometric) and 8 / 16-bit RGB[A] (-> luma, like the PNG
// reader), little or big endian, uncompressed, LZW (with or without the horizontal predictor), Deflate and
// PackBits. Tiles, palettes, sub-byte depths, JPEG-in-TIFF and planar RGB are refused with a message.
struct TiffReader {
    const std::vector<uint8_t>& f;
    const std::string& path;
    bool big = false;
    [[noreturn]] void fail(const char* what) const {
        throw std::runtime_error(path + ": " + what);
    }
    uint16_t u16(size_t at) const {
        if (at + 2 > f.size())
            fail("truncated TIFF");
        return big ? (uint16_t)(f[at] << 8 | f[at + 1]) : (uint16_t)(f[at] | f[at + 1] << 8);
    }
    uint32_t u32(size_t at) const {
        if (at + 4 > f.size())
            fail("truncated TIFF");
        return big ? ((uint32_t)f[at] << 24 | (uint32_t)f[at + 1] << 16 | (uint32_t)f[at + 2] << 8 | f[at + 3])
                   : ((uint32_t)f[at + 3] << 24 | (uint32_t)f[at + 2] << 16 | (uint32_t)f[at + 1] << 8 | f[at]);
    }
    // values of an IFD entry (types BYTE, SHORT, LONG), wherever they are stored
    std::vector<uint32_t> values(size_t entry) const {
        const uint16_t type = u16(entry + 2);
        const uint32_t count = u32(entry + 4);
        const size_t size = type == 1 ? 1 : type == 3 ? 2 : type == 4 ? 4 : 0;
        if (size == 0)
            fail("TIFF tag of an unsupported type");
        if (count > (1u << 24))
            fail("TIFF tag with an absurd count");
        size_t at = entry + 8;
        if (size * count > 4)
            at = u32(entry + 8);
        std::vector<uint32_t> v(count);
        for (uint32_t i = 0; i < count; ++i)
            v[i] = size == 1 ? (at + i < f.size() ? f[at + i] : (fail("truncated TIFF"), 0u)) : size == 2 ? u16(at + 2 * (size_t)i) : u32(at + 4 * (size_t)i);
        return v;
    }
};

// TIFF flavour of LZW: codes MSB first, 9 to 12 bits, width grows one code early, 256 = clear, 257 = end
void tiff_lzw(const uint8_t* src, size_t n, std::vector<uint8_t>& out, size_t expect) {
    struct Entry {
        uint16_t prefix;
        uint8_t last, first;
        uint16_t length;
    };
    std::vector<Entry> table(4096);
    for (int i = 0; i < 256; ++i)
        table[i] = { 0xFFFF, (uint8_t)i, (uint8_t)i, 1 };
    int next = 258, width = 9, prev = -1;
    uint32_t acc = 0;
    int bits = 0;
    size_t pos = 0;
    const size_t start = out.size();
    while (out.size() - start < expect) {
        while (bits < width && pos < n) {
            acc = (acc << 8) | src[pos++];
            bits += 8;
        }
        if (bits < width)
            break;
        const int code = (int)((acc >> (bits - width)) & ((1u << width) - 1));
        bits -= width;
        if (code == 257)
            break;
        if (code == 256) {
            next = 258;
            width = 9;
            prev = -1;
            continue;
        }
        Entry e;
        if (code < next && (code < 256 || code >= 258)) {
            e = table[code];
        } else if (code == next && prev >= 0) { // the string being defined: previous string + its own first byte
            e = { (uint16_t)prev, table[prev].first, table[prev].first, (uint16_t)(table[prev].length + 1) };
        } else {
            throw std::runtime_error("corrupt LZW data in TIFF");
        }
        const size_t at = out.size();
        out.resize(at + e.length);
        {
            size_t w = at + e.length;
            out[--w] = e.last;
            int c = e.prefix;
            while (c != 0xFFFF && w > at) {
                out[--w] = table[c].last;
                c = table[c].prefix;
            }
        }
        if (prev >= 0 && next < 4096) {
            table[next] = { (uint16_t)prev, out[at], table[prev].first, (uint16_t)(table[prev].length + 1) };
            ++next;
            if (next + 1 >= (1 << width) && width < 12)
                ++width;
        }
        prev = code;
    }
}

void tiff_packbits(const uint8_t* src, size_t n, std::vector<uint8_t>& out, size_t expect) {
    const size_t start = out.size();
    size_t pos = 0;
    while (pos < n && out.size() - start < expect) {
        const int8_t c = (int8_t)src[pos++];
        if (c >= 0) {
            const size_t len = (size_t)c + 1;
            if (pos + len > n)
                throw std::runtime_error("corrupt PackBits data in TIFF");
            out.insert(out.end(), src + pos, src + pos + len);
            pos += len;
        } else if (c != -128) {
            if (pos >= n)
                throw std::runtime_error("corrupt PackBits data in TIFF");
            out.insert(out.end(), (size_t)(1 - c), src[pos++]);
        }
    }
}

GrayImage read_tiff(const std::vector<uint8_t>& file, const std::string& path, bool& was_colour) {
    TiffReader t { file, path };
    t.big = file[0] == 'M';
    if (t.u16(2) != 42)
        t.fail("not a TIFF file (BigTIFF is not supported)");
    const size_t ifd = t.u32(4);
    const int entries = t.u16(ifd);
    uint32_t width = 0, height = 0, bits = 1, compression = 1, photometric = 1, spp = 1, rows_per_strip = 0xFFFFFFFFu;
    uint32_t planar = 1, predictor = 1, sample_format = 1;
    std::vector<uint32_t> offsets, counts;
    for (int e = 0; e < entries; ++e) {
        const size_t at = ifd + 2 + 12 * (size_t)e;
        const uint16_t tag = t.u16(at);
        auto first = [&] {
            const std::vector<uint32_t> v = t.values(at);
            if (v.empty())
                t.fail("empty TIFF tag");
            return v;
        };
        switch (tag) {
            case 256: width = first()[0]; break;
            case 257: height = first()[0]; break;
            case 258: {
                const std::vector<uint32_t> v = first();
                bits = v[0];
                for (uint32_t b: v)
                    if (b != bits)
                        t.fail("TIFF samples of different depths");
                break;
            }
            case 259: compression = first()[0]; break;
            case 262: photometric = first()[0]; break;
            case 273: offsets = first(); break;
            case 277: spp = first()[0]; break;
            case 278: rows_per_strip = first()[0]; break;
            case 279: counts = first(); break;
            case 284: planar = first()[0]; break;
            case 317: predictor = first()[0]; break;
            case 339: sample_format = first()[0]; break;
            case 322: case 323: case 324: case 325: t.fail("tiled TIFF is not supported");
            default: break;
        }
    }
    if (width == 0 || height == 0 || width > 32767u || height > 65535u)
        t.fail("TIFF without a size, or larger than 32767 x 65535");
    if (bits != 8 && bits != 16)
        t.fail("only 8- and 16-bit TIFF samples are supported");
    if (sample_format != 1)
        t.fail("only unsigned integer TIFF samples are supported");
    if (photometric > 2 || (photometric == 2 && spp < 3) || (photometric < 2 && spp > 2) || spp > 4)
        t.fail("unsupported TIFF photometric interpretation");
    if (planar != 1 && spp > 1)
        t.fail("planar TIFF is not supported");
    if (compression != 1 && compression != 5 && compression != 8 && compression != 32946 && compression != 32773)
        t.fail("unsupported TIFF compression (none, LZW, Deflate and PackBits are read)");
    if (predictor != 1 && predictor != 2)
        t.fail("unsupported TIFF predictor");
    if (offsets.empty() || offsets.size() != counts.size())
        t.fail("TIFF without strips");
    if (rows_per_strip == 0)
        t.fail("TIFF with zero rows per strip");
    rows_per_strip = std::min(rows_per_strip, height);
    if ((size_t)(height + rows_per_strip - 1) / rows_per_strip != offsets.size())
        t.fail("TIFF strip count does not match its height");

    const size_t bps = bits / 8;
    const size_t row_bytes = (size_t)width * spp * bps;
    std::vector<uint8_t> raw;
    raw.reserve(row_bytes * height);
    for (size_t sidx = 0; sidx < offsets.size(); ++sidx) {
        const size_t rows_here = std::min<size_t>(rows_per_strip, height - sidx * rows_per_strip);
        const size_t expect = rows_here * row_bytes;
        if ((size_t)offsets[sidx] + counts[sidx] > file.size())
            t.fail("TIFF strip beyond the end of the file");
        const uint8_t* src = &file[offsets[sidx]];
        const size_t before = raw.size();
        if (compression == 1) {
            if (counts[sidx] < expect)
                t.fail("short TIFF strip");
            raw.insert(raw.end(), src, src + expect);
        } else if (compression == 5) {
            tiff_lzw(src, counts[sidx], raw, expect);
        } else if (compression == 32773) {
            tiff_packbits(src, counts[sidx], raw, expect);
        } else {
            raw.resize(before + expect);
            uLongf out_len = expect;
            if (uncompress(&raw[before], &out_len, src, counts[sidx]) != Z_OK || out_len != expect)
                t.fail("TIFF strip does not inflate");
        }
        if (raw.size() - before < expect)
            t.fail("short TIFF strip");
        raw.resize(before + expect);
        if (predictor == 2) // horizontal differencing, per sample, in the file's byte order
            for (size_t y = 0; y < rows_here; ++y) {
                uint8_t* line = &raw[before + y * row_bytes];
                if (bps == 1) {
                    for (size_t i = spp; i < (size_t)width * spp; ++i)
                        line[i] = (uint8_t)(line[i] + line[i - spp]);
                } else {
                    auto get = [&](size_t i) { return t.big ? (uint16_t)(line[2 * i] << 8 | line[2 * i + 1]) : (uint16_t)(line[2 * i] | line[2 * i + 1] << 8); };
                    for (size_t i = spp; i < (size_t)width * spp; ++i) {
                        const uint16_t v = (uint16_t)(get(i) + get(i - spp));
                        line[2 * i + (t.big ? 0 : 1)] = (uint8_t)(v >> 8);
                        line[2 * i + (t.big ? 1 : 0)] = (uint8_t)v;
                    }
                }
            }
    }

    GrayImage img;
    img.rows = (int)height;
    img.cols = (int)width;
    img.bits = (int)bits;
    img.data.resize((size_t)width * height * bps);
    was_colour = photometric == 2;
    const uint32_t maxv = bits == 16 ? 65535u : 255u;
    for (size_t px = 0; px < (size_t)width * height; ++px) {
        auto sample = [&](size_t c) -> uint32_t {
            const uint8_t* p = &raw[(px * spp + c) * bps];
            return bps == 1 ? p[0] : t.big ? (uint32_t)(p[0] << 8 | p[1]) : (uint32_t)(p[0] | p[1] << 8);
        };
        uint32_t v = photometric == 2 ? luma(sample(0), sample(1), sample(2)) : sample(0);
        if (photometric == 0 && bps == 1)
            v = maxv - v; // WhiteIsZero: inverted for 8-bit samples only -- OpenCV's reader, i.e. what the reference sees, returns 16-bit samples as stored
        if (bps == 1) {
            img.data[px] = (uint8_t)v;
        } else {
            const uint16_t w = (uint16_t)v;
            std::memcpy(&img.data[2 * px], &w, 2);
        }
    }
    return img;
}

// the disparity TIFFs write_tiff produces, read back as a prior (bicos-cli --disparity-prior): one channel,
// uncompressed strips, int16 (SampleFormat 2) or float32 (SampleFormat 3), either byte order
DisparityImage read_disparity_tiff(const std::vector<uint8_t>& file, const std::string& path) {
    TiffReader t { file, path };
    if (file.size() < 8 || !((file[0] == 'I' && file[1] == 'I') || (file[0] == 'M' && file[1] == 'M')))
        t.fail("not a TIFF file");
    t.big = file[0] == 'M';
    if (t.u16(2) != 42)
        t.fail("not a TIFF file (BigTIFF is not supported)");
    const size_t ifd = t.u32(4);
    const int entries = t.u16(ifd);
    uint32_t width = 0, height = 0, bits = 1, compression = 1, spp = 1, rows_per_strip = 0xFFFFFFFFu, sample_format = 1;
    std::vector<uint32_t> offsets, counts;
    for (int e = 0; e < entries; ++e) {
        const size_t at = ifd + 2 + 12 * (size_t)e;
        const std::vector<uint32_t> v = t.values(at);
        if (v.empty())
            t.fail("empty TIFF tag");
        switch (t.u16(at)) {
            case 256: width = v[0]; break;
            case 257: height = v[0]; break;
            case 258: bits = v[0]; break;
            case 259: compression = v[0]; break;
            case 273: offsets = v; break;
            case 277: spp = v[0]; break;
            case 278: rows_per_strip = v[0]; break;
            case 279: counts = v; break;
            case 339: sample_format = v[0]; break;
            case 322: case 323: case 324: case 325: t.fail("tiled TIFF is not supported");
            default: break;
        }
    }
    if (width == 0 || height == 0 || width > 32767u || height > 65535u)
        t.fail("TIFF without a size, or larger than 32767 x 65535");
    if (spp != 1 || compression != 1 || !((bits == 16 && sample_format == 2) || (bits == 32 && sample_format == 3)))
        t.fail("a disparity TIFF is one uncompressed channel of int16 or float32");
    if (offsets.empty() || offsets.size() != counts.size() || rows_per_strip == 0)
        t.fail("TIFF without strips");
    rows_per_strip = std::min(rows_per_strip, height);
    if ((size_t)(height + rows_per_strip - 1) / rows_per_strip != offsets.size())
        t.fail("TIFF strip count does not match its height");
    const size_t bps = bits / 8, row_bytes = (size_t)width * bps;
    DisparityImage img;
    img.rows = (int)height;
    img.cols = (int)width;
    img.type = bits == 16 ? 3 : 5;
    img.data.reserve(row_bytes * height);
    for (size_t sidx = 0; sidx < offsets.size(); ++sidx) {
        const size_t expect = std::min<size_t>(rows_per_strip, height - sidx * rows_per_strip) * row_bytes;
        if ((size_t)offsets[sidx] + counts[sidx] > file.size() || counts[sidx] < expect)
            t.fail("short TIFF strip");
        img.data.insert(img.data.end(), &file[offsets[sidx]], &file[offsets[sidx]] + expect);
    }
    if (t.big) // to the host's (little-endian) order
        for (size_t i = 0; i < img.data.size(); i += bps)
            std::reverse(&img.data[i], &img.data[i] + bps);
    return img;
}

void put_be32(std::vector<uint8_t>& v, uint32_t x) {
    v.push_back(x >> 24);
    v.push_back(x >> 16);
    v.push_back(x >> 8);
    v.push_back(x);
}

void png_chunk(std::vector<uint8_t>& out, const char* type, const std::vector<uint8_t>& body) {
    put_be32(out, (uint32_t)body.size());
    const size_t start = out.size();
    out.insert(out.end(), type, type + 4);
    out.insert(out.end(), body.begin(), body.end());
    put_be32(out, (uint32_t)crc32(0, &out[start], (uInt)(out.size() - start)));
}

} // namespace

GrayImage read_image(const std::string& path, bool& was_colour) {
    was_colour = false;
    const std::vector<uint8_t> file = slurp(path);
    if (file.size() >= 2 && file[0] == 'P' && file[1] == '5')
        return read_pgm(file, path);
    if (file.size() >= 8 && ((file[0] == 'I' && file[1] == 'I') || (file[0] == 'M' && file[1] == 'M')))
        return read_tiff(file, path, was_colour);
    return read_png(file, path, was_colour);
}

DisparityImage read_disparity_tiff(const std::string& path) {
    return read_disparity_tiff(slurp(path), path);
}

#include "colormaps.inc"

void colormap_lut(Colormap map, uint8_t lut[256][3]) {
    std::memcpy(lut, map == Colormap::TURBO ? LUT_TURBO : LUT_VIRIDIS, 256 * 3);
}

void write_png_rgb(const std::string& path, int rows, int cols, const std::vector<uint8_t>& rgb) {
    std::vector<uint8_t> raw((size_t)rows * (3 * (size_t)cols + 1));
    for (int y = 0; y < rows; ++y) {
        raw[(size_t)y * (3 * cols + 1)] = 0; // filter: none
        std::memcpy(&raw[(size_t)y * (3 * cols + 1) + 1], &rgb[(size_t)y * 3 * cols], 3 * (size_t)cols);
    }
    uLongf zlen = compressBound(raw.size());
    std::vector<uint8_t> z(zlen);
    if (compress2(z.data(), &zlen, raw.data(), raw.size(), 6) != Z_OK)
        throw std::runtime_error("deflate failed for " + path);
    z.resize(zlen);
    std::vector<uint8_t> out = { 0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A };
    std::vector<uint8_t> ihdr;
    put_be32(ihdr, (uint32_t)cols);
    put_be32(ihdr, (uint32_t)rows);
    ihdr.insert(ihdr.end(), { 8, 2, 0, 0, 0 }); // 8-bit RGB, deflate, adaptive filtering, no interlace
    png_chunk(out, "IHDR", ihdr);
    png_chunk(out, "IDAT", z);
    png_chunk(out, "IEND", {});
    std::ofstream f(path, std::ios::binary);
    if (!f.write(reinterpret_cast<const char*>(out.data()), (std::streamsize)out.size()))
        throw std::runtime_error("cannot write " + path);
}

void write_tiff(const std::string& path, int rows, int cols, int bits, int sample_format, const void* data) {
    // little-endian baseline TIFF, one uncompressed strip
    const uint32_t nbytes = (uint32_t)((size_t)rows * cols * (bits / 8));
    std::vector<uint8_t> out;
    auto u16 = [&](uint16_t v) {
        out.push_back(v & 0xFF);
        out.push_back(v >> 8);
    };
    auto u32 = [&](uint32_t v) {
        for (int i = 0; i < 4; ++i)
            out.push_back((v >> (8 * i)) & 0xFF);
    };
    out.insert(out.end(), { 'I', 'I' });
    u16(42);
    u32(8 + nbytes + (nbytes & 1)); // IFD after the pixel data
    out.insert(out.end(), static_cast<const uint8_t*>(data), static_cast<const uint8_t*>(data) + nbytes);
    if (nbytes & 1)
        out.push_back(0);
    struct Entry {
        uint16_t tag, type;
        uint32_t count, value;
    };
    const Entry entries[] = {
        { 256, 4, 1, (uint32_t)cols }, // ImageWidth
        { 257, 4, 1, (uint32_t)rows }, // ImageLength
        { 258, 3, 1, (uint32_t)bits }, // BitsPerSample
        { 259, 3, 1, 1 }, // Compression: none
        { 262, 3, 1, 1 }, // Photometric: BlackIsZero
        { 273, 4, 1, 8 }, // StripOffsets
        { 277, 3, 1, 1 }, // SamplesPerPixel
        { 278, 4, 1, (uint32_t)rows }, // RowsPerStrip
        { 279, 4, 1, nbytes }, // StripByteCounts
        { 339, 3, 1, (uint32_t)sample_format }, // SampleFormat
    };
    u16(sizeof entries / sizeof entries[0]);
    for (const Entry& e: entries) {
        u16(e.tag);
        u16(e.type);
        u32(e.count);
        if (e.type == 3) {
            u16((uint16_t)e.value);
            u16(0);
        } else {
            u32(e.value);
        }
    }
    u32(0);
    std::ofstream f(path, std::ios::binary);
    if (!f.write(reinterpret_cast<const char*>(out.data()), (std::streamsize)out.size()))
        throw std::runtime_error("cannot write " + path);
}

std::vector<uint8_t> colorize(const void* image, int type, int rows, int cols, Colormap map) {
    const size_t n = (size_t)rows * cols;
    auto value = [&](size_t i, bool& valid) -> double {
        if (type == 3) {
            const int16_t v = static_cast<const int16_t*>(image)[i];
            valid = v != std::numeric_limits<int16_t>::lowest();
            return v;
        }
        const double v = type == 5 ? (double)static_cast<const float*>(image)[i] : static_cast<const double*>(image)[i];
        valid = v == v;
        return v;
    };
    double lo = std::numeric_limits<double>::infinity(), hi = -lo;
    for (size_t i = 0; i < n; ++i) {
        bool ok;
        const double v = value(i, ok);
        if (ok) {
            lo = std::fmin(lo, v);
            hi = std::fmax(hi, v);
        }
    }
    const double scale = hi > lo ? 255.0 / (hi - lo) : 0.0;
    uint8_t lut[256][3];
    colormap_lut(map, lut);
    std::vector<uint8_t> rgb(n * 3, 0);
    for (size_t i = 0; i < n; ++i) {
        bool ok;
        const double v = value(i, ok);
        if (!ok)
            continue; // invalid pixels stay black
        const int g = (int)std::fmin(255.0, std::fmax(0.0, std::nearbyint((v - lo) * scale)));
        std::memcpy(&rgb[3 * i], lut[g], 3);
    }
    return rgb;
}

bool read_q_matrix(const std::string& path, double q[16], std::string& error) {
    std::ifstream f(path);
    if (!f) {
        error = "cannot open " + path;
        return false;
    }
    std::stringstream ss;
    ss << f.rdbuf();
    const std::string text = ss.str();
    // YAML "Q: !!opencv-matrix ... data: [ ... ]" or XML "<Q ...> ... <data> ... </data>"
    size_t at = text.find("Q:");
    if (at == std::string::npos)
        at = text.find("<Q");
    if (at == std::string::npos) {
        error = "no matrix named Q in " + path;
        return false;
    }
    at = text.find("data", at);
    if (at == std::string::npos) {
        error = "matrix Q has no data in " + path;
        return false;
    }
    at += 4;
    int count = 0;
    const char* p = text.c_str() + at;
    while (*p && count < 16) {
        if (*p == ']' || (*p == '<' && p[1] == '/'))
            break;
        if (std::isdigit((unsigned char)*p) || *p == '-' || *p == '+' || (*p == '.' && std::isdigit((unsigned char)p[1]))) {
            char* end = nullptr;
            q[count++] = std::strtod(p, &end);
            p = end;
        } else {
            ++p;
        }
    }
    if (count != 16) {
        error = "matrix Q in " + path + " does not have 16 elements";
        return false;
    }
    return true;
}

} // namespace bicos_cli
