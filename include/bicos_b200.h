/* bicos_b200.h -- thin C ABI over the sm_100a kernels of the BICOS::match hot path.
 *
 * This is the drop-in boundary underneath the reference's public entry point
 *     void BICOS::match(const std::vector<Image>&, const std::vector<Image>&,
 *                       Image& disparity, Config, Image* corrmap [, Stream&])
 *     (reference include/match.hpp:31-41, defined src/lib.cpp:31-49)
 * and underneath its Python FFI (reference src/pybicos_c.cpp:92-209, declared for this
 * repository in include/pybicos_c.h). A maintainer of the reference would replace the body
 * of impl::cuda::match (reference src/impl/cuda.cu:465-524) by one call to
 * bicos_b200_match(); INTEGRATION.md shows that stub.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a
 * negative bicos_b200_status and records a message retrievable with
 * bicos_b200_last_error() (thread-local). No exceptions cross this boundary. All device
 * pointers must belong to the device the handle was created on. Work is enqueued on the
 * given stream (a cudaStream_t passed as void*; NULL = the legacy default stream) and is
 * NOT synchronised unless stated. There is no CPU fallback: without a CUDA device every
 * compute entry point fails with BICOS_B200_ERR_CUDA.
 */
#ifndef BICOS_B200_H
#define BICOS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BICOS_B200_MAX_IMAGES 65 /* 4n-6 <= 256 descriptor bits; reference src/impl/cuda.cu:107 */

typedef enum {
    BICOS_B200_OK = 0,
    BICOS_B200_ERR_INVALID = -1, /* BICOS::Exception / std::invalid_argument in the reference */
    BICOS_B200_ERR_CUDA = -2, /* assertCudaSuccess, reference include/impl/cuda/cutil.cuh:32-41 */
    BICOS_B200_ERR_NOMEM = -3
} bicos_b200_status;

/* OpenCV depth codes, as the reference's C ABI passes them (pybicos/__init__.py:79-83) */
#define BICOS_B200_8U 0
#define BICOS_B200_16U 2
#define BICOS_B200_16S 3
#define BICOS_B200_32F 5
#define BICOS_B200_64F 6

/* reference include/impl/common.hpp:46-47 */
#define BICOS_B200_FLAG_NODUPES 1
#define BICOS_B200_FLAG_CONSISTENCY 2
/* bicos_b200_search only, OR-ed into `flags`: the caller vouches that bit 32 K - 1 of every descriptor is zero
 * (true for everything bicos_b200_transform writes: 4n-6 and n^2-2n+3 are never multiples of 32). The
 * tensor-core engine then carries the tile column through that bit's operand byte (search_mma.cu, "CT"),
 * as bicos_b200_match does; a set top bit with this flag gives wrong matches. */
#define BICOS_B200_FLAG_TOP_BIT_FREE 4
/* bicos_b200_search only: bits 32 K - 1 AND 32 K - 2 of every descriptor are zero (also true for everything
 * bicos_b200_transform writes: 4n-6 <= 32K-2, and n^2-2n+3 mod 32 <= 27). With 128- or 256-bit descriptors and
 * flags = CONSISTENCY the tensor-core engine then takes both directions from ONE product (search_mma.cu,
 * search_mma3_kernel), as bicos_b200_match does. Implies TOP_BIT_FREE. */
#define BICOS_B200_FLAG_TOP2_BITS_FREE 8

/* Same fields, order and "negative float = unset" convention as the reference's BicosConfig
 * (src/pybicos_c.cpp:30-41 with BICOS_CUDA defined; pybicos/__init__.py:41-51), plus trailing
 * extension fields. Zero-initialise the struct: zero leaves every extension off. */
typedef struct {
    float nxcorr_threshold; /* < 0: no NXC stage, int16 result (Config::nxcorr_threshold = nullopt) */
    float subpixel_step; /* < 0: integer disparities */
    float min_variance; /* < 0: no variance test */
    int mode; /* 0 = TransformMode::LIMITED, 1 = FULL */
    int precision; /* 0 = Precision::SINGLE, 1 = DOUBLE */
    int variant_type; /* 0 = Variant::NoDuplicates, 1 = Variant::Consistency */
    int max_lr_diff; /* Consistency only */
    int no_dupes; /* Consistency only */
    /* extension, after the reference's fields: nonzero = nxcorr_threshold is a real threshold even
     * though it is negative (BICOS::Config{.nxcorr_threshold = -1.0f}: "evaluate the NXC, reject
     * nothing", what the reference CLI uses for --corrmap without --threshold, cli.cpp:150-153) */
    int negative_threshold_is_set;
    /* extension: nonzero = descriptors of 384 and 512 bits (12 / 16 words) are allowed, i.e. FULL
     * stacks of 17..23 images, which the reference rejects ("input stacks too large",
     * src/impl/cpu.cpp:154-155, src/impl/cuda.cu:519-520). 0 = the reference's limit of 256 bits. */
    int wide_descriptors;
    /* extension: nonzero = search only the pairs (left column i, right column j) with
     * min_disparity <= i - j <= max_disparity (inclusive; may be negative). The reference searches the
     * whole row (0 here). min_disparity > max_disparity is BICOS_B200_ERR_INVALID; other values are
     * accepted: bounds beyond +-(cols - 1) select no further pairs, and a range that covers the whole row
     * is the same as no range (same kernels, same results). A left pixel with no right column in range is invalid. The
     * forward search of pixel i runs over right columns [i - max, i - min], the reverse search of the
     * Consistency check from right column b over left columns [b + min, b + max]; ties as without a
     * range. The range bounds the search, not the refined value: the subpixel refinement still looks
     * at the neighbours b - 1, b + 1 of the match, so a subpixel disparity may lie up to 1 px outside
     * [min, max]. A ranged match runs as one unit (no row bands) on the integer-pipe engine; with
     * BICOS_B200_SEARCH_TENSOR forced it fails with BICOS_B200_ERR_CUDA. */
    int has_disparity_range;
    int min_disparity;
    int max_disparity;
} bicos_b200_config;

/* `mode` arguments outside a config (bicos_b200_descriptor_words, bicos_b200_transform): bit 0 is
 * the TransformMode, OR-ing this in allows wide descriptors as bicos_b200_config::wide_descriptors does */
#define BICOS_B200_MODE_WIDE 2

typedef struct bicos_b200_handle_s* bicos_b200_handle;

const char* bicos_b200_last_error(void);

/* Number of CUDA devices visible, or a negative status. */
int bicos_b200_device_count(void);

/* A handle owns the per-device workspace (descriptor buffers, search keys, the subpixel x
 * table, pinned staging for the *_host entry point). One handle serves one match at a time;
 * use one handle per concurrent stream. device < 0 = current device. */
int bicos_b200_create(bicos_b200_handle* out, int device);
int bicos_b200_destroy(bicos_b200_handle h);

/* Words (uint32) per descriptor the reference's dispatch picks for n images
 * (src/impl/cpu.cpp:122-156): 1/2/4/8, or BICOS_B200_ERR_INVALID above 256 bits (with
 * BICOS_B200_MODE_WIDE in `mode`: 12 / 16 up to 512 bits). */
int bicos_b200_descriptor_words(int n, int mode);

/* Result type codes for a configuration: disparity BICOS_B200_16S (no threshold) or
 * BICOS_B200_32F; corrmap BICOS_B200_32F / BICOS_B200_64F, 0 when no threshold is set. */
int bicos_b200_disparity_type(const bicos_b200_config* cfg);
int bicos_b200_corrmap_type(const bicos_b200_config* cfg);

/* ---- the path, stage by stage (device memory) --------------------------------------- */

/* Stage 1, reference descriptor_transform<>() (include/impl/cpu/descriptor_transform.hpp:125-138).
 * planes: host array of n device pointers to single-channel images [rows][pitch_bytes].
 * desc: device [rows][desc_pitch_words] uint32, K words per pixel, rows 16-byte aligned. */
int bicos_b200_transform(bicos_b200_handle h, const void* const* planes, int n, int rows, int cols,
                         size_t pitch_bytes, int depth, int mode, uint32_t* desc,
                         size_t desc_pitch_words, void* stream);

/* Stage 2+4a, reference bicos<>() search part (include/impl/cpu/bicos.hpp:50-76, 78-97).
 * All results are device [rows][cols] uint32 minima of keys cost << 16 | column, filled by
 * this call:
 *   fwd_first  per left pixel: lowest Hamming cost and the FIRST right column attaining it
 *   fwd_last   (FLAG_NODUPES) same cost with 65535 - column: the LAST right column attaining
 *              it; the match is unique iff both name the same column
 *   rev_first / rev_last  (FLAG_CONSISTENCY; rev_last only with FLAG_NODUPES as well) the same
 *              per right column over the left row: the reverse search of the consistency check */
int bicos_b200_search(bicos_b200_handle h, const uint32_t* desc0, const uint32_t* desc1, int K,
                      int rows, int cols, size_t desc_pitch_words, int flags, uint32_t* fwd_first,
                      uint32_t* fwd_last, uint32_t* rev_first, uint32_t* rev_last, void* stream);

/* Stage 2+4a over a disparity range (see bicos_b200_config::has_disparity_range): the same key arrays,
 * filled by this call, for the in-range pairs min_disparity <= i - j <= max_disparity only. fwd_last is
 * required for every `flags`: without FLAG_NODUPES it receives the mirror of fwd_first, and a pixel whose
 * window is empty gets 0xFFFFFFFF in both. Pass bicos_b200_refine a config with the same range: it then
 * compares fwd_first with fwd_last for every pixel, which rejects the empty windows. A range covering
 * the whole row runs bicos_b200_search. */
int bicos_b200_search_range(bicos_b200_handle h, const uint32_t* desc0, const uint32_t* desc1, int K,
                            int rows, int cols, size_t desc_pitch_words, int flags, uint32_t* fwd_first,
                            uint32_t* fwd_last, uint32_t* rev_first, uint32_t* rev_last,
                            int min_disparity, int max_disparity, void* stream);

/* ---- per-pixel disparity windows ----------------------------------------------------------
 * A window map bounds the search pixel by pixel instead of with one range for the frame: e.g. a prior from the previous
 * frame +- a margin, bounds from known geometry, or an empty window for every pixel outside a region of interest.
 * min_disparity / max_disparity: device int16 images [rows][pitch_bytes], one pitch for both, even and at least
 * cols * 2 (2-byte aligned pointers). Semantics:
 *   left pixel (r, i) pairs with right column j iff min(r, i) <= i - j <= max(r, i), clipped to the row; min > max is
 *   an empty window: the pixel is invalid (corrmap NaN) and nothing is searched or refined for it
 *   the reverse search of the Consistency check from right column b runs over the left columns a with
 *   min(r, a) <= a - b <= max(r, a): exactly the pairs the forward windows define (not necessarily contiguous)
 *   ties as without windows (the first strict minimum; with no-dupes a second minimum invalidates); the refine is
 *   unchanged, so a subpixel disparity may lie up to 1 px outside the window, as with a range
 * Constant maps (m, M) give bit for bit the result of bicos_b200_config's range [m, M] (keys, disparity, corrmap);
 * maps that cover the row, e.g. (-32768, 32767), give bit for bit the unranged match. Windows run on the integer-pipe
 * engine: with BICOS_B200_SEARCH_TENSOR forced they fail with BICOS_B200_ERR_CUDA. */
typedef struct {
    const int16_t* min_disparity;
    const int16_t* max_disparity;
    size_t pitch_bytes;
} bicos_b200_disparity_windows;

/* Stage 2+4a over window maps, with the key contract of bicos_b200_search_range: the key arrays are filled by this
 * call (the reverse ones prefilled here), fwd_last is required for every `flags` and always written (without
 * FLAG_NODUPES as the mirror of fwd_first), and an empty window gets 0xFFFFFFFF in both forward arrays. To refine
 * these keys, pass bicos_b200_refine a config with a range that does not cover the row (e.g. has_disparity_range = 1,
 * [0, 0]): that turns on its first / last comparison, which rejects the empty windows. */
int bicos_b200_search_windows(bicos_b200_handle h, const uint32_t* desc0, const uint32_t* desc1, int K, int rows, int cols,
                              size_t desc_pitch_words, int flags, uint32_t* fwd_first, uint32_t* fwd_last, uint32_t* rev_first,
                              uint32_t* rev_last, const bicos_b200_disparity_windows* windows, void* stream);

/* Stage 4b+3, reference bicos<>() postfilter (bicos.hpp:95-110) + agree / agree_subpixel
 * (include/impl/cpu/agree.hpp:53-191) on the keys of bicos_b200_search. raw_disp_out
 * (optional, dense int16 [rows][cols]) receives the postfilter result before the NXC test. */
int bicos_b200_refine(bicos_b200_handle h, const void* const* planes0, const void* const* planes1,
                      int n, int rows, int cols, size_t pitch_bytes, int depth,
                      const bicos_b200_config* cfg, const uint32_t* fwd_first, const uint32_t* fwd_last,
                      const uint32_t* rev_first, const uint32_t* rev_last, int16_t* raw_disp_out,
                      void* disparity, size_t disparity_pitch_bytes, void* corrmap,
                      size_t corrmap_pitch_bytes, void* stream);

/* ---- the whole path ------------------------------------------------------------------ */

/* Device-resident BICOS::match: transform x2 -> search -> postfilter+refine on `stream`.
 * disparity: int16 (no threshold) or float32 rows of disparity_pitch_bytes; integer mode with a
 * threshold keeps -32768.0f as the invalid marker, subpixel mode uses NaN (reference CPU
 * backend, src/impl/cpu.cpp:77-95). corrmap may be NULL; otherwise float32 (SINGLE) or
 * float64 (DOUBLE), NaN where no correlation was evaluated. */
int bicos_b200_match(bicos_b200_handle h, const void* const* planes0, const void* const* planes1,
                     int n, int rows, int cols, size_t pitch_bytes, int depth,
                     const bicos_b200_config* cfg, void* disparity, size_t disparity_pitch_bytes,
                     void* corrmap, size_t corrmap_pitch_bytes, void* stream);

/* bicos_b200_match over window maps (see bicos_b200_disparity_windows): the same outputs and types, the search
 * bounded per pixel. cfg->has_disparity_range must be 0 (windows and a range together are BICOS_B200_ERR_INVALID).
 * Runs as one unit on `stream` (no row bands); like every match it first waits for the handle's previous work when
 * that was enqueued on another stream. */
int bicos_b200_match_windows(bicos_b200_handle h, const void* const* planes0, const void* const* planes1, int n, int rows,
                             int cols, size_t pitch_bytes, int depth, const bicos_b200_config* cfg,
                             const bicos_b200_disparity_windows* windows, void* disparity, size_t disparity_pitch_bytes,
                             void* corrmap, size_t corrmap_pitch_bytes, void* stream);

/* Window maps from a prior disparity, one launch. prior: device int16 (BICOS_B200_16S) or float32 (BICOS_B200_32F)
 * [rows][prior_pitch_bytes], pitch a multiple of the element size. Per pixel:
 *   invalid prior (int16 -32768; float32 NaN, -32768.0f or +-inf): (fallback_min, fallback_max), which may be empty
 *   (min > max: the pixel is skipped) or cover the row
 *   valid prior d: min = clamp(floor(d) - margin), max = clamp(ceil(d) + margin), clamp to [-32768, 32767], computed
 *   exactly in double
 * margin 0..32767; fallback bounds within int16; rows 1..65535, cols 1..32767; min_out / max_out as in
 * bicos_b200_disparity_windows with windows_pitch_bytes. */
int bicos_b200_windows_from_disparity(bicos_b200_handle h, const void* prior, int prior_type, size_t prior_pitch_bytes, int rows,
                                      int cols, int margin, int fallback_min, int fallback_max, int16_t* min_out,
                                      int16_t* max_out, size_t windows_pitch_bytes, void* stream);

/* ---- rectification: raw camera stacks in ------------------------------------------------
 * The match expects rectified stacks (corresponding points on the same row). These entry points APPLY
 * rectification maps the caller already has, e.g. from OpenCV's cv::initUndistortRectifyMap with
 * m1type = CV_32FC1 (computing the maps from a calibration is a one-off host step and not part of this
 * library). Semantics, bit for bit those of OpenCV's CPU cv::remap(src, dst, map_x, map_y, INTER_LINEAR,
 * BORDER_CONSTANT, 0) on float32 maps:
 *   X = round_half_even(map_x(y, x) * 32), Y = likewise; x0 = X >> 5, y0 = Y >> 5 (floor), fx = X & 31, fy = Y & 31
 *   taps v00 = src(y0, x0), v01 = src(y0, x0 + 1), v10 = src(y0 + 1, x0), v11 = src(y0 + 1, x0 + 1); a tap
 *   outside the source reads 0
 *   8U:  dst = ((32-fx)(32-fy) v00 + fx(32-fy) v01 + (32-fx)fy v10 + fx fy v11 + 512) >> 10 (int32)
 *   16U: float32 weights w00 = (1-ay)(1-ax), w01 = (1-ay)ax, w10 = ay(1-ax), w11 = ay ax with ax = fx/32,
 *        ay = fy/32; dst = saturate_u16(round_half_even(((v00 w00 + v01 w01) + v10 w10) + v11 w11)), each
 *        product and sum rounded to float32 on its own
 *   a map value that is NaN, +-inf or of magnitude >= 2^25 gives 0
 * The output has the maps' size (rows x cols); the source size is independent. Both are at most 32767 x 32767.
 * Identity maps (map_x = x, map_y = y) reproduce the input exactly. */

/* Stage entry point: remaps n (1..65) device planes src_planes[i] [src_rows][src_pitch_bytes] through one map
 * pair (device float32 [rows][map_pitch_bytes], pitch a multiple of 4 and at least cols * 4) into
 * dst_planes[i] [rows][dst_pitch_bytes]. Writes exactly the rows * cols output pixels of each plane. */
int bicos_b200_remap(bicos_b200_handle h, const void* const* src_planes, int n, int src_rows, int src_cols,
                     size_t src_pitch_bytes, int depth, const float* map_x, const float* map_y, size_t map_pitch_bytes,
                     int rows, int cols, void* const* dst_planes, size_t dst_pitch_bytes, void* stream);

/* The map pairs of both cameras: device float32 [rows][map_pitch_bytes] each, one pitch for all four. */
typedef struct {
    const float* map_x0;
    const float* map_y0;
    const float* map_x1;
    const float* map_y1;
    size_t map_pitch_bytes;
} bicos_b200_rectify_maps;

/* bicos_b200_match on raw stacks: remaps planes0 through (map_x0, map_y0) and planes1 through (map_x1, map_y1)
 * (one launch for both) into a workspace the handle owns, then runs bicos_b200_match on the rectified
 * [rows][cols] stacks. The result is bit-identical to bicos_b200_remap of both stacks followed by
 * bicos_b200_match (row bands, overlap, engine choice and disparity range as for that match). The outputs
 * have the rectified size. The workspace grows on demand (128-byte aligned rows) and lives until
 * bicos_b200_destroy; like the rest of the handle's workspace it serves one match at a time, and a
 * rectified match enqueued on another stream than the handle's previous match first waits for that one. */
int bicos_b200_match_rectified(bicos_b200_handle h, const void* const* planes0, const void* const* planes1, int n,
                               int src_rows, int src_cols, size_t src_pitch_bytes, int depth,
                               const bicos_b200_rectify_maps* maps, int rows, int cols, const bicos_b200_config* cfg,
                               void* disparity, size_t disparity_pitch_bytes, void* corrmap, size_t corrmap_pitch_bytes,
                               void* stream);

/* ---- reprojection: disparity out, 3D points out -----------------------------------------
 * Turns a disparity map (of any match entry point) into 3D points through the 4x4 reprojection matrix Q of the
 * rectified rig, e.g. the Q of OpenCV's cv::stereoRectify (computing Q is a host step and not part of this
 * library). Semantics, bit for bit those of bicos-cli's point cloud, per disparity pixel (row r, column c) in
 * row-major order:
 *   skipped as invalid disparity: int16 -32768; float32 NaN or exactly -32768.0f (the marker of integer mode with
 *   a threshold, see bicos_b200_match)
 *   in = (c, r, d, 1.0) in double; o[k] = ((Q[4k] in0 + Q[4k+1] in1) + Q[4k+2] in2) + Q[4k+3] in3 for k = 0..3,
 *   every product and every sum rounded to double on its own (no FMA contraction)
 *   X = (float)(o0 / o3), Y = (float)(o1 / o3), Z = (float)(o2 / o3): IEEE division, correctly rounded; the
 *   conversion rounds to nearest even and keeps subnormals
 *   skipped as non-finite: X, Y or Z is +-inf or NaN (this includes W = o3 = 0 and values beyond the float range)
 *   skipped as negative Z: Z < 0.0f (-0.0 is kept), unless BICOS_B200_REPROJECT_ALLOW_NEGATIVE_Z is set
 *   kept: everything else
 * This is not the arithmetic of OpenCV's cv::reprojectImageTo3D, which accumulates Q's columns incrementally,
 * multiplies by 1/W and writes Z = 10000 for missing values; where both keep a point they agree within a few
 * float ULPs. */
#define BICOS_B200_REPROJECT_ALLOW_NEGATIVE_Z 1

/* Stage entry point, one launch. disparity: device int16 (BICOS_B200_16S) or float32 (BICOS_B200_32F)
 * [rows][disparity_pitch_bytes], pitch a multiple of the element size; rows and cols 1..32767. q: HOST array of
 * 16 doubles, row-major. Outputs (device; at least one of xyz and points):
 *   xyz          dense float32 [rows][xyz_pitch_bytes], X Y Z interleaved per pixel (pitch a multiple of 4 and at
 *                least cols * 12), NaN NaN NaN for every skipped pixel; may be NULL
 *   points       the kept points, float32 X Y Z (12 bytes each), densely packed in row-major pixel order: the
 *                order and content of bicos-cli's .xyz file; capacity rows * cols points; may be NULL
 *   pixel_index  int32 r * cols + c of each point, same order; capacity rows * cols; may be NULL, needs points
 *   counts       device unsigned long long [4]: kept, invalid disparity, non-finite, negative Z; they sum to
 *                rows * cols. Required with points (allowed with xyz alone). Only counts[0] entries of points
 *                and pixel_index are written.
 * Asynchronous. The call uses a workspace of the handle (grown on demand, freed by bicos_b200_destroy): a call on
 * another stream than the handle's previous work first waits for that work, as a match does. */
int bicos_b200_reproject(bicos_b200_handle h, const void* disparity, int disparity_type, size_t disparity_pitch_bytes,
                         int rows, int cols, const double q[16], int flags, float* xyz, size_t xyz_pitch_bytes,
                         float* points, int32_t* pixel_index, unsigned long long* counts, void* stream);

/* ---- speckle removal: disparity in, disparity out, in place ---------------------------------
 * Sets small connected blobs of a disparity map to `new_value`, like OpenCV's cv::filterSpeckles(img, newVal,
 * maxSpeckleSize, maxDiff), whose parameters come in the same order. disparity: device int16 (BICOS_B200_16S) or
 * float32 (BICOS_B200_32F) [rows][disparity_pitch_bytes], pitch a multiple of the element size; rows and cols
 * 1..32767. Semantics:
 *   parameters: int16: new = cvRound(new_value), diff = cvRound(max_diff), both rounded half to even; `new` outside
 *   int16 is BICOS_B200_ERR_INVALID; a diff beyond +-65535 acts as +-65535. float32: new = (float)new_value (NaN
 *   allowed), diff = (float)max_diff. A NaN max_diff is BICOS_B200_ERR_INVALID.
 *   members: pixels that are not an invalid marker (int16 -32768; float32 NaN or -32768.0f: the pixels
 *   bicos_b200_reproject skips) and not equal to `new`
 *   edges: two 4-neighbours are connected when both are members and |d(p) - d(q)| <= diff; int16 computes the
 *   difference in int32, float32 compares fabsf of the float32 difference rounded to nearest (no contraction), so
 *   inf - inf (NaN) gives no edge
 *   speckles: connected components of at most max_speckle_size members; every pixel of a speckle is set to `new`.
 *   Nothing else is written, the pitch padding included. max_speckle_size <= 0 changes nothing; a negative diff
 *   makes every member a component of its own.
 *   counts (optional, device unsigned long long [2], 8-byte aligned): the pixels set and the speckles removed.
 * For int16 with new_value = -32768, or with no -32768 pixels, the result is exactly cv::filterSpeckles' (for
 * diff <= 32767: OpenCV's IPP path truncates a larger maxDiff to int16, its plain path does not). The
 * deliberate differences: float32 is supported, and markers are never members whatever new_value is.
 * Asynchronous; four launches on every input, whatever its content. The call uses a workspace of the handle (8
 * bytes per pixel, grown on demand, freed by bicos_b200_destroy): a call on another stream than the handle's
 * previous work first waits for that work, as a match does. */
int bicos_b200_filter_speckles(bicos_b200_handle h, void* disparity, int disparity_type, size_t disparity_pitch_bytes, int rows,
                               int cols, double new_value, int max_speckle_size, double max_diff, unsigned long long* counts,
                               void* stream);

/* Throughput mode: `count` independent stereo stacks of one shape, type and configuration (BASELINE.json's batch
 * configuration). planes0[f] / planes1[f] are the n plane pointers of frame f, disparity[f] / corrmap[f] its outputs
 * (corrmap may be NULL, or hold NULL entries). Same results as `count` calls of bicos_b200_match, but the frames
 * flow through two internal streams: the transform + search of frame f + 1 (tensor cores) runs beside the
 * postfilter + refine of frame f (FP32 pipe), which the register budget of the search kernel is laid out for.
 * `stream` is joined on both sides: earlier work on it completes before the first frame starts, and it continues
 * only after the last frame is complete. The reference has no batch entry point: its callers loop over
 * BICOS::match (src/cli.cpp:188-215 per stack). */
int bicos_b200_match_batch(bicos_b200_handle h, int count, const void* const* const* planes0,
                           const void* const* const* planes1, int n, int rows, int cols, size_t pitch_bytes,
                           int depth, const bicos_b200_config* cfg, void* const* disparity,
                           size_t disparity_pitch_bytes, void* const* corrmap, size_t corrmap_pitch_bytes,
                           void* stream);

/* Whether bicos_b200_match and bicos_b200_match_batch may run the search of one unit (row band, frame) beside the
 * refine of the previous one on the handle's two internal streams (default: yes). 0 = every kernel of a match one
 * after the other on the caller's stream, as in the reference (src/impl/cuda.cu:148-458): same results, used for
 * A/B timing and when a caller wants nothing enqueued outside its own stream. */
int bicos_b200_set_overlap(bicos_b200_handle h, int enabled);

/* Host-resident variant (what pybicos' BICOS_Match needs): dense host images in, dense host
 * results out; uploads, runs bicos_b200_match and downloads through the handle's pinned
 * staging buffers, then synchronises. */
int bicos_b200_match_host(bicos_b200_handle h, const void* const* host_planes0,
                          const void* const* host_planes1, int n, int rows, int cols, int depth,
                          const bicos_b200_config* cfg, void* host_disparity, void* host_corrmap);

/* The same in two halves, for callers that keep several frames in flight (one handle per
 * frame in flight): _begin validates, enqueues all copies and kernels on the handle's own
 * streams and returns; _end blocks until the host buffers hold the results. The host buffers
 * must stay valid, and should be pinned, between the two calls. A second _begin on a handle
 * whose previous host match has not been ended is an error. */
int bicos_b200_match_host_begin(bicos_b200_handle h, const void* const* host_planes0,
                                const void* const* host_planes1, int n, int rows, int cols, int depth,
                                const bicos_b200_config* cfg, void* host_disparity, void* host_corrmap);
int bicos_b200_match_host_end(bicos_b200_handle h);

/* Row-sharded variant for one process driving several GPUs: rows [row_begin, row_end) of the
 * same device-resident inputs are matched on this handle's device and written into the
 * matching rows of the (possibly peer-mapped) output buffers. Rows are independent
 * (SURVEY.md 8e), so no halo and no collective is involved. */
int bicos_b200_match_rows(bicos_b200_handle h, const void* const* planes0,
                          const void* const* planes1, int n, int rows, int cols, size_t pitch_bytes,
                          int depth, const bicos_b200_config* cfg, int row_begin, int row_end,
                          void* disparity, size_t disparity_pitch_bytes, void* corrmap,
                          size_t corrmap_pitch_bytes, void* stream);

/* ---- peer-memory output assembly for a row-sharded match, one process per GPU -------------
 * Rows are independent, so the only exchange of a row-sharded match is the assembly of the
 * output rows on one GPU. Instead of a gather after the kernels, the assembling rank allocates
 * the output images with bicos_b200_shared_alloc and publishes the 64-byte handles (over any
 * channel: torch.distributed, MPI, a pipe); every other rank maps them once with
 * bicos_b200_shared_open and passes mapped + row_begin * pitch as the disparity / corrmap
 * pointer of bicos_b200_match on ITS rows. Its refine kernel then stores its rows straight
 * into the assembling GPU's memory over NVLink; after a stream synchronisation and a barrier
 * the result is complete. Inside one process, BICOS::match_sharded does the same with
 * cudaDeviceEnablePeerAccess. */
#define BICOS_B200_IPC_HANDLE_BYTES 64
int bicos_b200_shared_alloc(int device, size_t bytes, void** dev_ptr, void* handle_out);
int bicos_b200_shared_open(int device, const void* handle, void** dev_ptr);
int bicos_b200_shared_close(int device, void* dev_ptr); /* for pointers from _shared_open */
int bicos_b200_shared_free(int device, void* dev_ptr); /* for pointers from _shared_alloc */

/* Blocks until all work enqueued through this handle's internal streams and `stream` is done. */
int bicos_b200_synchronize(bicos_b200_handle h, void* stream);

/* Per-stage device timing for benchmarks: while enabled, every match records CUDA events
 * around its three stages (0 = both descriptor transforms, 1 = search, 2 = postfilter+refine)
 * on the stream it runs on. bicos_b200_stage_times() waits for the device, then returns the
 * accumulated milliseconds per stage and the number of matches they cover. */
int bicos_b200_set_profiling(bicos_b200_handle h, int enabled);
int bicos_b200_stage_times(bicos_b200_handle h, double* ms_out3, long long* matches_out);

/* How many kernels of this library have been launched through the handle (bench bookkeeping). */
long long bicos_b200_kernel_launches(bicos_b200_handle h);

/* The search stage has two engines with identical results: BICOS_B200_SEARCH_TENSOR computes the
 * row's Hamming matrix as an int8 GEMM on the tensor cores (tcgen05, accumulators in TMEM, argmin as
 * epilogue; descriptors of 4/8/12/16 words, rows of up to 8192 pixels), BICOS_B200_SEARCH_POPC is the
 * XOR + POPC kernel on the integer pipes (any descriptor, rows of up to 32767 pixels). AUTO (the
 * default, also settable as environment BICOS_B200_SEARCH_ENGINE = auto | popc | mma) takes the
 * tensor-core engine wherever it applies. Process-wide; forcing TENSOR makes unsupported shapes
 * fail with BICOS_B200_ERR_CUDA instead of falling back. */
enum { BICOS_B200_SEARCH_AUTO = 0, BICOS_B200_SEARCH_POPC = 1, BICOS_B200_SEARCH_TENSOR = 2 };
int bicos_b200_set_search_engine(int engine);
int bicos_b200_get_search_engine(void);

/* Name of the kernel the calling thread's last search dispatched, e.g. "mma2<K=4,nodupes=0,ct=1,dirs=2>",
 * "mma1<...>", "popc<K=4,flags=2>", with a disparity range "range<K=4,flags=2>" and with window maps "windows<K=4,flags=2>"; "" before the first search. For tests and benchmarks that must know
 * which of the engine's kernels they exercised. The string is thread-local and valid until the next search. */
const char* bicos_b200_last_search_kernel(void);

#ifdef __cplusplus
}
#endif
#endif /* BICOS_B200_H */
