// Internal launch interface between the C-ABI layer (cabi.cu) and the three sm_100a
// kernels of the BICOS::match hot path. Device pointers only; every function enqueues
// on `stream` and returns the CUDA status of the launch.
//
// Data layout in HBM (see DESIGN.md):
//   input stacks   n planar single-channel images per side, each [rows][pitch] bytes,
//                  passed as a by-value table of plane pointers (no host-mapped tables)
//   descriptors    [rows][desc_pitch_words] uint32, K = 1/2/4/8 words per pixel,
//                  bit i of a descriptor = bit i%32 of word i/32; rows start 16 B aligned
//   search result  four [rows][cols] uint32 key arrays, all minima of cost<<16 | column:
//                  fwd_first (cost<<16 | col1) / fwd_last (cost<<16 | 65535-col1): per left
//                  pixel, first and last right column attaining the minimal cost;
//                  rev_first (cost<<16 | col0) / rev_last (cost<<16 | 65535-col0): the same per
//                  right column over the left row, for the consistency check
//   outputs        disparity int16 or float32, corrmap float32 or float64, both pitched
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace bicos_b200 {

constexpr int MAX_IMAGES = 65; // 4n-6 <= 256 bits (reference src/impl/cuda.cu:107 "Bad number of images")
constexpr int FLAG_NODUPES = 1; // reference include/impl/common.hpp:46
constexpr int FLAG_CONSISTENCY = 2; // reference include/impl/common.hpp:47
constexpr uint32_t KEY_NONE = 0xFFFFFFFFu;

struct PlaneTable {
    const void* p[MAX_IMAGES];
};

struct RefineParams {
    int n, rows, cols;
    size_t in_pitch; // bytes, same for every plane of both stacks
    int is_u16;
    int is_double;
    int consistency; // postfilter: left-right check against rev_first / rev_last
    int nodupes_reverse; // consistency with no_dupes: reverse search must be unique too
    int max_lr_diff;
    int has_threshold;
    float threshold;
    int has_minvar;
    float minvar_times_n; // min_variance * n, in float (reference src/impl/cpu.cpp:127)
    int subpixel;
    int nsteps; // number of x values of the float loop x=-1; x<=1; x+=step
    const float* xs; // device array [nsteps] with exactly those float values
    float one; // 1.0f, passed at run time so that ptxas cannot fold x * one (refine.cu, fma2 note)
    float inv_n; // RN(1 / n) in float: the float means are sum / n as three FMA-pipe operations (refine.cu, mean_of_sum)
    int nodupes_forward; // forward search must be unique: compare fwd_first with fwd_last
    const uint32_t* fwd_first;
    const uint32_t* fwd_last;
    const uint32_t* rev_first;
    const uint32_t* rev_last;
    int16_t* raw_out; // optional [rows][cols] dense: postfilter result before the NXC test
    void* disp_out; // int16 if !has_threshold else float32
    size_t disp_pitch; // bytes
    void* corr_out; // float32 or float64, may be null
    size_t corr_pitch; // bytes
};

// kernel 1: temporal descriptor transform (reference a2/a3/a4)
cudaError_t launch_transform(
    const PlaneTable& planes,
    int n,
    int rows,
    int cols,
    size_t in_pitch,
    int is_u16,
    int mode_full,
    int K,
    uint32_t* desc,
    size_t desc_pitch_words,
    cudaStream_t stream
);

// kernel 2: row-wise Hamming argmin, forward (per left pixel) and, with
// FLAG_CONSISTENCY, the column-wise minima of the same W x W cost tile (reference a5/a6/a7).
// Key arrays in use must be pre-filled with KEY_NONE by the caller when search_needs_prefill()
// says so (fwd_last / rev_last are only touched with FLAG_NODUPES, rev_* only with FLAG_CONSISTENCY).
cudaError_t launch_search(
    const uint32_t* desc0,
    const uint32_t* desc1,
    int K,
    int rows,
    int cols,
    size_t desc_pitch_words,
    int flags,
    uint32_t* fwd_first,
    uint32_t* fwd_last,
    uint32_t* rev_first,
    uint32_t* rev_last,
    cudaStream_t stream,
    int free_top_bits = 0
);

// The two engines behind launch_search. `popc` (search.cu): XOR + POPC on the integer pipes, any
// K and width. `mma` (search_mma.cu): the row's Hamming matrix as an int8 GEMM on the tensor
// cores (tcgen05, TMEM accumulators) with the argmin as epilogue; K = 4/8/12/16 and rows of up
// to 8192 pixels. Identical key arrays. launch_search picks by search_engine():
// 0 = auto (mma where supported), 1 = popc, 2 = mma (error where unsupported).
cudaError_t launch_search_popc(
    const uint32_t* desc0,
    const uint32_t* desc1,
    int K,
    int rows,
    int cols,
    size_t desc_pitch_words,
    int flags,
    uint32_t* fwd_first,
    uint32_t* fwd_last,
    uint32_t* rev_first,
    uint32_t* rev_last,
    cudaStream_t stream
);
cudaError_t launch_search_mma(
    const uint32_t* desc0,
    const uint32_t* desc1,
    int K,
    int rows,
    int cols,
    size_t desc_pitch_words,
    int flags,
    uint32_t* fwd_first,
    uint32_t* fwd_last,
    uint32_t* rev_first,
    uint32_t* rev_last,
    cudaStream_t stream,
    int free_top_bits = 0 // how many of the top bits (32 K - 1, 32 K - 2) are zero in every descriptor: the transform's
                          // output has 2 (4n-6 <= 32K-2; n^2-2n+3 mod 32 <= 27); 1 enables the column-term kernels, 2 the
                          // one-pass consistency kernel as well
);
bool search_mma_colterm(); // see search_mma.cu, fold32
void set_search_mma_colterm(bool on);
bool search_mma_supports(int K, int cols);
bool search_mma_onepass_applies(int K, int cols, int flags, int free_top_bits); // would launch_search_mma take search_mma3_kernel?
int search_mma_smem_bytes(int K);
int search_mma_variant(); // tensor-core kernel variant, see search_mma.cu
void set_search_mma_variant(int v);
int search_engine(); // initial value: environment BICOS_B200_SEARCH_ENGINE = auto | popc | mma
void set_search_engine(int engine);
// Which kernel the calling thread's last launch_search dispatched, e.g. "mma2<K=4,nodupes=0,ct=1,dirs=2>" or
// "popc<K=4,flags=2>" ("" before the first search): lets tests assert that the kernel they mean to cover ran.
bool search_needs_prefill(int K, int cols); // must the caller fill the key arrays with KEY_NONE? (popcount engine only)
const char* last_search_kernel();
void note_search_kernel(const char* fmt, ...);
// Nonzero once if a wait inside a tensor-core search kernel timed out (pipeline bug, or a device stalled for
// longer than BICOS_B200_MMA_TIMEOUT_MS, default 10 s): its keys are garbage. Clears the flag.
unsigned int search_mma_take_timeout();

// kernel 2, windowed (search_range.cu): the same search over the pairs (left i, right j) with
// dmin <= i - j <= dmax only (Config::disparity_range; the range is clipped to [-cols, cols] here,
// which selects the same pairs). Integer pipes, K = 1/2/4/8/12/16, rows of up to 32767 pixels, the key format of
// launch_search. rev_first / rev_last (in use with FLAG_CONSISTENCY) must be pre-filled with
// KEY_NONE by the caller; fwd_first and fwd_last are stored for every pixel.
// Contract with the refine, which cannot tell that a window was empty (a left pixel with
// i - dmin < 0 or i - dmax > cols - 1): fwd_last is ALWAYS written and required, with FLAG_NODUPES
// as the real last-minimum key, otherwise as the mirror cost << 16 | (65535 - best) of fwd_first;
// an empty window gets KEY_NONE in both. The refine must therefore run with nodupes_forward = 1 on
// these keys: its first / last comparison rejects exactly the empty windows before it reads anything
// else (rev_first of column 65535 in particular).
cudaError_t launch_search_range(
    const uint32_t* desc0,
    const uint32_t* desc1,
    int K,
    int rows,
    int cols,
    size_t desc_pitch_words,
    int flags,
    int dmin,
    int dmax,
    uint32_t* fwd_first,
    uint32_t* fwd_last,
    uint32_t* rev_first,
    uint32_t* rev_last,
    cudaStream_t stream
);
// The same kernel over per-pixel windows (bicos_b200_search_windows): left pixel (r, i) pairs with right column j iff
// wmin[r][i] <= i - j <= wmax[r][i], wmin / wmax int16 [rows][wpitch elements], advanced to the first row. Same key
// contract as launch_search_range (fwd_last always written, rev_* pre-filled by the caller, KEY_NONE in both forward
// arrays for an empty window, refine with nodupes_forward = 1).
cudaError_t launch_search_windows(
    const uint32_t* desc0,
    const uint32_t* desc1,
    int K,
    int rows,
    int cols,
    size_t desc_pitch_words,
    int flags,
    const int16_t* wmin,
    const int16_t* wmax,
    size_t wpitch,
    uint32_t* fwd_first,
    uint32_t* fwd_last,
    uint32_t* rev_first,
    uint32_t* rev_last,
    cudaStream_t stream
);
// Clips [*dmin, *dmax] to [-cols, cols] in place (i - j lies in [-(cols-1), cols-1], so the pairs stay the
// same); false when the range covers every pair of the row, i.e. means exactly "no range" and the full-row
// search applies.
bool disparity_range_clip(int cols, int* dmin, int* dmax);

// kernel 3: postfilter (no-duplicates / left-right consistency) fused with the NXC
// agree / agree_subpixel refinement (reference a7 tail, a8, a9, a10, a11)
cudaError_t launch_refine(
    const PlaneTable& stack0,
    const PlaneTable& stack1,
    const RefineParams& prm,
    cudaStream_t stream
);

int search_smem_bytes(int K, int cols, int flags);

// stage 0 (remap.cu): rectification of n planes per side through one map pair per side, with the semantics of
// cv::remap(INTER_LINEAR, BORDER_CONSTANT 0) on float32 maps (bicos_b200_remap). Output [rows][cols], source
// [src_rows][src_cols], both at most 32767; maps are float32 [rows][map_pitch bytes].
struct RemapSide {
    PlaneTable src;
    PlaneTable dst; // written, despite PlaneTable's const
    const float* map_x;
    const float* map_y;
};

struct RemapParams {
    RemapSide side[2];
    int n, src_rows, src_cols, rows, cols;
    size_t src_pitch, map_pitch, dst_pitch; // bytes
};

// `sides` = 1 or 2: blockIdx.z picks prm.side[z], so both stacks of a match are one launch
cudaError_t launch_remap(const RemapParams& prm, int sides, int is_u16, cudaStream_t stream);

// stage 4 (reproject.cu): disparity -> 3D points through Q with the arithmetic bicos_b200_reproject states. One
// launch writes the dense map `xyz` and / or the ordered point list (`points`, `pixel_index`) with `counts`.
// The list and the counters need `work` and `status` zeroed before the launch (one cudaMemsetAsync of
// sizeof(ReprojectWork) + reproject_tiles() status words); a dense map alone runs without them.
struct ReprojectWork {
    unsigned int ticket; // next tile to hand out
    unsigned int done; // CTAs that have added their counters
    unsigned long long count[4]; // kept, invalid disparity, non-finite, negative Z
};

struct ReprojectParams {
    const void* disparity; // int16 or float32 [rows][disparity_pitch bytes]
    size_t disparity_pitch;
    int rows, cols; // 1 .. 32767
    double q[16]; // row-major
    int allow_negative_z;
    float* xyz; // [rows][xyz_pitch bytes], 3 floats per pixel; may be null
    size_t xyz_pitch;
    float* points; // [rows * cols][3]; may be null
    int32_t* pixel_index; // [rows * cols]; may be null
    unsigned long long* counts; // [4]; required with points
    ReprojectWork* work; // required with points or counts
    unsigned long long* status; // [reproject_tiles()] look-back status words, after `work`
};

int reproject_tiles(int rows, int cols);
cudaError_t launch_reproject(const ReprojectParams& prm, int is_float, cudaStream_t stream);

// speckle removal (speckles.cu): in place on an int16 or float32 disparity with the semantics
// bicos_b200_filter_speckles states. Four launches on every input (tile labelling, border merge, flatten and size,
// write); `parent` and `size` are rows * cols int32 each and need no initialisation, `counts` ([2]: pixels set,
// speckles removed) is added to and must be zeroed before the launch.
struct SpeckleParams {
    void* disparity; // int16 or float32 [rows][disparity_pitch bytes], written in place
    size_t disparity_pitch;
    int rows, cols; // 1 .. 32767
    int new_i, diff_i; // int16: the converted new_value and max_diff
    float new_f, diff_f; // float32: the same
    int max_size; // components of at most this many members are speckles
    int* parent; // [rows * cols] union-find parents (pixel indices)
    int* size; // [rows * cols] component sizes, at the roots
    unsigned long long* counts; // [2] or null
};

cudaError_t launch_speckles(const SpeckleParams& prm, int is_float, cudaStream_t stream);

// disparity windows from a prior (windows.cu), with the semantics bicos_b200_windows_from_disparity states; one launch
struct WindowsParams {
    const void* prior; // int16 or float32 [rows][prior_pitch bytes]
    size_t prior_pitch;
    int rows, cols; // 1 .. 32767 columns, 1 .. 65535 rows
    int margin; // 0 .. 32767
    int fallback_min, fallback_max; // int16 values, for an invalid prior
    int16_t* min_out; // [rows][out_pitch elements]
    int16_t* max_out;
    size_t out_pitch;
};

cudaError_t launch_windows_from_disparity(const WindowsParams& p, int is_float, cudaStream_t stream);

} // namespace bicos_b200
