// Kernel 2, windowed: the Hamming argmin of search.cu restricted to a disparity range
// (Config::disparity_range). A pair (left column i, right column j) is in range iff
// dmin <= i - j <= dmax; the forward search of i runs over j in [i - dmax, i - dmin], the reverse
// search of right column j over i in [j + dmin, j + dmax], both clipped to the row. Work is
// W * D * H pairs (D = dmax - dmin + 1) instead of the full row's W * W * H.
//
// Shape: a CTA owns 128 left pixels of one row (one per thread) and stages the union of its warps'
// windows of right descriptors in shared memory (in chunks when D is large). Each warp walks only
// its own window [x_w - dmax, x_w + 31 - dmin], D + 31 columns for 32 lanes that need D each, with
// warp-uniform (broadcast) loads of the right descriptor. Only the first and last 31 columns of a
// warp's window hold pairs outside the range for some lane; the interior runs without the mask.
//
// Keys, trees and exactness as in search.cu (search_common.cuh): min(cost << 16 | column) over the
// in-range pairs is the first strict minimum of the window, cost << 16 | (65535 - column) the last.
// The reverse minima of a right column come from every CTA whose left pixels reach it: warps merge
// per CTA with REDUX + shared atomics, CTAs with global atomicMin into key arrays the caller has
// filled with KEY_NONE. Every left pixel belongs to one CTA, so the forward keys are plain stores
// and fwd_last is always written (the contract with the refine in kernels.cuh).
//
// Windows (MAPS, bicos_b200_search_windows): the bounds come per left pixel from two int16 maps instead of one range.
// Each lane clips its own window to the row and walks the same masked test with its own lo and span; the warp walks the
// union of its lanes' windows, unmasked over their intersection, and the CTA stages the union of its warps' windows.
// A lane with an empty window, or past the end of the row, gets lo = WIN_EMPTY_LO and span 0: j - lo is negative for
// every column j of the row, so the unsigned test fails everywhere.

#include "kernels.cuh"
#include "search_common.cuh"

#include <climits>

namespace bicos_b200 {
namespace {

constexpr int RT = 128; // threads per CTA = left pixels per CTA
constexpr int RANGE_CHUNK_BYTES = 16 * 1024; // right-row descriptor bytes staged per pass

struct RangeArgs {
    const uint32_t* desc0;
    const uint32_t* desc1;
    int cols;
    size_t pitch_words;
    int dmin, dmax; // clipped to [-cols, cols], dmin <= dmax
    int chunk; // right descriptors staged per pass, a multiple of 4 (16 B aligned staging for K = 1, 2)
    uint32_t one, two, shl16; // 1, 2 and 65536 as run-time values, see mad()
    uint32_t* fwd_first;
    uint32_t* fwd_last;
    uint32_t* rev_first;
    uint32_t* rev_last;
    const int16_t* wmin; // MAPS: [rows][wpitch] per-pixel bounds of i - j, advanced to the unit's first row
    const int16_t* wmax;
    size_t wpitch; // elements
};

constexpr int WIN_EMPTY_LO = 0x40000000; // see the header comment: fails (uint32_t)(j - lo) <= 0 for every j of a row

template<int K>
__device__ __forceinline__ uint32_t make_key(uint32_t h, uint32_t col, const Weights w) {
    if constexpr (K >= 8)
        return mad(h, w.shl16, col); // ALU-pipe bound widths: the key on the FMA pipe, as in search.cu
    else
        return (h << 16) + col;
}

// Columns [ja, jb) of the staged chunk that starts at column c0, against the warp's 32 left pixels.
// MASKED: pairs outside the range become KEY_NONE; lane i is in range of column j iff
// 0 <= j - (i - dmax) <= dmax - dmin.
template<int K, int FLAGS, bool MASKED>
__device__ __forceinline__ void walk(
    const uint32_t* s_right,
    int c0,
    int ja,
    int jb,
    const Desc<K>& l,
    int lo, // i - dmax
    uint32_t span, // dmax - dmin
    uint32_t icol,
    uint32_t icol_rev,
    int lane,
    const Weights wts,
    uint32_t& mf,
    uint32_t& ml,
    uint32_t* s_colf,
    uint32_t* s_coll
) {
    constexpr bool NODUPES = (FLAGS & FLAG_NODUPES) != 0;
    constexpr bool REVERSE = (FLAGS & FLAG_CONSISTENCY) != 0;
    // groups of 32 columns: lane u keeps the warp's reverse minimum of column u of the group (search.cu)
    for (int g0 = ja; g0 < jb; g0 += 32) {
        const int m = min(32, jb - g0);
        uint32_t colf = KEY_NONE, coll = KEY_NONE;
#pragma unroll 4
        for (int u = 0; u < m; ++u) {
            const int j = g0 + u;
            const Desc<K> r = load_desc<K>(s_right + (size_t)(j - c0) * K); // warp-uniform: broadcast
            const uint32_t h = hamming<K>(l, r, false, wts);
            const bool in = !MASKED || (uint32_t)(j - lo) <= span;
            mf = min(mf, in ? make_key<K>(h, (uint32_t)j, wts) : KEY_NONE);
            if constexpr (NODUPES)
                ml = min(ml, in ? make_key<K>(h, 65535u - (uint32_t)j, wts) : KEY_NONE);
            if constexpr (REVERSE) {
                const uint32_t ck = __reduce_min_sync(0xFFFFFFFFu, in ? make_key<K>(h, icol, wts) : KEY_NONE);
                if (lane == u)
                    colf = ck;
                if constexpr (NODUPES) {
                    const uint32_t ckl = __reduce_min_sync(0xFFFFFFFFu, in ? make_key<K>(h, icol_rev, wts) : KEY_NONE);
                    if (lane == u)
                        coll = ckl;
                }
            }
        }
        if constexpr (REVERSE) {
            if (lane < m) {
                atomicMin(&s_colf[g0 - c0 + lane], colf);
                if constexpr (NODUPES)
                    atomicMin(&s_coll[g0 - c0 + lane], coll);
            }
        }
    }
}

// MAPS: the first and the last column of each warp's union of windows
__device__ __forceinline__ int* window_bounds() {
    __shared__ int s_win[2 * (RT / 32)];
    return s_win;
}

template<int K, int FLAGS, bool MAPS>
__global__ void __launch_bounds__(RT) search_range_kernel(const RangeArgs p) {
    constexpr bool NODUPES = (FLAGS & FLAG_NODUPES) != 0;
    constexpr bool REVERSE = (FLAGS & FLAG_CONSISTENCY) != 0;
    extern __shared__ uint4 smem_raw[];
    uint32_t* const s_right = reinterpret_cast<uint32_t*>(smem_raw);
    uint32_t* const s_colf = s_right + (size_t)p.chunk * K;
    uint32_t* const s_coll = s_colf + p.chunk;

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int cols = p.cols;
    const int row = blockIdx.y;
    const int x0 = blockIdx.x * RT;
    const int i = x0 + tid;
    const bool valid = i < cols;
    const Weights wts = { p.one, p.two, p.shl16 };

    const uint32_t* const row0 = p.desc0 + (size_t)row * p.pitch_words;
    const uint32_t* const row1 = p.desc1 + (size_t)row * p.pitch_words;
    const Desc<K> l = load_desc<K>(row0 + (size_t)(valid ? i : cols - 1) * K);
    // lanes past the end of the row carry bit 31 so that they never win a column minimum (search.cu)
    const uint32_t icol = valid ? (uint32_t)i : (0x80000000u | (uint32_t)i);
    const uint32_t icol_rev = valid ? (uint32_t)(65535 - i) : (0x80000000u | (uint32_t)i);
    uint32_t mf = KEY_NONE, ml = KEY_NONE;

    // the warp's pixels [xw, xe] and window [wlo, whi]; interior [ilo, ihi]: every valid lane in range
    const int xw = x0 + (tid & ~31);
    const int xe = min(xw + 31, cols - 1);
    int wlo = max(0, xw - p.dmax), whi = min(cols - 1, xe - p.dmin);
    int ilo = xe - p.dmax, ihi = xw - p.dmin;
    uint32_t span = (uint32_t)(p.dmax - p.dmin);
    // the CTA's window: the union of its warps' windows (they overlap or touch), start 16 B aligned
    int clo = max(0, x0 - p.dmax) & ~3;
    int chi = min(cols - 1, min(x0 + RT, cols) - 1 - p.dmin);
    int lo = 0; // MAPS: this lane's first right column (the range passes i - dmax)
    if constexpr (MAPS) {
        int* const s_win = window_bounds();
        // this lane's right columns [i - max, i - min], clipped to the row (int16 bounds: no overflow)
        int a = cols, b = -1;
        if (valid) {
            const size_t at = (size_t)row * p.wpitch + i;
            a = max(0, i - (int)p.wmax[at]);
            b = min(cols - 1, i - (int)p.wmin[at]);
        }
        const bool empty = a > b; // also every lane past the end of the row
        lo = empty ? WIN_EMPTY_LO : a;
        span = empty ? 0u : (uint32_t)(b - a);
        // union over all lanes; intersection over the lanes in the row (an empty one empties it): past-the-end lanes
        // carry bit 31 in their reverse keys and store nothing, so they may run unmasked (search.cu)
        wlo = __reduce_min_sync(0xFFFFFFFFu, empty ? INT_MAX : a);
        whi = __reduce_max_sync(0xFFFFFFFFu, empty ? -1 : b);
        ilo = __reduce_max_sync(0xFFFFFFFFu, !valid ? INT_MIN : empty ? INT_MAX : a);
        ihi = __reduce_min_sync(0xFFFFFFFFu, !valid ? INT_MAX : empty ? -1 : b);
        if (lane == 0) {
            s_win[tid >> 5] = wlo;
            s_win[(tid >> 5) + RT / 32] = whi;
        }
        __syncthreads();
        clo = INT_MAX;
        chi = -1;
#pragma unroll
        for (int w = 0; w < RT / 32; ++w) {
            clo = min(clo, s_win[w]);
            chi = max(chi, s_win[w + RT / 32]);
        }
        clo &= ~3; // every pixel of the CTA empty: clo = INT_MAX & ~3 > chi = -1 skips the staging
    }

    for (int c0 = clo; c0 <= chi; c0 += p.chunk) {
        const int cnt = min(p.chunk, chi + 1 - c0);
        __syncthreads(); // previous chunk fully consumed and flushed
        {
            const uint4* src = reinterpret_cast<const uint4*>(row1 + (size_t)c0 * K);
            const int nvec = (cnt * K + 3) / 4;
            for (int v = tid; v < nvec; v += RT)
                smem_raw[v] = src[v];
            if constexpr (REVERSE) {
                for (int v = tid; v < cnt; v += RT) {
                    s_colf[v] = KEY_NONE;
                    if constexpr (NODUPES)
                        s_coll[v] = KEY_NONE;
                }
            }
        }
        __syncthreads();

        if (xw < cols) { // warp-uniform; an all-empty warp of a window map has wlo > whi and walks nothing
            const int a = max(wlo, c0), b = min(whi + 1, c0 + cnt);
            if (a < b) {
                const int ia = min(max(ilo, a), b), ib = min(max(ihi + 1, ia), b);
                walk<K, FLAGS, true>(s_right, c0, a, ia, l, MAPS ? lo : i - p.dmax, span, icol, icol_rev, lane, wts, mf, ml, s_colf, s_coll);
                walk<K, FLAGS, false>(s_right, c0, ia, ib, l, MAPS ? lo : i - p.dmax, span, icol, icol_rev, lane, wts, mf, ml, s_colf, s_coll);
                walk<K, FLAGS, true>(s_right, c0, ib, b, l, MAPS ? lo : i - p.dmax, span, icol, icol_rev, lane, wts, mf, ml, s_colf, s_coll);
            }
        }

        if constexpr (REVERSE) {
            __syncthreads();
            uint32_t* const gf = p.rev_first + (size_t)row * cols + c0;
            uint32_t* const gl = p.rev_last + (size_t)row * cols + c0;
            for (int v = tid; v < cnt; v += RT) {
                if (s_colf[v] != KEY_NONE)
                    atomicMin(gf + v, s_colf[v]);
                if constexpr (NODUPES)
                    if (s_coll[v] != KEY_NONE)
                        atomicMin(gl + v, s_coll[v]);
            }
        }
    }

    if (valid) {
        const size_t at = (size_t)row * cols + i;
        p.fwd_first[at] = mf;
        // without NODUPES the mirror of fwd_first, so that the refine's first / last comparison passes every
        // non-empty window and rejects the empty ones (KEY_NONE in both)
        if constexpr (NODUPES)
            p.fwd_last[at] = ml;
        else
            p.fwd_last[at] = mf == KEY_NONE ? KEY_NONE : (mf & 0xFFFF0000u) | (65535u - (mf & 0xFFFFu));
    }
}

int range_chunk(int K, int dmin, int dmax) {
    const long long window = ((long long)RT + (dmax - dmin) + 3 + 3) & ~3LL; // CTA window plus alignment slack
    const int cap = (RANGE_CHUNK_BYTES / (4 * K)) & ~3;
    return window < cap ? (int)window : cap;
}

int range_smem_bytes(int K, int chunk, int flags) {
    int bytes = chunk * K * 4;
    if (flags & FLAG_CONSISTENCY)
        bytes += chunk * 4 * ((flags & FLAG_NODUPES) ? 2 : 1);
    return bytes;
}

template<int K, int FLAGS, bool MAPS>
cudaError_t launch_one(const RangeArgs& p, int rows, cudaStream_t stream) {
    const int smem = range_smem_bytes(K, p.chunk, FLAGS);
    auto kernel = search_range_kernel<K, FLAGS, MAPS>;
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess)
        return err;
    const dim3 grid((unsigned)((p.cols + RT - 1) / RT), (unsigned)rows);
    kernel<<<grid, RT, smem, stream>>>(p);
    return cudaGetLastError();
}

template<int K, bool MAPS>
cudaError_t launch_k(const RangeArgs& p, int rows, int flags, cudaStream_t stream) {
    switch (flags) {
        case FLAG_NODUPES:
            return launch_one<K, FLAG_NODUPES, MAPS>(p, rows, stream);
        case FLAG_CONSISTENCY:
            return launch_one<K, FLAG_CONSISTENCY, MAPS>(p, rows, stream);
        case FLAG_NODUPES | FLAG_CONSISTENCY:
            return launch_one<K, FLAG_NODUPES | FLAG_CONSISTENCY, MAPS>(p, rows, stream);
        case 0:
            return launch_one<K, 0, MAPS>(p, rows, stream);
    }
    return cudaErrorInvalidValue;
}

template<bool MAPS>
cudaError_t launch_args(RangeArgs& p, int K, int rows, int flags, cudaStream_t stream) {
    p.one = 1u;
    p.two = 2u;
    p.shl16 = 65536u;
    switch (K) {
        case 1:
            return launch_k<1, MAPS>(p, rows, flags, stream);
        case 2:
            return launch_k<2, MAPS>(p, rows, flags, stream);
        case 4:
            return launch_k<4, MAPS>(p, rows, flags, stream);
        case 8:
            return launch_k<8, MAPS>(p, rows, flags, stream);
        case 12:
            return launch_k<12, MAPS>(p, rows, flags, stream);
        case 16:
            return launch_k<16, MAPS>(p, rows, flags, stream);
    }
    return cudaErrorInvalidValue;
}

} // namespace

bool disparity_range_clip(int cols, int* dmin, int* dmax) {
    // i - j lies in [-(cols - 1), cols - 1]: clipping to +-cols selects the same pairs, an empty range included
    *dmin = *dmin < -cols ? -cols : *dmin > cols ? cols : *dmin;
    *dmax = *dmax < -cols ? -cols : *dmax > cols ? cols : *dmax;
    return !(*dmin <= -(cols - 1) && *dmax >= cols - 1);
}

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
) {
    if (rows <= 0 || rows > 65535 || cols <= 0 || cols > 32767 || dmin > dmax || !fwd_last)
        return cudaErrorInvalidValue;
    disparity_range_clip(cols, &dmin, &dmax);
    note_search_kernel("range<K=%d,flags=%d>", K, flags);
    RangeArgs p {};
    p.desc0 = desc0;
    p.desc1 = desc1;
    p.cols = cols;
    p.pitch_words = desc_pitch_words;
    p.dmin = dmin;
    p.dmax = dmax;
    p.chunk = range_chunk(K, dmin, dmax);
    p.fwd_first = fwd_first;
    p.fwd_last = fwd_last;
    p.rev_first = rev_first;
    p.rev_last = rev_last;
    return launch_args<false>(p, K, rows, flags, stream);
}

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
) {
    if (rows <= 0 || rows > 65535 || cols <= 0 || cols > 32767 || !wmin || !wmax || wpitch < (size_t)cols || !fwd_last)
        return cudaErrorInvalidValue;
    note_search_kernel("windows<K=%d,flags=%d>", K, flags);
    RangeArgs p {};
    p.desc0 = desc0;
    p.desc1 = desc1;
    p.cols = cols;
    p.pitch_words = desc_pitch_words;
    // a CTA stages at most the whole row; the windows are only known on the device, so the chunk is the cap
    const int cap = (RANGE_CHUNK_BYTES / (4 * K)) & ~3;
    const int row4 = (cols + 3) & ~3;
    p.chunk = row4 < cap ? row4 : cap;
    p.fwd_first = fwd_first;
    p.fwd_last = fwd_last;
    p.rev_first = rev_first;
    p.rev_last = rev_last;
    p.wmin = wmin;
    p.wmax = wmax;
    p.wpitch = wpitch;
    return launch_args<true>(p, K, rows, flags, stream);
}

} // namespace bicos_b200
