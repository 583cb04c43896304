// Reprojection stage after the match: disparity -> 3D points through a 4x4 matrix Q (what cv::stereoRectify
// returns), with the arithmetic of bicos-cli's former host loop, bit for bit (DESIGN.md §3.8; include/bicos_b200.h
// states it, tests/test_reproject.py restates it in numpy):
//   skip the invalid disparities (int16 -32768; float32 NaN or -32768.0f)
//   in = (c, r, d, 1.0) in double; o[k] = ((Q[4k] in0 + Q[4k+1] in1) + Q[4k+2] in2) + Q[4k+3] in3, every product
//   and sum rounded to double on its own (no FMA contraction: it changes the float32 result on constructed inputs)
//   X = (float)(o0 / o3), Y, Z likewise (IEEE division, round to nearest even, subnormals kept)
//   skip non-finite X / Y / Z, then Z < 0 unless allow_negative_z; keep the rest
//
// One launch writes the dense map (NaN NaN NaN where skipped), the ordered point list, or both. The list is a
// stream compaction in row-major pixel order done in one pass with a decoupled look-back scan: each CTA takes a
// tile of TILE consecutive pixel indices (tiles ignore row boundaries), numbered by an atomic ticket so that every
// tile a CTA waits on has already started, publishes its kept count as one 64-bit status word (flag | value),
// then sums its predecessors' words 32 at a time with one warp until it meets an inclusive prefix, and publishes
// its own. The four counters (kept, invalid, non-finite, negative Z) are block-reduced and added atomically into
// the workspace; the CTA that finishes last copies them to the caller's `counts`. The workspace is zeroed by one
// cudaMemsetAsync per call (cabi.cu).

#include "kernels.cuh"

namespace bicos_b200 {
namespace {

constexpr int THREADS = 256;
constexpr int ITEMS = 8; // pixels per thread: item k of thread t is pixel tile * TILE + k * THREADS + t
constexpr int TILE = THREADS * ITEMS;
constexpr int WARPS = THREADS / 32;
constexpr int CHUNKS = TILE / 32; // 32-pixel chunks of a tile, in pixel order: chunk k * WARPS + warp

constexpr unsigned long long FLAG_AGGREGATE = 1ull << 62; // status word: the tile's own kept count
constexpr unsigned long long FLAG_PREFIX = 2ull << 62; // status word: kept count of tiles 0..tile, inclusive
constexpr unsigned long long VALUE_MASK = (1ull << 62) - 1;

enum { KEPT = 0, INVALID = 1, NON_FINITE = 2, NEGATIVE_Z = 3 };

// ((q0 in0 + q1 in1) + q2 in2) + q3 * 1.0 for row k of Q, each operation rounded on its own
__device__ __forceinline__ double row_of_q(const ReprojectParams& prm, int k, double in0, double in1, double in2) {
    double s = __dadd_rn(__dmul_rn(prm.q[4 * k], in0), __dmul_rn(prm.q[4 * k + 1], in1));
    s = __dadd_rn(s, __dmul_rn(prm.q[4 * k + 2], in2));
    return __dadd_rn(s, __dmul_rn(prm.q[4 * k + 3], 1.0));
}

template<typename T>
__device__ __forceinline__ bool load_disparity(const ReprojectParams& prm, int r, int c, double& d) {
    const T v = __ldg(reinterpret_cast<const T*>(static_cast<const char*>(prm.disparity) + (size_t)r * prm.disparity_pitch) + c);
    if constexpr (sizeof(T) == 2) {
        d = (double)v;
        return v != (T)-32768;
    } else {
        d = (double)v;
        return !(v != v) && v != -32768.0f;
    }
}

__device__ __forceinline__ unsigned long long load_status(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void store_status(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Warp 0: the number of points kept by tiles 0 .. tile - 1. Predecessors publish FLAG_AGGREGATE before they look
// back themselves, and every one of them holds an SM (their tickets are older), so the wait ends.
__device__ unsigned long long look_back(unsigned long long* status, int tile, int lane) {
    unsigned long long exclusive = 0;
    for (int base = tile - 1;; base -= 32) {
        const int idx = base - lane;
        unsigned long long s = FLAG_PREFIX; // before tile 0: an empty prefix
        for (;;) {
            if (idx >= 0)
                s = load_status(status + idx);
            if (!__any_sync(0xffffffffu, (s >> 62) == 0))
                break;
            __nanosleep(32);
        }
        const unsigned prefix_lanes = __ballot_sync(0xffffffffu, (s & ~VALUE_MASK) == FLAG_PREFIX);
        const int stop = prefix_lanes ? __ffs(prefix_lanes) - 1 : 31; // the nearest inclusive prefix ends the walk
        unsigned long long v = lane <= stop ? (s & VALUE_MASK) : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
            v += __shfl_xor_sync(0xffffffffu, v, o);
        exclusive += v;
        if (prefix_lanes)
            return exclusive;
    }
}

template<typename T, bool DENSE, bool LIST>
__global__ void __launch_bounds__(THREADS) reproject_kernel(const ReprojectParams prm) {
    __shared__ unsigned s_mask[CHUNKS]; // ballot of kept pixels per 32-pixel chunk
    __shared__ unsigned s_chunk_offset[CHUNKS]; // kept pixels of the tile before each chunk
    __shared__ unsigned s_count[WARPS][4];
    __shared__ unsigned long long s_tile_offset;
    __shared__ int s_tile;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int total = prm.rows * prm.cols; // < 2^30: rows and cols are at most 32767
    int tile = blockIdx.x;
    if (prm.work) {
        if (tid == 0)
            s_tile = (int)atomicAdd(&prm.work->ticket, 1u);
        __syncthreads();
        tile = s_tile;
    }

    unsigned count[4] = { 0, 0, 0, 0 };
    float X[ITEMS], Y[ITEMS], Z[ITEMS];
    bool kept[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const int p = tile * TILE + k * THREADS + tid;
        kept[k] = false;
        X[k] = Y[k] = Z[k] = __int_as_float(0x7fffffff);
        if (p >= total)
            continue;
        const int r = (int)((unsigned)p / (unsigned)prm.cols), c = p - r * prm.cols;
        double d;
        if (!load_disparity<T>(prm, r, c, d)) {
            count[INVALID] += 1;
        } else {
            const double in0 = (double)c, in1 = (double)r;
            const double o0 = row_of_q(prm, 0, in0, in1, d), o1 = row_of_q(prm, 1, in0, in1, d);
            const double o2 = row_of_q(prm, 2, in0, in1, d), o3 = row_of_q(prm, 3, in0, in1, d);
            const float x = __double2float_rn(__ddiv_rn(o0, o3));
            const float y = __double2float_rn(__ddiv_rn(o1, o3));
            const float z = __double2float_rn(__ddiv_rn(o2, o3));
            if (!isfinite(x) || !isfinite(y) || !isfinite(z)) {
                count[NON_FINITE] += 1;
            } else if (!prm.allow_negative_z && z < 0.0f) {
                count[NEGATIVE_Z] += 1;
            } else {
                count[KEPT] += 1;
                kept[k] = true;
                X[k] = x;
                Y[k] = y;
                Z[k] = z;
            }
        }
        if constexpr (DENSE) {
            float* o = reinterpret_cast<float*>(reinterpret_cast<char*>(prm.xyz) + (size_t)r * prm.xyz_pitch) + 3 * (size_t)c;
            o[0] = X[k];
            o[1] = Y[k];
            o[2] = Z[k];
        }
    }

    if (!prm.work) // dense map alone: no list, no counters
        return;

    if constexpr (LIST) {
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const unsigned m = __ballot_sync(0xffffffffu, kept[k]);
            if (lane == 0)
                s_mask[k * WARPS + warp] = m;
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const unsigned v = __reduce_add_sync(0xffffffffu, count[j]);
        if (lane == 0)
            s_count[warp][j] = v;
    }
    __syncthreads();

    if constexpr (LIST) {
        if (warp == 0) {
            // exclusive scan of the CHUNKS (= 64) chunk counts, two consecutive chunks per lane
            static_assert(CHUNKS == 64, "two chunks per lane");
            const unsigned a = __popc(s_mask[2 * lane]), b = __popc(s_mask[2 * lane + 1]);
            unsigned incl = a + b;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o)
                    incl += t;
            }
            s_chunk_offset[2 * lane] = incl - a - b;
            s_chunk_offset[2 * lane + 1] = incl - b;
            const unsigned aggregate = __shfl_sync(0xffffffffu, incl, 31);
            unsigned long long* status = prm.status;
            unsigned long long offset = 0;
            if (tile == 0) {
                if (lane == 0)
                    store_status(status, FLAG_PREFIX | aggregate);
            } else {
                if (lane == 0)
                    store_status(status + tile, FLAG_AGGREGATE | aggregate);
                offset = look_back(status, tile, lane);
                if (lane == 0)
                    store_status(status + tile, FLAG_PREFIX | (offset + aggregate));
            }
            if (lane == 0)
                s_tile_offset = offset;
        }
        __syncthreads();
        const unsigned long long base = s_tile_offset;
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            if (!kept[k])
                continue;
            const int chunk = k * WARPS + warp;
            const unsigned long long i = base + s_chunk_offset[chunk] + __popc(s_mask[chunk] & ((1u << lane) - 1u));
            float* pt = prm.points + 3 * i;
            pt[0] = X[k];
            pt[1] = Y[k];
            pt[2] = Z[k];
            if (prm.pixel_index)
                prm.pixel_index[i] = tile * TILE + k * THREADS + tid;
        }
    }

    if (tid == 0) {
        ReprojectWork* w = prm.work;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            unsigned long long sum = 0;
            for (int q = 0; q < WARPS; ++q)
                sum += s_count[q][j];
            if (sum)
                atomicAdd(&w->count[j], sum);
        }
        __threadfence();
        if (atomicAdd(&w->done, 1u) == gridDim.x - 1) { // every other CTA has added its counts
            __threadfence();
#pragma unroll
            for (int j = 0; j < 4; ++j)
                prm.counts[j] = atomicAdd(&w->count[j], 0ull);
        }
    }
}

template<typename T>
cudaError_t launch_typed(const ReprojectParams& prm, unsigned grid, cudaStream_t stream) {
    const bool dense = prm.xyz != nullptr, list = prm.points != nullptr;
    if (dense && list)
        reproject_kernel<T, true, true><<<grid, THREADS, 0, stream>>>(prm);
    else if (dense)
        reproject_kernel<T, true, false><<<grid, THREADS, 0, stream>>>(prm);
    else
        reproject_kernel<T, false, true><<<grid, THREADS, 0, stream>>>(prm);
    return cudaGetLastError();
}

} // namespace

int reproject_tiles(int rows, int cols) {
    return (int)(((long long)rows * cols + TILE - 1) / TILE);
}

cudaError_t launch_reproject(const ReprojectParams& prm, int is_float, cudaStream_t stream) {
    if (prm.rows <= 0 || prm.cols <= 0 || prm.rows > 32767 || prm.cols > 32767 || (!prm.xyz && !prm.points) ||
        (prm.points && (!prm.work || !prm.counts)) || (prm.counts && !prm.work))
        return cudaErrorInvalidValue;
    const unsigned grid = (unsigned)reproject_tiles(prm.rows, prm.cols);
    return is_float ? launch_typed<float>(prm, grid, stream) : launch_typed<int16_t>(prm, grid, stream);
}

} // namespace bicos_b200
