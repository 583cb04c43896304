// Speckle removal after the match, in place (DESIGN.md §3.9; include/bicos_b200.h states the semantics,
// tests/test_speckles.py restates them with scipy's connected components and pins that to cv::filterSpeckles):
//   members: pixels that are not an invalid marker (int16 -32768; float32 NaN or -32768.0f) and not equal to `new`
//   edges: 4-neighbours that are both members with |d(p) - d(q)| <= diff (int16: in int32; float32: fabsf of the
//   difference rounded to nearest, so inf - inf gives no edge)
//   every pixel of a component with at most max_speckle_size members is set to `new`; nothing else is written
//
// A union-find connected-component labelling in four launches, the same four on every input:
//   1. tile pass: a CTA labels a TILE_W x TILE_H tile in shared memory: runs inside 32-pixel row segments from a
//      warp ballot, then union by index between them (the larger root hooked under the smaller with atomicCAS,
//      finds with path splitting); it writes every pixel's tile root as a global pixel index to `parent` and the
//      tile component's size at its root to `size` (0 for every other pixel)
//   2. border merge: one thread per 4-neighbour pair across a tile edge unions the two trees in global memory with
//      the same hooking; only tile roots are ever hooked, so every parent is a tile root and parent[p] <= p
//   3. flatten and size: each tile root (size > 0 after pass 1) finds its global root R, points straight at it and
//      adds its partial size to size[R] with one atomic: one atomic per tile component, not per pixel. The walk does
//      not split paths, so the only parent written in this pass is a final root
//   4. write: parent[parent[p]] is the root of every member p; p is set to `new` when size[root] <= max_speckle_size;
//      warp-aggregated counts of the pixels set and the roots (= speckles) removed
// The labels are the components of a graph, so the result does not depend on the order in which the unions ran.

#include "kernels.cuh"

namespace bicos_b200 {
namespace {

constexpr int TILE_W = 128; // wide in x: a warp loads 32 consecutive pixels of a row
constexpr int TILE_H = 16;
constexpr int TILE = TILE_W * TILE_H;
constexpr int THREADS = 256;
constexpr int ITEMS = TILE / THREADS; // item k of thread t is tile pixel k * THREADS + t
constexpr int FLAT_THREADS = 256; // passes 3 and 4: one thread per pixel, a row segment per CTA

template<typename T>
__device__ __forceinline__ T load_px(const SpeckleParams& prm, int r, int c) {
    return reinterpret_cast<const T*>(static_cast<const char*>(prm.disparity) + (size_t)r * prm.disparity_pitch)[c];
}

__device__ __forceinline__ bool is_member(int16_t v, const SpeckleParams& prm) {
    return v != (int16_t)-32768 && (int)v != prm.new_i;
}
__device__ __forceinline__ bool is_member(float v, const SpeckleParams& prm) {
    return !(v != v) && v != -32768.0f && v != prm.new_f;
}

__device__ __forceinline__ bool is_edge(int16_t a, int16_t b, const SpeckleParams& prm) {
    const int d = (int)a - (int)b;
    return (d < 0 ? -d : d) <= prm.diff_i;
}
__device__ __forceinline__ bool is_edge(float a, float b, const SpeckleParams& prm) {
    return fabsf(__fsub_rn(a, b)) <= prm.diff_f; // NaN (inf - inf) compares false
}

// root of x with path splitting (every node on the path is pointed at its grandparent). Only roots are hooked and a
// hooked root only moves up, so a stale read is still an ancestor: concurrent finds and hooks stay correct.
__device__ __forceinline__ int find_root(volatile int* parent, int x) {
    int cur = parent[x];
    if (cur != x) {
        int prev = x, next;
        while (cur > (next = parent[cur])) {
            parent[prev] = next;
            prev = cur;
            cur = next;
        }
    }
    return cur;
}

// the same walk without writes (pass 3, where every write must be a final root)
__device__ __forceinline__ int find_root_readonly(volatile int* parent, int x) {
    int next;
    while ((next = parent[x]) != x)
        x = next;
    return x;
}

// join the trees of a and b: hook the larger root under the smaller one, retrying where another thread hooked first
__device__ __forceinline__ void unite(volatile int* parent, int* parent_atomic, int a, int b) {
    a = find_root(parent, a);
    b = find_root(parent, b);
    while (a != b) {
        if (a < b) {
            const int t = a;
            a = b;
            b = t;
        }
        const int old = atomicCAS(parent_atomic + a, a, b);
        if (old == a)
            return;
        a = find_root(parent, old);
    }
}

// Pass 1. Each warp owns 32-pixel row segments (item k of warp w: row 2k + w / 4, columns 32 (w % 4) ..). Runs of
// connected pixels inside a segment come from one ballot and need no union: every member starts with its run's
// first pixel as parent. Unions are left for the joins between segments of a row and between rows, and a vertical
// join is skipped where the left neighbours already make it (p ~ p - 1 ~ p - 1 - W ~ p - W inside the segments).
template<typename T>
__global__ void __launch_bounds__(THREADS) speckle_tile_kernel(const SpeckleParams prm) {
    __shared__ T s_val[TILE];
    __shared__ int s_lab[TILE]; // tile-local parent, -1 for non-members and pixels outside the image
    __shared__ int s_run[TILE]; // first pixel of the run inside the segment (-1 for non-members), then component sizes

    const int tid = threadIdx.x, lane = tid & 31;
    const unsigned below = (1u << lane) - 1u; // lanes before this one
    const int r0 = blockIdx.y * TILE_H, c0 = blockIdx.x * TILE_W;
    T v[ITEMS];
    bool member[ITEMS];
    unsigned starts[ITEMS], members[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const int i = k * THREADS + tid;
        const int r = r0 + i / TILE_W, c = c0 + i % TILE_W;
        member[k] = false;
        v[k] = T(0);
        if (r < prm.rows && c < prm.cols) {
            v[k] = load_px<T>(prm, r, c);
            member[k] = is_member(v[k], prm);
        }
        const T left = __shfl_up_sync(0xffffffffu, v[k], 1);
        const bool left_member = __shfl_up_sync(0xffffffffu, member[k], 1);
        const bool link = lane > 0 && member[k] && left_member && is_edge(v[k], left, prm);
        members[k] = __ballot_sync(0xffffffffu, member[k]);
        starts[k] = __ballot_sync(0xffffffffu, member[k] && !link);
        const int run = member[k] ? i - lane + 31 - __clz(starts[k] & (below | (1u << lane))) : -1;
        s_val[i] = v[k];
        s_lab[i] = run;
        s_run[i] = run;
    }
    __syncthreads();

    volatile int* lab = s_lab;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const int i = k * THREADS + tid;
        if (member[k] && lane == 0 && i % TILE_W > 0 && s_run[i - 1] >= 0 && is_edge(v[k], s_val[i - 1], prm))
            unite(lab, s_lab, i, i - 1);
        // i - W and i - W - 1 in one run, i and i - 1 in one run, and i - 1 joined to i - 1 - W: already connected
        const bool up = member[k] && i >= TILE_W && s_run[i - TILE_W] >= 0 && is_edge(v[k], s_val[i - TILE_W], prm);
        const bool up_left = __shfl_up_sync(0xffffffffu, up, 1);
        const bool implied = lane > 0 && up_left && s_run[i - 1] == s_run[i] && s_run[i - TILE_W - 1] == s_run[i - TILE_W];
        if (up && !implied)
            unite(lab, s_lab, i, i - TILE_W);
    }
    __syncthreads();

    // one shared atomic per run: its length onto the size of its root (s_run becomes the size array)
    int root[ITEMS];
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const int i = k * THREADS + tid;
        const bool first = member[k] && (starts[k] >> lane & 1u);
        root[k] = first ? find_root(lab, i) : -1;
        const int start_lane = member[k] ? 31 - __clz(starts[k] & (below | (1u << lane))) : lane;
        root[k] = __shfl_sync(0xffffffffu, root[k], start_lane);
        s_run[i] = 0;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        if (member[k] && (starts[k] >> lane & 1u)) {
            const unsigned ends = (starts[k] | ~members[k]) & ~(below | (1u << lane)); // lanes that end this run
            const int len = (ends ? __ffs(ends) - 1 : 32) - lane;
            atomicAdd(&s_run[root[k]], len);
        }
    }
    __syncthreads();

#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const int i = k * THREADS + tid;
        const int r = r0 + i / TILE_W, c = c0 + i % TILE_W;
        if (r >= prm.rows || c >= prm.cols)
            continue;
        const int p = r * prm.cols + c; // < 2^30
        int gp = -1;
        if (member[k]) // tile-local order is row-major, so the smallest local index is the smallest global one
            gp = (r0 + root[k] / TILE_W) * prm.cols + c0 + root[k] % TILE_W;
        prm.parent[p] = gp;
        prm.size[p] = member[k] && root[k] == i ? s_run[i] : 0;
    }
}

// pass 2: edges [0, cols * (tiles_y - 1)) cross the horizontal tile edges, the rest cross the vertical ones
template<typename T>
__global__ void __launch_bounds__(THREADS) speckle_border_kernel(const SpeckleParams prm, long long horizontal, long long total) {
    const long long e = (long long)blockIdx.x * THREADS + threadIdx.x;
    if (e >= total)
        return;
    int ra, ca, rb, cb;
    if (e < horizontal) {
        ca = cb = (int)(e % prm.cols);
        rb = (int)(e / prm.cols + 1) * TILE_H;
        ra = rb - 1;
        if (rb >= prm.rows)
            return;
    } else {
        const long long f = e - horizontal;
        ra = rb = (int)(f % prm.rows);
        cb = (int)(f / prm.rows + 1) * TILE_W;
        ca = cb - 1;
        if (cb >= prm.cols)
            return;
    }
    const T a = load_px<T>(prm, ra, ca), b = load_px<T>(prm, rb, cb);
    if (!is_member(a, prm) || !is_member(b, prm) || !is_edge(a, b, prm))
        return;
    unite(prm.parent, prm.parent, ra * prm.cols + ca, rb * prm.cols + cb);
}

__global__ void __launch_bounds__(FLAT_THREADS) speckle_flatten_kernel(const SpeckleParams prm) {
    const int c = blockIdx.x * FLAT_THREADS + threadIdx.x, r = blockIdx.y;
    if (c >= prm.cols)
        return;
    const int p = r * prm.cols + c;
    const int partial = prm.size[p]; // > 0 exactly at tile roots; only global roots gain, and they skip below
    if (partial == 0)
        return;
    volatile int* parent = prm.parent;
    const int root = find_root_readonly(parent, p); // other threads only write final roots here, so no splitting
    if (root == p)
        return;
    parent[p] = root;
    atomicAdd(prm.size + root, partial);
}

template<typename T>
__global__ void __launch_bounds__(FLAT_THREADS) speckle_write_kernel(const SpeckleParams prm) {
    const int c = blockIdx.x * FLAT_THREADS + threadIdx.x, r = blockIdx.y;
    unsigned set = 0, speckles = 0;
    if (c < prm.cols) {
        T* row = reinterpret_cast<T*>(static_cast<char*>(prm.disparity) + (size_t)r * prm.disparity_pitch);
        const int p = r * prm.cols + c;
        if (is_member(row[c], prm)) {
            const int root = __ldg(prm.parent + __ldg(prm.parent + p)); // pixel -> tile root -> global root
            if (__ldg(prm.size + root) <= prm.max_size) {
                row[c] = sizeof(T) == 2 ? T(prm.new_i) : T(prm.new_f);
                set = 1;
                speckles = root == p;
            }
        }
    }
    if (!prm.counts)
        return;
    set = __reduce_add_sync(0xffffffffu, set);
    speckles = __reduce_add_sync(0xffffffffu, speckles);
    if ((threadIdx.x & 31) == 0 && set) {
        atomicAdd(prm.counts, (unsigned long long)set);
        if (speckles)
            atomicAdd(prm.counts + 1, (unsigned long long)speckles);
    }
}

template<typename T>
cudaError_t launch_typed(const SpeckleParams& prm, cudaStream_t stream) {
    const dim3 tiles((prm.cols + TILE_W - 1) / TILE_W, (prm.rows + TILE_H - 1) / TILE_H);
    speckle_tile_kernel<T><<<tiles, THREADS, 0, stream>>>(prm);
    const long long horizontal = (long long)prm.cols * (tiles.y - 1);
    const long long total = horizontal + (long long)prm.rows * (tiles.x - 1);
    const unsigned border_blocks = total > 0 ? (unsigned)((total + THREADS - 1) / THREADS) : 1u;
    speckle_border_kernel<T><<<border_blocks, THREADS, 0, stream>>>(prm, horizontal, total);
    const dim3 rows((prm.cols + FLAT_THREADS - 1) / FLAT_THREADS, prm.rows);
    speckle_flatten_kernel<<<rows, FLAT_THREADS, 0, stream>>>(prm);
    speckle_write_kernel<T><<<rows, FLAT_THREADS, 0, stream>>>(prm);
    return cudaGetLastError();
}

} // namespace

cudaError_t launch_speckles(const SpeckleParams& prm, int is_float, cudaStream_t stream) {
    if (prm.rows <= 0 || prm.cols <= 0 || prm.rows > 32767 || prm.cols > 32767 || !prm.parent || !prm.size)
        return cudaErrorInvalidValue;
    return is_float ? launch_typed<float>(prm, stream) : launch_typed<int16_t>(prm, stream);
}

} // namespace bicos_b200
