// Kernel 2 of the BICOS::match hot path: row-wise brute-force Hamming argmin.
//
// Replaces (behaviour, not structure):
//   reference include/impl/cpu/bicos.hpp:29-76   ham / bicos_search
//   reference include/impl/cuda/bicos.cuh:50-176 bicos_search / bicos_kernel[_smem]
//
// Work = rows x units x columns: a unit is a block of 128*A left pixels of one row, whose
// descriptors a CTA keeps in registers (A per thread) while the right row streams through
// shared memory in chunks, read with warp-uniform (broadcast) vector loads. One CTA handles one
// unit, or 1/splits of its columns when the image has too few units to give every SM its
// share of CTAs (row bands of the host pipeline, row shards on 8 GPUs); the pieces of a split
// unit are merged with atomicMin. A is chosen per image width so that units tile the row with
// the least padding (1280 and 1920 columns: A = 5). The kernel is bound by the POPC pipe, so
// an SM that is left with fewer CTAs near the end simply runs them faster: a persistent grid
// with a work queue (tried, tools/search_tune.cu history) was 5 % slower than this plain grid.
//
// Exactness without the reference's serial scan:
//  * key = cost << 16 | column. min(key) over any partition of the row is the lowest cost
//    and, among equal costs, the lowest column: the reference's "first strict minimum"
//    (bicos.hpp:57-60).
//  * NODUPES (bicos.hpp:62-71: any later tie with the final minimum invalidates): a second
//    key cost << 16 | (65535 - column) finds the LAST column with the minimal cost; a
//    duplicate exists iff first != last. Both are plain min-reductions, so they merge
//    associatively across lanes, chunks and CTAs. The comparison itself happens in the
//    postfilter (refine.cu), which reads both keys.
//  * CONSISTENCY (bicos.hpp:99-106 runs a second full search from the matched right pixel
//    over the left row): Hamming distance is symmetric, so the same W x W cost tile feeds the
//    column-wise minima. Each warp min-reduces its 32*A costs for the current right column
//    with REDUX and merges into a per-CTA shared array, which is flushed to global memory
//    with atomicMin. The postfilter then only looks up rev[best_col1].
//
// Popcount pipe is the bound (16 POPC/clk/SM): carry-save compression brings a 128-bit
// distance from 4 to 3 POPC and a 256-bit distance from 8 to 4 POPC.

#include "kernels.cuh"
#include "search_common.cuh"

#include <atomic>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace bicos_b200 {
namespace {

constexpr int THREADS = 128;
constexpr int CHUNK_BYTES = 16 * 1024; // right-row descriptor bytes staged per pass
constexpr int STEP_ALIGN = 8; // CTA shares start on multiples of 8 columns (16 B aligned staging for every K)
constexpr int CTAS_PER_SM_WANTED = 20; // split units until the grid has about this many CTAs per SM
constexpr int MAX_SPLITS = 8;

// how many of a thread's A left pixels use the `light` distance
template<int K>
constexpr int DEFAULT_MIX = 0;

struct SearchArgs {
    const uint32_t* desc0;
    const uint32_t* desc1;
    int cols;
    size_t pitch_words;
    int chunk; // right descriptors staged per pass
    int units_per_row;
    int steps_per_unit; // cols rounded up to STEP_ALIGN
    long long total_steps; // rows * units_per_row * steps_per_unit
    int splits; // CTAs per unit
    uint32_t one, two, shl16; // 1, 2 and 65536 as run-time values, see mad()
    uint32_t* fwd_first;
    uint32_t* fwd_last;
    uint32_t* rev_first;
    uint32_t* rev_last;
};

// All steps [s, s_end) of the (row, unit, column) space, unit by unit.
template<int K, int FLAGS, int A, int NT, int UNROLL, int MIX>
__device__ __forceinline__ void search_range(const SearchArgs& p, long long s, const long long s_end, uint4* smem_raw) {
    constexpr bool NODUPES = (FLAGS & FLAG_NODUPES) != 0;
    constexpr bool REVERSE = (FLAGS & FLAG_CONSISTENCY) != 0;
    constexpr int UNIT = NT * A; // left pixels per unit

    uint32_t* const s_right = reinterpret_cast<uint32_t*>(smem_raw);
    uint32_t* const s_colf = s_right + (size_t)p.chunk * K;
    uint32_t* const s_coll = s_colf + p.chunk;

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int cols = p.cols;
    const Weights wts = { p.one, p.two, p.shl16 };

    while (s < s_end) {
        const long long ru = s / p.steps_per_unit;
        const int jb = (int)(s - ru * p.steps_per_unit);
        const int je = (int)min((long long)p.steps_per_unit, jb + (s_end - s));
        s += je - jb;
        const int j_end = min(je, cols);
        if (jb >= j_end)
            continue; // only the alignment padding of this unit was left
        const int row = (int)(ru / p.units_per_row);
        const int unit = (int)(ru - (long long)row * p.units_per_row);
        const bool whole = jb == 0 && je == p.steps_per_unit; // no other CTA works on this unit

        const uint32_t* const row0 = p.desc0 + (size_t)row * p.pitch_words;
        const uint32_t* const row1 = p.desc1 + (size_t)row * p.pitch_words;

        Desc<K> l[A];
        uint32_t icol[A], icol_rev[A];
        uint32_t mf[A], ml[A];
#pragma unroll
        for (int a = 0; a < A; ++a) {
            const int i = unit * UNIT + a * NT + tid;
            const bool valid = i < cols;
            l[a] = load_desc<K>(row0 + (size_t)(valid ? i : cols - 1) * K);
            // lanes past the end of the row carry bit 31 so that they never win a column minimum
            icol[a] = valid ? (uint32_t)i : (0x80000000u | (uint32_t)i);
            icol_rev[a] = valid ? (uint32_t)(65535 - i) : (0x80000000u | (uint32_t)i);
            mf[a] = KEY_NONE;
            ml[a] = KEY_NONE;
        }

        for (int j0 = jb; j0 < j_end; j0 += p.chunk) {
            const int cnt = min(p.chunk, j_end - j0);
            __syncthreads(); // previous chunk fully consumed and flushed

            // stage the right descriptors [j0, j0+cnt) (rows are 16 B aligned and padded)
            {
                const uint4* src = reinterpret_cast<const uint4*>(row1 + (size_t)j0 * K);
                const int nvec = (cnt * K + 3) / 4;
                for (int v = tid; v < nvec; v += NT)
                    smem_raw[v] = src[v];
                if constexpr (REVERSE) {
                    for (int v = tid; v < cnt; v += NT) {
                        s_colf[v] = KEY_NONE;
                        if constexpr (NODUPES)
                            s_coll[v] = KEY_NONE;
                    }
                }
            }
            __syncthreads();

            // Columns in groups of 32: lane u of every warp keeps the warp's minimum over its
            // 32*A left pixels for column u of the group, and one conflict-free shared-memory
            // atomic per group merges the warps (a per-column atomic from one lane would share
            // the MIO queue with the POPCs that bound this kernel).
            for (int jj0 = 0; jj0 < cnt; jj0 += 32) {
                const int m = min(32, cnt - jj0);
                uint32_t colf = KEY_NONE, coll = KEY_NONE;
#pragma unroll(UNROLL)
                for (int u = 0; u < m; ++u) {
                    const Desc<K> r = load_desc<K>(s_right + (size_t)(jj0 + u) * K); // warp-uniform: broadcast
                    const uint32_t j = (uint32_t)(j0 + jj0 + u);
                    uint32_t jrev = 65535u - j;
                    if constexpr (NODUPES)
                        asm("" : "+r"(jrev)); // one subtraction per column, not re-associated into every pair's add
                    uint32_t ck = KEY_NONE, ckl = KEY_NONE;
#pragma unroll
                    for (int a = 0; a < A; ++a) {
                        const uint32_t h = hamming<K>(l[a], r, a >= A - MIX, wts);
                        if constexpr (K >= 8) {
                            // ALU-pipe bound widths: keys built by IMAD (run-time 65536), only the minima on the ALU pipe
                            mf[a] = min(mf[a], mad(h, wts.shl16, j));
                            if constexpr (NODUPES)
                                ml[a] = min(ml[a], mad(h, wts.shl16, jrev));
                            if constexpr (REVERSE) {
                                ck = min(ck, mad(h, wts.shl16, icol[a]));
                                if constexpr (NODUPES)
                                    ckl = min(ckl, mad(h, wts.shl16, icol_rev[a]));
                            }
                        } else {
                            const uint32_t cost16 = h << 16;
                            mf[a] = min(mf[a], cost16 + j);
                            if constexpr (NODUPES)
                                ml[a] = min(ml[a], cost16 + jrev);
                            if constexpr (REVERSE) {
                                ck = min(ck, cost16 + icol[a]);
                                if constexpr (NODUPES)
                                    ckl = min(ckl, cost16 + icol_rev[a]);
                            }
                        }
                    }
                    if constexpr (REVERSE) {
                        ck = __reduce_min_sync(0xFFFFFFFFu, ck);
                        if (lane == u)
                            colf = ck;
                        if constexpr (NODUPES) {
                            ckl = __reduce_min_sync(0xFFFFFFFFu, ckl);
                            if (lane == u)
                                coll = ckl;
                        }
                    }
                }
                if constexpr (REVERSE) {
                    if (lane < m) {
                        atomicMin(&s_colf[jj0 + lane], colf);
                        if constexpr (NODUPES)
                            atomicMin(&s_coll[jj0 + lane], coll);
                    }
                }
            }

            if constexpr (REVERSE) {
                __syncthreads();
                uint32_t* const gf = p.rev_first + (size_t)row * cols + j0;
                uint32_t* const gl = p.rev_last + (size_t)row * cols + j0;
                for (int v = tid; v < cnt; v += NT) {
                    atomicMin(gf + v, s_colf[v]);
                    if constexpr (NODUPES)
                        atomicMin(gl + v, s_coll[v]);
                }
            }
        }

        // forward keys of this unit; the postfilter decodes them (and compares first / last)
#pragma unroll
        for (int a = 0; a < A; ++a) {
            const int i = unit * UNIT + a * NT + tid;
            if (i < cols) {
                const size_t at = (size_t)row * cols + i;
                if (whole) {
                    p.fwd_first[at] = mf[a];
                    if constexpr (NODUPES)
                        p.fwd_last[at] = ml[a];
                } else {
                    atomicMin(p.fwd_first + at, mf[a]);
                    if constexpr (NODUPES)
                        atomicMin(p.fwd_last + at, ml[a]);
                }
            }
        }
    }
}

// `splits` CTAs per unit, each an equal slice of the unit's columns.
template<int K, int FLAGS, int A, int NT, int UNROLL, int MIX>
__global__ void __launch_bounds__(NT) search_kernel(const SearchArgs p) {
    extern __shared__ uint4 smem_raw[];
    const long long ru = blockIdx.x / p.splits;
    const int part = blockIdx.x - (int)ru * p.splits;
    const int span = ((p.steps_per_unit + p.splits - 1) / p.splits + STEP_ALIGN - 1) & ~(STEP_ALIGN - 1);
    const long long base = ru * p.steps_per_unit;
    const long long s = base + (long long)part * span;
    const long long s_end = min(base + p.steps_per_unit, s + span);
    if (s < s_end)
        search_range<K, FLAGS, A, NT, UNROLL, MIX>(p, s, s_end, smem_raw);
}

int chunk_for(int K, int cols) {
    const int cap = CHUNK_BYTES / (4 * K);
    const int padded = (cols + 3) & ~3;
    return padded < cap ? padded : cap;
}

// left descriptors per thread: the unit width 128*A that tiles `cols` with the least padding
int pick_a(int cols) {
    int best_a = 4;
    long long best_pad = -1;
    for (int a: { 4, 5, 3 }) {
        const long long unit = (long long)THREADS * a;
        const long long padded = (cols + unit - 1) / unit * unit;
        if (best_pad < 0 || padded < best_pad) {
            best_pad = padded;
            best_a = a;
        }
    }
    return best_a;
}

int sm_count() {
    static thread_local int cached_dev = -1, cached_sms = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess)
        return 148;
    if (dev != cached_dev) {
        if (cudaDeviceGetAttribute(&cached_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
            cached_sms = 148;
        cached_dev = dev;
    }
    return cached_sms;
}

// splits <= 0: chosen here from the grid size
template<int K, int FLAGS, int A, int NT = THREADS, int UNROLL = 2, int MIX = DEFAULT_MIX<K>>
cudaError_t launch_one(
    const uint32_t* desc0,
    const uint32_t* desc1,
    int rows,
    int cols,
    size_t pitch_words,
    uint32_t* fwd_first,
    uint32_t* fwd_last,
    uint32_t* rev_first,
    uint32_t* rev_last,
    cudaStream_t stream,
    int splits = 0
) {
    SearchArgs p;
    p.desc0 = desc0;
    p.desc1 = desc1;
    p.cols = cols;
    p.pitch_words = pitch_words;
    p.chunk = chunk_for(K, cols);
    const int unit = NT * A;
    p.units_per_row = (cols + unit - 1) / unit;
    p.steps_per_unit = (cols + STEP_ALIGN - 1) / STEP_ALIGN * STEP_ALIGN;
    p.total_steps = (long long)rows * p.units_per_row * p.steps_per_unit;
    const long long units = (long long)rows * p.units_per_row;
    if (splits <= 0) {
        // about 512 columns per CTA (measured best at 2048 columns: tools/search_tune), down to
        // 256 when the image has too few units to give every SM its share of CTAs
        splits = p.steps_per_unit / 512;
        const long long wanted = (long long)sm_count() * CTAS_PER_SM_WANTED;
        if (units * splits < wanted)
            splits = p.steps_per_unit / 256;
        splits = splits > MAX_SPLITS ? MAX_SPLITS : splits < 1 ? 1 : splits;
    }
    p.splits = splits;
    p.one = 1u;
    p.two = 2u;
    p.shl16 = 65536u;
    p.fwd_first = fwd_first;
    p.fwd_last = fwd_last;
    p.rev_first = rev_first;
    p.rev_last = rev_last;
    const int smem = search_smem_bytes(K, cols, FLAGS);
    auto kernel = search_kernel<K, FLAGS, A, NT, UNROLL, MIX>;
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (err != cudaSuccess)
        return err;
    const long long grid = units * p.splits;
    if (grid <= 0 || grid > 0x7FFFFFFFLL)
        return cudaErrorInvalidConfiguration;
    kernel<<<(unsigned)grid, NT, smem, stream>>>(p);
    return cudaGetLastError();
}

template<int K, int FLAGS>
cudaError_t launch_a(
    const uint32_t* desc0,
    const uint32_t* desc1,
    int rows,
    int cols,
    size_t pitch_words,
    uint32_t* fwd_first,
    uint32_t* fwd_last,
    uint32_t* rev_first,
    uint32_t* rev_last,
    cudaStream_t stream
) {
    switch (pick_a(cols)) {
        case 3:
            return launch_one<K, FLAGS, 3>(desc0, desc1, rows, cols, pitch_words, fwd_first, fwd_last, rev_first, rev_last, stream);
        case 5:
            return launch_one<K, FLAGS, 5>(desc0, desc1, rows, cols, pitch_words, fwd_first, fwd_last, rev_first, rev_last, stream);
        default:
            return launch_one<K, FLAGS, 4>(desc0, desc1, rows, cols, pitch_words, fwd_first, fwd_last, rev_first, rev_last, stream);
    }
}

template<int K>
cudaError_t launch_k(
    const uint32_t* desc0,
    const uint32_t* desc1,
    int rows,
    int cols,
    size_t pitch_words,
    int flags,
    uint32_t* fwd_first,
    uint32_t* fwd_last,
    uint32_t* rev_first,
    uint32_t* rev_last,
    cudaStream_t stream
) {
    switch (flags) {
        case FLAG_NODUPES:
            return launch_a<K, FLAG_NODUPES>(desc0, desc1, rows, cols, pitch_words, fwd_first, fwd_last, rev_first, rev_last, stream);
        case FLAG_CONSISTENCY:
            return launch_a<K, FLAG_CONSISTENCY>(desc0, desc1, rows, cols, pitch_words, fwd_first, fwd_last, rev_first, rev_last, stream);
        case FLAG_NODUPES | FLAG_CONSISTENCY:
            return launch_a<K, FLAG_NODUPES | FLAG_CONSISTENCY>(desc0, desc1, rows, cols, pitch_words, fwd_first, fwd_last, rev_first, rev_last, stream);
        case 0: // plain first-minimum search (building block, not reachable from Config)
            return launch_a<K, 0>(desc0, desc1, rows, cols, pitch_words, fwd_first, fwd_last, rev_first, rev_last, stream);
    }
    return cudaErrorInvalidValue;
}

} // namespace

int search_smem_bytes(int K, int cols, int flags) {
    const int chunk = chunk_for(K, cols);
    int bytes = chunk * K * 4;
    if (flags & FLAG_CONSISTENCY)
        bytes += chunk * 4 * ((flags & FLAG_NODUPES) ? 2 : 1);
    return bytes;
}

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
) {
    if (rows <= 0 || cols <= 0 || cols > 32767)
        return cudaErrorInvalidValue;
    note_search_kernel("popc<K=%d,flags=%d>", K, flags);
    switch (K) {
        case 1:
            return launch_k<1>(desc0, desc1, rows, cols, desc_pitch_words, flags, fwd_first, fwd_last, rev_first, rev_last, stream);
        case 2:
            return launch_k<2>(desc0, desc1, rows, cols, desc_pitch_words, flags, fwd_first, fwd_last, rev_first, rev_last, stream);
        case 4:
            return launch_k<4>(desc0, desc1, rows, cols, desc_pitch_words, flags, fwd_first, fwd_last, rev_first, rev_last, stream);
        case 8:
            return launch_k<8>(desc0, desc1, rows, cols, desc_pitch_words, flags, fwd_first, fwd_last, rev_first, rev_last, stream);
        case 12: // wide-descriptor extension (bicos_b200_config::wide_descriptors): FULL stacks of 17..20 images
            return launch_k<12>(desc0, desc1, rows, cols, desc_pitch_words, flags, fwd_first, fwd_last, rev_first, rev_last, stream);
        case 16: // FULL stacks of 21..23 images
            return launch_k<16>(desc0, desc1, rows, cols, desc_pitch_words, flags, fwd_first, fwd_last, rev_first, rev_last, stream);
    }
    return cudaErrorInvalidValue;
}

namespace {
std::atomic<int> g_engine { -1 };
thread_local char g_last_kernel[96] = "";
}

const char* last_search_kernel() {
    return g_last_kernel;
}

void note_search_kernel(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_last_kernel, sizeof g_last_kernel, fmt, ap);
    va_end(ap);
}

int search_engine() {
    int e = g_engine.load(std::memory_order_relaxed);
    if (e < 0) {
        const char* v = getenv("BICOS_B200_SEARCH_ENGINE");
        e = !v ? 0 : !strcmp(v, "popc") ? 1 : !strcmp(v, "mma") ? 2 : 0;
        g_engine.store(e, std::memory_order_relaxed);
    }
    return e;
}

void set_search_engine(int engine) {
    g_engine.store(engine < 0 || engine > 2 ? 0 : engine, std::memory_order_relaxed);
}

bool search_needs_prefill(int K, int cols) {
    const int engine = search_engine();
    return !(engine == 2 || (engine == 0 && search_mma_supports(K, cols)));
}

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
    int free_top_bits
) {
    const int engine = search_engine();
    if (engine == 2 || (engine == 0 && search_mma_supports(K, cols)))
        return launch_search_mma(desc0, desc1, K, rows, cols, desc_pitch_words, flags, fwd_first, fwd_last, rev_first, rev_last, stream, free_top_bits);
    return launch_search_popc(desc0, desc1, K, rows, cols, desc_pitch_words, flags, fwd_first, fwd_last, rev_first, rev_last, stream);
}

} // namespace bicos_b200
