// C-ABI layer (include/bicos_b200.h) over the three kernels: argument validation with the
// reference's error behaviour, the per-device workspace, stage sequencing, and the
// host-buffer variant that pybicos' BICOS_Match builds on.
//
// Reference behaviour mirrored here (not its structure):
//   src/impl/cpu.cpp:100-159 / src/impl/cuda.cu:465-524   validation + descriptor width choice
//   src/impl/cpu.cpp:35-98                                 stage order and output types
//   src/pybicos_c.cpp:56-89                                negative float = unset optional

#include "../../include/bicos_b200.h"
#include "kernels.cuh"

#include <nvtx3/nvToolsExt.h> // header-only; a no-op unless a profiler injects itself

#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

using namespace bicos_b200;

namespace {

thread_local std::string g_error;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
    return code;
}

int cuda_fail(cudaError_t err, const char* what) {
    return fail(BICOS_B200_ERR_CUDA, "%s: %s (%s)", what, cudaGetErrorString(err), cudaGetErrorName(err));
}

// a tensor-core search kernel gave up on a wait since the last check (search_mma.cu, mbar_wait_slow)
int check_search_timeout() {
    if (const unsigned int v = search_mma_take_timeout())
        return fail(BICOS_B200_ERR_CUDA,
                    "search pipeline timeout (CTA %u): a wait inside the tensor-core search kernel exceeded BICOS_B200_MMA_TIMEOUT_MS; "
                    "results of that match are invalid (BICOS_B200_SEARCH_ENGINE=popc selects the other engine)", v - 1);
    return 0;
}

#define CU(call) \
    do { \
        cudaError_t err__ = (call); \
        if (err__ != cudaSuccess) \
            return cuda_fail(err__, #call); \
    } while (0)

// NVTX range around a host-side section (stage launches, host staging): shows up on the ncu / nsys timeline
struct Range {
    explicit Range(const char* name) {
        nvtxRangePushA(name);
    }
    ~Range() {
        nvtxRangePop();
    }
    Range(const Range&) = delete;
    Range& operator=(const Range&) = delete;
};

struct DeviceBuffer {
    void* ptr = nullptr;
    size_t cap = 0;

    // grow-only; a reallocation waits for the device so no kernel still reads the old block
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap)
            return cudaSuccess;
        cudaError_t err = cudaDeviceSynchronize();
        if (err != cudaSuccess)
            return err;
        if (ptr)
            cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
        err = cudaMalloc(&ptr, bytes);
        if (err == cudaSuccess)
            cap = bytes;
        return err;
    }
    void release() {
        if (ptr)
            cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
    }
};

struct PinnedBuffer {
    void* ptr = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap)
            return cudaSuccess;
        release();
        cudaError_t err = cudaHostAlloc(&ptr, bytes, cudaHostAllocDefault);
        if (err == cudaSuccess)
            cap = bytes;
        else
            ptr = nullptr;
        return err;
    }
    void release() {
        if (ptr)
            cudaFreeHost(ptr);
        ptr = nullptr;
        cap = 0;
    }
};

// A few persistent host threads for memcpy between pageable caller memory and the pinned staging
// buffers of the host-buffer entry points (one thread moves ~10 GB/s, PCIe wants 50).
class CopyPool {
public:
    static CopyPool& get() {
        static CopyPool pool;
        return pool;
    }
    // fn(i) for i in [0, count), spread over the workers and the calling thread; returns when all ran
    void parallel_for(int count, const std::function<void(int)>& fn) {
        if (count <= 0)
            return;
        std::unique_lock<std::mutex> call_lock(call_mutex_); // one job at a time
        {
            std::lock_guard<std::mutex> lk(m_);
            job_ = &fn;
            next_ = 0;
            count_ = count;
            pending_ = count;
            ++generation_;
        }
        cv_.notify_all();
        run_some();
        std::unique_lock<std::mutex> lk(m_);
        cv_done_.wait(lk, [&] { return pending_ == 0; });
        job_ = nullptr;
    }

private:
    CopyPool() {
        unsigned hw = std::thread::hardware_concurrency();
        int n = hw >= 16 ? 7 : hw >= 8 ? 3 : 1; // plus the calling thread
        for (int i = 0; i < n; ++i)
            workers_.emplace_back([this] { worker(); });
    }
    ~CopyPool() {
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto& t: workers_)
            t.join();
    }
    void run_some() {
        for (;;) {
            int i;
            const std::function<void(int)>* fn;
            {
                std::lock_guard<std::mutex> lk(m_);
                if (!job_ || next_ >= count_)
                    return;
                i = next_++;
                fn = job_;
            }
            (*fn)(i);
            {
                std::lock_guard<std::mutex> lk(m_);
                if (--pending_ == 0)
                    cv_done_.notify_all();
            }
        }
    }
    void worker() {
        unsigned long long seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return stop_ || generation_ != seen; });
                if (stop_)
                    return;
                seen = generation_;
            }
            run_some();
        }
    }
    std::vector<std::thread> workers_;
    std::mutex m_, call_mutex_;
    std::condition_variable cv_, cv_done_;
    const std::function<void(int)>* job_ = nullptr;
    int next_ = 0, count_ = 0, pending_ = 0;
    unsigned long long generation_ = 0;
    bool stop_ = false;
};

// pageable (unregistered) host memory? Pinned and registered memory can be handed to the DMA
// engines directly; everything else goes through the handle's pinned staging buffers.
bool is_pageable(const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return attr.type == cudaMemoryTypeUnregistered;
}

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&prev) != cudaSuccess)
            ok = false;
        else if (prev != device && cudaSetDevice(device) != cudaSuccess)
            ok = false;
    }
    ~DeviceGuard() {
        if (prev >= 0)
            cudaSetDevice(prev);
    }
};

int descriptor_bits(int n, int mode) {
    // src/impl/cpu.cpp:122-124 (LIMITED is undercounted by one there; no bucket boundary moves)
    return mode ? n * n - 2 * n + 3 : 4 * n - 7;
}

// src/impl/cpu.cpp:131-156: 32 / 64 / 128 / 256 bits, more is rejected. `wide` (extension, off by
// default): 384 and 512 bits as well, i.e. FULL stacks of 17..23 images.
int words_for_bits(int bits, bool wide) {
    if (bits <= 32)
        return 1;
    if (bits <= 64)
        return 2;
    if (bits <= 128)
        return 4;
    if (bits <= 256)
        return 8;
    if (wide && bits <= 384)
        return 12;
    if (wide && bits <= 512)
        return 16;
    return -1;
}

// `mode` arguments of the stage entry points: bit 0 = FULL, bit 1 = BICOS_B200_MODE_WIDE
bool mode_is_full(int mode) {
    return (mode & 1) != 0;
}
bool cfg_is_wide(const bicos_b200_config* cfg) {
    return cfg->wide_descriptors != 0 || (cfg->mode & BICOS_B200_MODE_WIDE) != 0;
}

// is the NXC stage on? (see bicos_b200_config::negative_threshold_is_set)
bool has_thr(const bicos_b200_config* cfg) {
    return cfg->nxcorr_threshold >= 0 || cfg->negative_threshold_is_set != 0;
}

// the configuration's disparity range clipped to the row; false when there is none or it covers the whole row,
// which is the same search (bicos_b200_config::has_disparity_range)
bool cfg_range(const bicos_b200_config* cfg, int cols, int* dmin, int* dmax) {
    if (!cfg->has_disparity_range)
        return false;
    *dmin = cfg->min_disparity;
    *dmax = cfg->max_disparity;
    return disparity_range_clip(cols, dmin, dmax);
}

// the windowed search has no tensor-core kernel: a forced tensor engine fails as for its other unsupported shapes
int check_range_engine() {
    if (search_engine() == 2)
        return fail(BICOS_B200_ERR_CUDA, "the tensor-core search engine has no disparity-range kernel (BICOS_B200_SEARCH_AUTO or "
                                         "BICOS_B200_SEARCH_POPC run ranged searches)");
    return 0;
}

size_t depth_bytes(int depth) {
    return depth == BICOS_B200_16U ? 2 : 1;
}

} // namespace

constexpr int MAX_BANDS = 16;
constexpr int PIN_SLOTS = 3;
constexpr int N_STAGES = 3; // transform (both stacks), search, refine

struct bicos_b200_handle_s {
    int device = 0;
    DeviceBuffer desc0, desc1, keys, xs; // keys: up to four [rows][cols] uint32 search-key arrays
    DeviceBuffer stage_in, stage_disp, stage_corr;
    DeviceBuffer rect; // bicos_b200_match_rectified: both rectified stacks, [2n][rows][rect pitch]
    DeviceBuffer reproj; // bicos_b200_reproject: ReprojectWork + one look-back status word per tile
    DeviceBuffer speckle; // bicos_b200_filter_speckles: union-find parents and component sizes, int32 [2][rows * cols]
    float xs_step = -1.f;
    int xs_count = 0;
    bool host_pending = false; // between bicos_b200_match_host_begin and _end
    // pageable callers: ring of pinned band buffers for the inputs, pinned images for the outputs
    PinnedBuffer pin_in[PIN_SLOTS], pin_disp, pin_corr;
    cudaEvent_t ev_slot[PIN_SLOTS] = {};
    void *user_disp = nullptr, *user_corr = nullptr; // where _end copies the pinned outputs to
    size_t user_disp_bytes = 0, user_corr_bytes = 0;
    long long launches = 0;
    // the workspace (descriptors, keys, x table) is shared by all matches of the handle: a match enqueued on
    // another stream than the previous one first waits for it (do_match)
    cudaEvent_t ev_last = nullptr;
    cudaStream_t last_stream = nullptr;
    bool has_last = false;
    // host-buffer pipeline (bicos_b200_match_host): upload / compute / download streams
    cudaStream_t s_in = nullptr, s_compute = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[MAX_BANDS] = {}, ev_done[MAX_BANDS] = {};
    // two-stream pipeline of bicos_b200_match_batch: transform + search of unit u + 1 beside the refine of unit u
    DeviceBuffer keys_b; // second set of key arrays (unit parity)
    bool overlap = true; // bicos_b200_set_overlap
    cudaStream_t p_search = nullptr, p_refine = nullptr;
    cudaEvent_t p_start = nullptr, p_done = nullptr, p_searched[2] = {}, p_refined[2] = {};
    // optional per-stage timing (bicos_b200_set_profiling)
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events; // a (begin, end) event pair per recorded stage, stage index in prof_stage
    std::vector<int> prof_stage;
    size_t prof_used = 0;
    double stage_ms[N_STAGES] = { 0, 0, 0 };
    long long stage_count = 0;
};

namespace {

int validate_common(int n, int rows, int cols, int depth, const bicos_b200_config* cfg, int* K_out) {
    if (!cfg)
        return fail(BICOS_B200_ERR_INVALID, "config is null");
    if (n < 2)
        return fail(BICOS_B200_ERR_INVALID, "need at least two images"); // cpu.cpp:110-111
    if (depth != BICOS_B200_8U && depth != BICOS_B200_16U)
        return fail(BICOS_B200_ERR_INVALID, "bad input depths, only CV_8UC1 and CV_16UC1 are supported"); // cpu.cpp:113-114
    const int bits = descriptor_bits(n, mode_is_full(cfg->mode));
    const int K = words_for_bits(bits, cfg_is_wide(cfg));
    if (K < 0 || n > MAX_IMAGES)
        return fail(BICOS_B200_ERR_INVALID, "input stacks too large, would require %d bits", bits); // cpu.cpp:154-155
    if (rows <= 0 || cols <= 0)
        return fail(BICOS_B200_ERR_INVALID, "empty images");
    if (cols > 32767 || rows > 65535)
        return fail(BICOS_B200_ERR_INVALID, "image too large: at most 32767 columns (int16 disparity) and 65535 rows");
    if (has_thr(cfg) && cfg->subpixel_step == 0.0f)
        return fail(BICOS_B200_ERR_INVALID, "subpixel_step must be positive (the reference loops forever on 0)");
    if (cfg->has_disparity_range && cfg->min_disparity > cfg->max_disparity)
        return fail(BICOS_B200_ERR_INVALID, "disparity range [%d, %d]: min > max", cfg->min_disparity, cfg->max_disparity);
    if (K_out)
        *K_out = K;
    return 0;
}

int search_flags(const bicos_b200_config* cfg) {
    // src/impl/cpu.cpp:68-75
    if (cfg->variant_type != 0)
        return FLAG_CONSISTENCY | (cfg->no_dupes ? FLAG_NODUPES : 0);
    return FLAG_NODUPES;
}

int fill_table(PlaneTable& t, const void* const* planes, int n, size_t row_offset_bytes) {
    for (int i = 0; i < n; ++i) {
        if (!planes[i])
            return fail(BICOS_B200_ERR_INVALID, "image %d is null", i);
        t.p[i] = static_cast<const char*>(planes[i]) + row_offset_bytes;
    }
    for (int i = n; i < MAX_IMAGES; ++i)
        t.p[i] = nullptr;
    return 0;
}

// the x values of `for (float x = -1.f; x <= 1.f; x += step)` (agree.hpp:165), cached per step
int prepare_steps(bicos_b200_handle h, float step, cudaStream_t stream) {
    if (h->xs_count > 0 && h->xs_step == step)
        return 0;
    std::vector<float> xs;
    for (float x = -1.f; x <= 1.f; x += step) {
        xs.push_back(x);
        if (xs.size() > (1u << 16))
            return fail(BICOS_B200_ERR_INVALID, "subpixel_step %g too small (more than 65536 steps)", (double)step);
    }
    CU(h->xs.reserve(xs.size() * sizeof(float)));
    CU(cudaMemcpyAsync(h->xs.ptr, xs.data(), xs.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
    CU(cudaStreamSynchronize(stream)); // xs is a stack-owned pageable buffer
    h->xs_step = step;
    h->xs_count = (int)xs.size();
    return 0;
}

// Stage timing: an event before and after a stage on the stream it runs on (the stages of a match may run on
// different streams, bicos_b200_match_batch), folded into stage_ms by prof_collect.
int prof_event(bicos_b200_handle h, int stage, cudaStream_t stream) {
    if (!h->profiling)
        return 0;
    if (h->prof_used == h->prof_events.size()) {
        cudaEvent_t e;
        CU(cudaEventCreate(&e));
        h->prof_events.push_back(e);
        h->prof_stage.push_back(0);
    }
    h->prof_stage[h->prof_used] = stage;
    CU(cudaEventRecord(h->prof_events[h->prof_used++], stream));
    return 0;
}

struct StageTimer {
    bicos_b200_handle h;
    int stage;
    cudaStream_t stream;
    int rc;
    StageTimer(bicos_b200_handle h_, int stage_, cudaStream_t stream_): h(h_), stage(stage_), stream(stream_) {
        rc = prof_event(h, stage, stream);
    }
    int end() {
        return rc ? rc : prof_event(h, stage, stream);
    }
};

// fold all completed (begin, end) pairs into stage_ms; requires the work to be finished
int prof_collect(bicos_b200_handle h) {
    for (size_t g = 0; g + 2 <= h->prof_used; g += 2) {
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, h->prof_events[g], h->prof_events[g + 1]));
        h->stage_ms[h->prof_stage[g]] += ms;
    }
    h->prof_used = 0;
    return 0;
}

size_t desc_pitch_for(int cols, int K) {
    return ((size_t)cols * K + 3) & ~(size_t)3; // rows start 16 B aligned
}

// `ranged`: the windowed search writes fwd_last for every flags (launch_search_range)
int key_arrays(int flags, bool ranged) {
    return 1 + ((flags & FLAG_NODUPES) || ranged ? 1 : 0) + ((flags & FLAG_CONSISTENCY) ? ((flags & FLAG_NODUPES) ? 2 : 1) : 0);
}

struct KeyArrays {
    uint32_t *fwd_first, *fwd_last, *rev_first, *rev_last;
};

KeyArrays split_keys(uint32_t* base, size_t px, int flags, bool ranged) {
    KeyArrays k { base, nullptr, nullptr, nullptr };
    uint32_t* next = base + px;
    if ((flags & FLAG_NODUPES) || ranged) {
        k.fwd_last = next;
        next += px;
    }
    if (flags & FLAG_CONSISTENCY) {
        k.rev_first = next;
        next += px;
        if (flags & FLAG_NODUPES)
            k.rev_last = next;
    }
    return k;
}

int do_refine(
    bicos_b200_handle h,
    const PlaneTable& t0,
    const PlaneTable& t1,
    int n,
    int rows,
    int cols,
    size_t pitch_bytes,
    int depth,
    const bicos_b200_config* cfg,
    const uint32_t* fwd_first,
    const uint32_t* fwd_last,
    const uint32_t* rev_first,
    const uint32_t* rev_last,
    int16_t* raw_out,
    void* disparity,
    size_t disparity_pitch,
    void* corrmap,
    size_t corrmap_pitch,
    cudaStream_t stream,
    bool windowed = false
) {
    RefineParams prm {};
    prm.n = n;
    prm.rows = rows;
    prm.cols = cols;
    prm.in_pitch = pitch_bytes;
    prm.is_u16 = depth == BICOS_B200_16U;
    prm.is_double = cfg->precision != 0;
    prm.consistency = cfg->variant_type != 0;
    prm.nodupes_reverse = prm.consistency && cfg->no_dupes;
    prm.max_lr_diff = cfg->max_lr_diff;
    prm.has_threshold = has_thr(cfg);
    prm.threshold = cfg->nxcorr_threshold;
    prm.has_minvar = cfg->min_variance >= 0;
    prm.minvar_times_n = prm.has_minvar ? cfg->min_variance * (float)n : 0.f; // cpu.cpp:127
    prm.subpixel = prm.has_threshold && cfg->subpixel_step >= 0;
    prm.nsteps = 0;
    prm.xs = nullptr;
    prm.one = 1.0f;
    prm.inv_n = 1.0f / (float)n; // IEEE single-precision division on the host: RN(1 / n)
    if (prm.subpixel) {
        if (int rc = prepare_steps(h, cfg->subpixel_step, stream))
            return rc;
        prm.nsteps = h->xs_count;
        prm.xs = static_cast<const float*>(h->xs.ptr);
    }
    int dmin = 0, dmax = 0;
    // ranged and windowed keys: the first / last comparison also rejects the empty windows (launch_search_range)
    prm.nodupes_forward = (search_flags(cfg) & FLAG_NODUPES) != 0 || cfg_range(cfg, cols, &dmin, &dmax) || windowed;
    prm.fwd_first = fwd_first;
    prm.fwd_last = fwd_last;
    prm.rev_first = rev_first;
    prm.rev_last = rev_last;
    prm.raw_out = raw_out;
    prm.disp_out = disparity;
    prm.disp_pitch = disparity_pitch;
    prm.corr_out = prm.has_threshold ? corrmap : nullptr;
    prm.corr_pitch = corrmap_pitch;
    CU(launch_refine(t0, t1, prm, stream));
    h->launches += 1;
    return 0;
}

// One unit of work of the path: rows [row_begin, row_end) of one stereo stack, with the output rows it writes.
struct Unit {
    PlaneTable t0, t1; // plane pointers already advanced to row_begin
    int row_begin = 0;
    int nrows = 0;
    char* disp_rows = nullptr;
    char* corr_rows = nullptr;
};

struct MatchShape {
    int n, cols, K, depth, flags;
    bool ranged; // a disparity range that excludes some pairs, or window maps: the windowed search, [dmin, dmax] clipped
    int dmin, dmax;
    const int16_t* wmin; // window maps (bicos_b200_match_windows), [rows][wpitch elements] from the match's row 0; or null
    const int16_t* wmax;
    size_t wpitch;
    size_t pitch_bytes, disparity_pitch, corrmap_pitch;
    const bicos_b200_config* cfg;
};

int make_unit(Unit& u, const void* const* planes0, const void* const* planes1, const MatchShape& sh, int row_begin, int row_end,
              void* disparity, void* corrmap) {
    if (int rc = fill_table(u.t0, planes0, sh.n, (size_t)row_begin * sh.pitch_bytes))
        return rc;
    if (int rc = fill_table(u.t1, planes1, sh.n, (size_t)row_begin * sh.pitch_bytes))
        return rc;
    u.row_begin = row_begin;
    u.nrows = row_end - row_begin;
    u.disp_rows = static_cast<char*>(disparity) + (size_t)row_begin * sh.disparity_pitch;
    u.corr_rows = corrmap ? static_cast<char*>(corrmap) + (size_t)row_begin * sh.corrmap_pitch : nullptr;
    return 0;
}

// stages 1 + 2 of a unit: both descriptor transforms and the search, keys into `keys`
int enqueue_search_stage(bicos_b200_handle h, const Unit& u, const MatchShape& sh, uint32_t* keys, cudaStream_t stream) {
    const size_t dpw = desc_pitch_for(sh.cols, sh.K);
    const size_t px = (size_t)u.nrows * sh.cols;
    uint32_t* d0 = static_cast<uint32_t*>(h->desc0.ptr);
    uint32_t* d1 = static_cast<uint32_t*>(h->desc1.ptr);
    const int is_u16 = sh.depth == BICOS_B200_16U;
    {
        Range nvtx("bicos_b200::transform x2");
        StageTimer timer(h, 0, stream);
        CU(launch_transform(u.t0, sh.n, u.nrows, sh.cols, sh.pitch_bytes, is_u16, mode_is_full(sh.cfg->mode), sh.K, d0, dpw, stream));
        CU(launch_transform(u.t1, sh.n, u.nrows, sh.cols, sh.pitch_bytes, is_u16, mode_is_full(sh.cfg->mode), sh.K, d1, dpw, stream));
        h->launches += 2;
        if (int rc = timer.end())
            return rc;
    }
    Range nvtx("bicos_b200::search");
    StageTimer timer(h, 1, stream);
    KeyArrays ka = split_keys(keys, px, sh.flags, sh.ranged);
    if (sh.ranged) {
        if (sh.flags & FLAG_CONSISTENCY) // reverse minima merge across CTAs with atomicMin; the forward keys are stored
            CU(cudaMemsetAsync(ka.rev_first, 0xFF, px * sizeof(uint32_t) * ((sh.flags & FLAG_NODUPES) ? 2 : 1), stream));
        if (sh.wmin) {
            const size_t w0 = (size_t)u.row_begin * sh.wpitch;
            CU(launch_search_windows(d0, d1, sh.K, u.nrows, sh.cols, dpw, sh.flags, sh.wmin + w0, sh.wmax + w0, sh.wpitch, ka.fwd_first,
                                     ka.fwd_last, ka.rev_first, ka.rev_last, stream));
        } else {
            CU(launch_search_range(d0, d1, sh.K, u.nrows, sh.cols, dpw, sh.flags, sh.dmin, sh.dmax, ka.fwd_first, ka.fwd_last,
                                   ka.rev_first, ka.rev_last, stream));
        }
        h->launches += 1;
        return timer.end();
    }
    if (search_needs_prefill(sh.K, sh.cols)) // the popcount engine merges with atomicMin; the tensor-core engine stores every key
        CU(cudaMemsetAsync(keys, 0xFF, px * sizeof(uint32_t) * key_arrays(sh.flags, false), stream));
    // descriptors of our own transform: 4n - 6 or n^2 - 2n + 3 bits, never all 32 K, so the top bit is free
    CU(launch_search(d0, d1, sh.K, u.nrows, sh.cols, dpw, sh.flags, ka.fwd_first, ka.fwd_last, ka.rev_first, ka.rev_last, stream, 2)); // the transform leaves the top two descriptor bits clear
    h->launches += 1;
    return timer.end();
}

// stages 4 + 3 of a unit: postfilter and NXC refinement from `keys` into the unit's output rows
int enqueue_refine_stage(bicos_b200_handle h, const Unit& u, const MatchShape& sh, uint32_t* keys, cudaStream_t stream) {
    Range nvtx("bicos_b200::postfilter+refine");
    StageTimer timer(h, 2, stream);
    KeyArrays ka = split_keys(keys, (size_t)u.nrows * sh.cols, sh.flags, sh.ranged);
    if (int rc = do_refine(h, u.t0, u.t1, sh.n, u.nrows, sh.cols, sh.pitch_bytes, sh.depth, sh.cfg, ka.fwd_first, ka.fwd_last, ka.rev_first,
                           ka.rev_last, nullptr, u.disp_rows, sh.disparity_pitch, u.corr_rows, sh.corrmap_pitch, stream, sh.wmin != nullptr))
        return rc;
    return timer.end();
}

int validate_match(const void* const* planes0, const void* const* planes1, int n, int rows, int cols, size_t pitch_bytes, int depth,
                   const bicos_b200_config* cfg, const void* disparity, MatchShape& sh) {
    int K = 0;
    if (int rc = validate_common(n, rows, cols, depth, cfg, &K))
        return rc;
    if (!planes0 || !planes1 || !disparity)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    if (pitch_bytes < (size_t)cols * depth_bytes(depth))
        return fail(BICOS_B200_ERR_INVALID, "pitch smaller than a row");
    sh.n = n;
    sh.cols = cols;
    sh.K = K;
    sh.depth = depth;
    sh.flags = search_flags(cfg);
    sh.ranged = cfg_range(cfg, cols, &sh.dmin, &sh.dmax);
    if (sh.ranged)
        if (int rc = check_range_engine())
            return rc;
    sh.pitch_bytes = pitch_bytes;
    sh.cfg = cfg;
    return 0;
}

int reserve_workspace(bicos_b200_handle h, const MatchShape& sh, int max_unit_rows, bool second_keys) {
    const size_t dpw = desc_pitch_for(sh.cols, sh.K);
    CU(h->desc0.reserve(dpw * max_unit_rows * sizeof(uint32_t)));
    CU(h->desc1.reserve(dpw * max_unit_rows * sizeof(uint32_t)));
    // key arrays, contiguous so that one memset initialises them: fwd_first, then fwd_last
    // (NODUPES), rev_first (CONSISTENCY), rev_last (both)
    const size_t key_bytes = (size_t)max_unit_rows * sh.cols * sizeof(uint32_t) * key_arrays(sh.flags, sh.ranged);
    CU(h->keys.reserve(key_bytes));
    if (second_keys)
        CU(h->keys_b.reserve(key_bytes));
    return 0;
}

// the handle's workspace is shared by everything enqueued through it: order after its previous user
int enter_workspace(bicos_b200_handle h, cudaStream_t stream) {
    if (int rc = check_search_timeout())
        return rc;
    if (h->has_last && h->last_stream != stream)
        CU(cudaStreamWaitEvent(stream, h->ev_last, 0));
    return 0;
}

int leave_workspace(bicos_b200_handle h, cudaStream_t stream) {
    if (!h->ev_last)
        CU(cudaEventCreateWithFlags(&h->ev_last, cudaEventDisableTiming));
    CU(cudaEventRecord(h->ev_last, stream));
    h->last_stream = stream;
    h->has_last = true;
    return 0;
}

// window maps for rows of `cols` pixels (bicos_b200_disparity_windows)
int validate_windows(const bicos_b200_disparity_windows* w, int cols) {
    if (!w || !w->min_disparity || !w->max_disparity)
        return fail(BICOS_B200_ERR_INVALID, "disparity windows: a map is null");
    if (w->pitch_bytes % 2 != 0 || w->pitch_bytes < (size_t)cols * 2 || reinterpret_cast<uintptr_t>(w->min_disparity) % 2 != 0 ||
        reinterpret_cast<uintptr_t>(w->max_disparity) % 2 != 0)
        return fail(BICOS_B200_ERR_INVALID, "disparity windows: pitch %zu must be even and at least cols * 2 = %d, maps 2-byte aligned",
                    w->pitch_bytes, cols * 2);
    return 0;
}

int do_match(
    bicos_b200_handle h,
    const void* const* planes0,
    const void* const* planes1,
    int n,
    int rows,
    int cols,
    size_t pitch_bytes,
    int depth,
    const bicos_b200_config* cfg,
    int row_begin,
    int row_end,
    void* disparity,
    size_t disparity_pitch,
    void* corrmap,
    size_t corrmap_pitch,
    cudaStream_t stream,
    const bicos_b200_disparity_windows* windows = nullptr
) {
    MatchShape sh {};
    if (int rc = validate_match(planes0, planes1, n, rows, cols, pitch_bytes, depth, cfg, disparity, sh))
        return rc;
    if (windows) {
        if (cfg->has_disparity_range)
            return fail(BICOS_B200_ERR_INVALID, "disparity windows and a disparity range exclude each other");
        if (int rc = validate_windows(windows, cols))
            return rc;
        if (int rc = check_range_engine())
            return rc;
        sh.ranged = true;
        sh.wmin = windows->min_disparity;
        sh.wmax = windows->max_disparity;
        sh.wpitch = windows->pitch_bytes / 2;
    }
    if (row_begin < 0 || row_end > rows || row_begin >= row_end)
        return fail(BICOS_B200_ERR_INVALID, "bad row range [%d, %d) of %d", row_begin, row_end, rows);
    sh.disparity_pitch = disparity_pitch;
    sh.corrmap_pitch = corrmap_pitch;
    Range nvtx_match("bicos_b200::match");
    Unit u;
    if (int rc = make_unit(u, planes0, planes1, sh, row_begin, row_end, disparity, corrmap))
        return rc;
    if (int rc = enter_workspace(h, stream))
        return rc;
    if (int rc = reserve_workspace(h, sh, u.nrows, false))
        return rc;
    uint32_t* keys = static_cast<uint32_t*>(h->keys.ptr);
    if (int rc = enqueue_search_stage(h, u, sh, keys, stream))
        return rc;
    if (int rc = enqueue_refine_stage(h, u, sh, keys, stream))
        return rc;
    h->stage_count += 1;
    return leave_workspace(h, stream);
}

// Units through two internal streams: transform + search of unit u + 1 (tensor pipe; high-priority stream, so that its
// one-CTA-per-SM grid is placed as soon as an SM has room) beside postfilter + refine of unit u (FP32 pipe). The
// search kernel holds 40 K of an SM's 64 K registers (search_mma.cu, setmaxnreg), which leaves room for one refine
// CTA; key arrays alternate between two buffers, descriptors need one (both their producer and their consumer are on
// the search stream). `stream` is joined on both sides: everything enqueued before this call is complete before the
// first unit starts, and `stream` continues after the last refine.
int run_pipeline(bicos_b200_handle h, const std::vector<Unit>& units, const MatchShape& sh, cudaStream_t stream) {
    if (!h->p_search) {
        int least = 0, greatest = 0;
        CU(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        CU(cudaStreamCreateWithPriority(&h->p_search, cudaStreamNonBlocking, greatest));
        CU(cudaStreamCreateWithPriority(&h->p_refine, cudaStreamNonBlocking, least));
        for (cudaEvent_t* e: { &h->p_start, &h->p_done, &h->p_searched[0], &h->p_searched[1], &h->p_refined[0], &h->p_refined[1] })
            CU(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    }
    if (int rc = enter_workspace(h, stream))
        return rc;
    int max_rows = 0;
    for (const Unit& u: units)
        max_rows = u.nrows > max_rows ? u.nrows : max_rows;
    if (int rc = reserve_workspace(h, sh, max_rows, true))
        return rc;
    uint32_t* const keys[2] = { static_cast<uint32_t*>(h->keys.ptr), static_cast<uint32_t*>(h->keys_b.ptr) };
    if (sh.cfg->subpixel_step >= 0 && has_thr(sh.cfg))
        if (int rc = prepare_steps(h, sh.cfg->subpixel_step, stream)) // before the fork: may synchronise `stream`
            return rc;
    CU(cudaEventRecord(h->p_start, stream));
    CU(cudaStreamWaitEvent(h->p_search, h->p_start, 0));
    CU(cudaStreamWaitEvent(h->p_refine, h->p_start, 0));
    for (size_t i = 0; i < units.size(); ++i) {
        const int slot = (int)(i & 1);
        if (i >= 2)
            CU(cudaStreamWaitEvent(h->p_search, h->p_refined[slot], 0)); // the refine that read this key buffer
        if (int rc = enqueue_search_stage(h, units[i], sh, keys[slot], h->p_search))
            return rc;
        CU(cudaEventRecord(h->p_searched[slot], h->p_search));
        CU(cudaStreamWaitEvent(h->p_refine, h->p_searched[slot], 0));
        if (int rc = enqueue_refine_stage(h, units[i], sh, keys[slot], h->p_refine))
            return rc;
        CU(cudaEventRecord(h->p_refined[slot], h->p_refine));
    }
    CU(cudaEventRecord(h->p_done, h->p_refine)); // in stream order after every refine, each after its search
    CU(cudaStreamWaitEvent(stream, h->p_done, 0));
    return leave_workspace(h, stream);
}

} // namespace

extern "C" {

const char* bicos_b200_last_error(void) {
    return g_error.c_str();
}

int bicos_b200_device_count(void) {
    int n = 0;
    cudaError_t err = cudaGetDeviceCount(&n);
    if (err != cudaSuccess)
        return cuda_fail(err, "cudaGetDeviceCount");
    return n;
}

int bicos_b200_create(bicos_b200_handle* out, int device) {
    if (!out)
        return fail(BICOS_B200_ERR_INVALID, "out is null");
    *out = nullptr;
    int count = 0;
    CU(cudaGetDeviceCount(&count));
    if (count <= 0)
        return fail(BICOS_B200_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
    if (device < 0)
        CU(cudaGetDevice(&device));
    if (device >= count)
        return fail(BICOS_B200_ERR_INVALID, "device %d out of range (%d visible)", device, count);
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(BICOS_B200_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    bicos_b200_handle h = new (std::nothrow) bicos_b200_handle_s();
    if (!h)
        return fail(BICOS_B200_ERR_NOMEM, "out of host memory");
    h->device = device;
    *out = h;
    return 0;
}

int bicos_b200_destroy(bicos_b200_handle h) {
    if (!h)
        return 0;
    {
        DeviceGuard g(h->device);
        cudaDeviceSynchronize();
        for (DeviceBuffer* b: { &h->desc0, &h->desc1, &h->keys, &h->xs, &h->stage_in, &h->stage_disp, &h->stage_corr, &h->rect, &h->reproj,
                                &h->speckle })
            b->release();
        for (cudaEvent_t e: h->prof_events)
            cudaEventDestroy(e);
        if (h->ev_last)
            cudaEventDestroy(h->ev_last);
        h->keys_b.release();
        for (cudaEvent_t e: { h->p_start, h->p_done, h->p_searched[0], h->p_searched[1], h->p_refined[0], h->p_refined[1] })
            if (e)
                cudaEventDestroy(e);
        for (cudaStream_t st: { h->p_search, h->p_refine })
            if (st)
                cudaStreamDestroy(st);
        for (int k = 0; k < PIN_SLOTS; ++k) {
            h->pin_in[k].release();
            if (h->ev_slot[k])
                cudaEventDestroy(h->ev_slot[k]);
        }
        h->pin_disp.release();
        h->pin_corr.release();
        for (int b = 0; b < MAX_BANDS; ++b) {
            if (h->ev_in[b])
                cudaEventDestroy(h->ev_in[b]);
            if (h->ev_done[b])
                cudaEventDestroy(h->ev_done[b]);
        }
        for (cudaStream_t st: { h->s_in, h->s_compute, h->s_out })
            if (st)
                cudaStreamDestroy(st);
    }
    delete h;
    return 0;
}

int bicos_b200_descriptor_words(int n, int mode) {
    if (n < 2)
        return fail(BICOS_B200_ERR_INVALID, "need at least two images");
    const int bits = descriptor_bits(n, mode_is_full(mode));
    const int K = words_for_bits(bits, (mode & BICOS_B200_MODE_WIDE) != 0);
    if (K < 0 || n > MAX_IMAGES)
        return fail(BICOS_B200_ERR_INVALID, "input stacks too large, would require %d bits", bits);
    return K;
}

int bicos_b200_disparity_type(const bicos_b200_config* cfg) {
    return has_thr(cfg) ? BICOS_B200_32F : BICOS_B200_16S;
}

int bicos_b200_corrmap_type(const bicos_b200_config* cfg) {
    if (!has_thr(cfg))
        return 0;
    return cfg->precision != 0 ? BICOS_B200_64F : BICOS_B200_32F;
}

int bicos_b200_transform(bicos_b200_handle h, const void* const* planes, int n, int rows, int cols,
                         size_t pitch_bytes, int depth, int mode, uint32_t* desc,
                         size_t desc_pitch_words, void* stream) {
    if (!h || !planes || !desc)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    bicos_b200_config cfg {};
    cfg.nxcorr_threshold = -1.f;
    cfg.mode = mode;
    int K = 0;
    if (int rc = validate_common(n, rows, cols, depth, &cfg, &K))
        return rc;
    if (desc_pitch_words < (size_t)cols * K || (desc_pitch_words % 4) != 0 || (reinterpret_cast<uintptr_t>(desc) % 16) != 0)
        return fail(BICOS_B200_ERR_INVALID, "descriptor rows must be 16-byte aligned and hold cols*K words");
    DeviceGuard g(h->device);
    PlaneTable t;
    if (int rc = fill_table(t, planes, n, 0))
        return rc;
    CU(launch_transform(t, n, rows, cols, pitch_bytes, depth == BICOS_B200_16U, mode_is_full(mode), K, desc, desc_pitch_words, static_cast<cudaStream_t>(stream)));
    h->launches += 1;
    return 0;
}

int bicos_b200_search(bicos_b200_handle h, const uint32_t* desc0, const uint32_t* desc1, int K,
                      int rows, int cols, size_t desc_pitch_words, int flags, uint32_t* fwd_first,
                      uint32_t* fwd_last, uint32_t* rev_first, uint32_t* rev_last, void* stream) {
    if (!h || !desc0 || !desc1 || !fwd_first)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    if (K != 1 && K != 2 && K != 4 && K != 8 && K != 12 && K != 16)
        return fail(BICOS_B200_ERR_INVALID, "K must be 1, 2, 4 or 8 (12 or 16 for wide descriptors)");
    if (flags < 0 || flags > 15)
        return fail(BICOS_B200_ERR_INVALID, "bad flags");
    const int free_top_bits = (flags & BICOS_B200_FLAG_TOP2_BITS_FREE) ? 2 : (flags & BICOS_B200_FLAG_TOP_BIT_FREE) ? 1 : 0;
    flags &= 3;
    if (rows <= 0 || cols <= 0 || cols > 32767)
        return fail(BICOS_B200_ERR_INVALID, "bad image size");
    if ((flags & FLAG_NODUPES) && !fwd_last)
        return fail(BICOS_B200_ERR_INVALID, "no-duplicates search needs fwd_last");
    if ((flags & FLAG_CONSISTENCY) && (!rev_first || ((flags & FLAG_NODUPES) && !rev_last)))
        return fail(BICOS_B200_ERR_INVALID, "consistency search needs rev_first (and rev_last with no_dupes)");
    if (desc_pitch_words < (size_t)cols * K || (desc_pitch_words % 4) != 0)
        return fail(BICOS_B200_ERR_INVALID, "descriptor rows must be 16-byte aligned and hold cols*K words");
    DeviceGuard g(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t bytes = (size_t)rows * cols * sizeof(uint32_t);
    if (search_needs_prefill(K, cols)) {
        CU(cudaMemsetAsync(fwd_first, 0xFF, bytes, s));
        if (flags & FLAG_NODUPES)
            CU(cudaMemsetAsync(fwd_last, 0xFF, bytes, s));
        if (flags & FLAG_CONSISTENCY) {
            CU(cudaMemsetAsync(rev_first, 0xFF, bytes, s));
            if (flags & FLAG_NODUPES)
                CU(cudaMemsetAsync(rev_last, 0xFF, bytes, s));
        }
    }
    CU(launch_search(desc0, desc1, K, rows, cols, desc_pitch_words, flags, fwd_first, fwd_last, rev_first, rev_last, s, free_top_bits));
    h->launches += 1;
    return 0;
}

int bicos_b200_search_range(bicos_b200_handle h, const uint32_t* desc0, const uint32_t* desc1, int K, int rows, int cols,
                            size_t desc_pitch_words, int flags, uint32_t* fwd_first, uint32_t* fwd_last, uint32_t* rev_first,
                            uint32_t* rev_last, int min_disparity, int max_disparity, void* stream) {
    if (min_disparity > max_disparity)
        return fail(BICOS_B200_ERR_INVALID, "disparity range [%d, %d]: min > max", min_disparity, max_disparity);
    if (cols <= 0 || !disparity_range_clip(cols, &min_disparity, &max_disparity))
        return bicos_b200_search(h, desc0, desc1, K, rows, cols, desc_pitch_words, flags, fwd_first, fwd_last, rev_first, rev_last,
                                 stream);
    if (!h || !desc0 || !desc1 || !fwd_first || !fwd_last)
        return fail(BICOS_B200_ERR_INVALID, "null argument (a ranged search always needs fwd_last)");
    if (K != 1 && K != 2 && K != 4 && K != 8 && K != 12 && K != 16)
        return fail(BICOS_B200_ERR_INVALID, "K must be 1, 2, 4 or 8 (12 or 16 for wide descriptors)");
    if (flags < 0 || flags > 15)
        return fail(BICOS_B200_ERR_INVALID, "bad flags");
    flags &= 3; // the top-bit promises only matter to the tensor-core engine
    if (rows <= 0 || rows > 65535 || cols > 32767)
        return fail(BICOS_B200_ERR_INVALID, "bad image size");
    if ((flags & FLAG_CONSISTENCY) && (!rev_first || ((flags & FLAG_NODUPES) && !rev_last)))
        return fail(BICOS_B200_ERR_INVALID, "consistency search needs rev_first (and rev_last with no_dupes)");
    if (desc_pitch_words < (size_t)cols * K || (desc_pitch_words % 4) != 0)
        return fail(BICOS_B200_ERR_INVALID, "descriptor rows must be 16-byte aligned and hold cols*K words");
    if (int rc = check_range_engine())
        return rc;
    DeviceGuard g(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t bytes = (size_t)rows * cols * sizeof(uint32_t);
    if (flags & FLAG_CONSISTENCY) {
        CU(cudaMemsetAsync(rev_first, 0xFF, bytes, s));
        if (flags & FLAG_NODUPES)
            CU(cudaMemsetAsync(rev_last, 0xFF, bytes, s));
    }
    CU(launch_search_range(desc0, desc1, K, rows, cols, desc_pitch_words, flags, min_disparity, max_disparity, fwd_first, fwd_last,
                           rev_first, rev_last, s));
    h->launches += 1;
    return 0;
}

int bicos_b200_search_windows(bicos_b200_handle h, const uint32_t* desc0, const uint32_t* desc1, int K, int rows, int cols,
                              size_t desc_pitch_words, int flags, uint32_t* fwd_first, uint32_t* fwd_last, uint32_t* rev_first,
                              uint32_t* rev_last, const bicos_b200_disparity_windows* windows, void* stream) {
    if (!h || !desc0 || !desc1 || !fwd_first || !fwd_last)
        return fail(BICOS_B200_ERR_INVALID, "null argument (a windowed search always needs fwd_last)");
    if (K != 1 && K != 2 && K != 4 && K != 8 && K != 12 && K != 16)
        return fail(BICOS_B200_ERR_INVALID, "K must be 1, 2, 4 or 8 (12 or 16 for wide descriptors)");
    if (flags < 0 || flags > 15)
        return fail(BICOS_B200_ERR_INVALID, "bad flags");
    flags &= 3; // the top-bit promises only matter to the tensor-core engine
    if (rows <= 0 || rows > 65535 || cols <= 0 || cols > 32767)
        return fail(BICOS_B200_ERR_INVALID, "bad image size");
    if ((flags & FLAG_CONSISTENCY) && (!rev_first || ((flags & FLAG_NODUPES) && !rev_last)))
        return fail(BICOS_B200_ERR_INVALID, "consistency search needs rev_first (and rev_last with no_dupes)");
    if (desc_pitch_words < (size_t)cols * K || (desc_pitch_words % 4) != 0)
        return fail(BICOS_B200_ERR_INVALID, "descriptor rows must be 16-byte aligned and hold cols*K words");
    if (int rc = validate_windows(windows, cols))
        return rc;
    if (int rc = check_range_engine())
        return rc;
    DeviceGuard g(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t bytes = (size_t)rows * cols * sizeof(uint32_t);
    if (flags & FLAG_CONSISTENCY) {
        CU(cudaMemsetAsync(rev_first, 0xFF, bytes, s));
        if (flags & FLAG_NODUPES)
            CU(cudaMemsetAsync(rev_last, 0xFF, bytes, s));
    }
    CU(launch_search_windows(desc0, desc1, K, rows, cols, desc_pitch_words, flags, windows->min_disparity, windows->max_disparity,
                             windows->pitch_bytes / 2, fwd_first, fwd_last, rev_first, rev_last, s));
    h->launches += 1;
    return 0;
}

int bicos_b200_refine(bicos_b200_handle h, const void* const* planes0, const void* const* planes1,
                      int n, int rows, int cols, size_t pitch_bytes, int depth,
                      const bicos_b200_config* cfg, const uint32_t* fwd_first, const uint32_t* fwd_last,
                      const uint32_t* rev_first, const uint32_t* rev_last, int16_t* raw_disp_out,
                      void* disparity, size_t disparity_pitch_bytes, void* corrmap,
                      size_t corrmap_pitch_bytes, void* stream) {
    if (!h || !planes0 || !planes1 || !fwd_first || !disparity)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    if (int rc = validate_common(n, rows, cols, depth, cfg, nullptr))
        return rc;
    int dmin = 0, dmax = 0;
    if ((search_flags(cfg) & FLAG_NODUPES) && !fwd_last)
        return fail(BICOS_B200_ERR_INVALID, "no-duplicates postfilter needs fwd_last");
    if (cfg_range(cfg, cols, &dmin, &dmax) && !fwd_last)
        return fail(BICOS_B200_ERR_INVALID, "a ranged postfilter needs fwd_last (bicos_b200_search_range)");
    if (cfg->variant_type != 0 && (!rev_first || (cfg->no_dupes && !rev_last)))
        return fail(BICOS_B200_ERR_INVALID, "consistency postfilter needs rev_first (and rev_last with no_dupes)");
    DeviceGuard g(h->device);
    PlaneTable t0, t1;
    if (int rc = fill_table(t0, planes0, n, 0))
        return rc;
    if (int rc = fill_table(t1, planes1, n, 0))
        return rc;
    return do_refine(h, t0, t1, n, rows, cols, pitch_bytes, depth, cfg, fwd_first, fwd_last, rev_first, rev_last,
                     raw_disp_out, disparity, disparity_pitch_bytes, corrmap, corrmap_pitch_bytes,
                     static_cast<cudaStream_t>(stream));
}

// A single match of a large image with the subpixel refine (the FP32-heavy one): as row bands through the two-stream
// pipeline, band b + 1's search beside band b's refine. Rows are independent, so the result is the same. Measured with
// tools/overlap_probe.py --frames 1: 1536 rows 2.01 ms as one unit, 1.93 / 1.91 / 1.91 ms as 2 / 3 / 4 bands; 768 rows
// (a shard of a two-GPU match) 1.025 -> 0.991 / 0.989 ms as 2 / 3 bands; 384 rows: no gain. Small images, integer
// refinement, the popcount engine (which leaves no issue slots free) and ranged matches run as one unit.
static int match_banded_or_whole(bicos_b200_handle h, const void* const* planes0, const void* const* planes1, int n, int rows,
                                 int cols, size_t pitch_bytes, int depth, const bicos_b200_config* cfg, void* disparity,
                                 size_t disparity_pitch, void* corrmap, size_t corrmap_pitch, cudaStream_t stream) {
    const int BANDS = rows >= 1152 ? 3 : 2;
    constexpr int MIN_BAND_ROWS = 320;
    MatchShape sh {};
    if (int rc = validate_match(planes0, planes1, n, rows, cols, pitch_bytes, depth, cfg, disparity, sh))
        return rc;
    const bool subpixel = has_thr(cfg) && cfg->subpixel_step >= 0;
    // the one-pass consistency search takes its SM's whole register file: nothing runs beside it, and bands would only add
    // launches (1.71 against 1.63 ms on the metric configuration)
    const bool onepass = search_engine() != 1 && search_mma_supports(sh.K, cols) && search_mma_onepass_applies(sh.K, cols, sh.flags, 2);
    if (!h->overlap || !subpixel || onepass || sh.ranged || rows < BANDS * MIN_BAND_ROWS || search_needs_prefill(sh.K, cols) ||
        (sh.K != 4 && sh.K != 8))
        return do_match(h, planes0, planes1, n, rows, cols, pitch_bytes, depth, cfg, 0, rows, disparity, disparity_pitch, corrmap,
                        corrmap_pitch, stream);
    sh.disparity_pitch = disparity_pitch;
    sh.corrmap_pitch = corrmap_pitch;
    std::vector<Unit> units((size_t)BANDS);
    for (int b = 0; b < BANDS; ++b)
        if (int rc = make_unit(units[(size_t)b], planes0, planes1, sh, (int)((long long)rows * b / BANDS),
                               (int)((long long)rows * (b + 1) / BANDS), disparity, corrmap))
            return rc;
    Range nvtx("bicos_b200::match (banded)");
    if (int rc = run_pipeline(h, units, sh, stream))
        return rc;
    h->stage_count += 1;
    return 0;
}

int bicos_b200_match(bicos_b200_handle h, const void* const* planes0, const void* const* planes1,
                     int n, int rows, int cols, size_t pitch_bytes, int depth,
                     const bicos_b200_config* cfg, void* disparity, size_t disparity_pitch_bytes,
                     void* corrmap, size_t corrmap_pitch_bytes, void* stream) {
    if (!h)
        return fail(BICOS_B200_ERR_INVALID, "null handle");
    DeviceGuard g(h->device);
    return match_banded_or_whole(h, planes0, planes1, n, rows, cols, pitch_bytes, depth, cfg, disparity,
                                 disparity_pitch_bytes, corrmap, corrmap_pitch_bytes, static_cast<cudaStream_t>(stream));
}

int bicos_b200_match_windows(bicos_b200_handle h, const void* const* planes0, const void* const* planes1, int n, int rows,
                             int cols, size_t pitch_bytes, int depth, const bicos_b200_config* cfg,
                             const bicos_b200_disparity_windows* windows, void* disparity, size_t disparity_pitch_bytes,
                             void* corrmap, size_t corrmap_pitch_bytes, void* stream) {
    if (!h)
        return fail(BICOS_B200_ERR_INVALID, "null handle");
    if (!windows)
        return fail(BICOS_B200_ERR_INVALID, "disparity windows are null");
    DeviceGuard g(h->device);
    return do_match(h, planes0, planes1, n, rows, cols, pitch_bytes, depth, cfg, 0, rows, disparity, disparity_pitch_bytes, corrmap,
                    corrmap_pitch_bytes, static_cast<cudaStream_t>(stream), windows);
}

int bicos_b200_windows_from_disparity(bicos_b200_handle h, const void* prior, int prior_type, size_t prior_pitch_bytes, int rows,
                                      int cols, int margin, int fallback_min, int fallback_max, int16_t* min_out,
                                      int16_t* max_out, size_t windows_pitch_bytes, void* stream) {
    if (!h || !prior || !min_out || !max_out)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    if (prior_type != BICOS_B200_16S && prior_type != BICOS_B200_32F)
        return fail(BICOS_B200_ERR_INVALID, "bad prior type %d: only int16 (CV_16SC1) and float32 (CV_32FC1)", prior_type);
    if (rows < 1 || cols < 1 || rows > 65535 || cols > 32767)
        return fail(BICOS_B200_ERR_INVALID, "prior of %d x %d: rows 1 to 65535, cols 1 to 32767", rows, cols);
    const size_t es = prior_type == BICOS_B200_16S ? 2 : 4;
    if (prior_pitch_bytes < (size_t)cols * es || prior_pitch_bytes % es != 0 || reinterpret_cast<uintptr_t>(prior) % es != 0)
        return fail(BICOS_B200_ERR_INVALID, "prior rows must be aligned to and hold cols elements");
    if (margin < 0 || margin > 32767)
        return fail(BICOS_B200_ERR_INVALID, "margin %d outside 0..32767", margin);
    if (fallback_min < -32768 || fallback_min > 32767 || fallback_max < -32768 || fallback_max > 32767)
        return fail(BICOS_B200_ERR_INVALID, "fallback window [%d, %d] outside int16", fallback_min, fallback_max);
    const bicos_b200_disparity_windows w { min_out, max_out, windows_pitch_bytes };
    if (int rc = validate_windows(&w, cols))
        return rc;
    DeviceGuard g(h->device);
    WindowsParams prm {};
    prm.prior = prior;
    prm.prior_pitch = prior_pitch_bytes;
    prm.rows = rows;
    prm.cols = cols;
    prm.margin = margin;
    prm.fallback_min = fallback_min;
    prm.fallback_max = fallback_max;
    prm.min_out = min_out;
    prm.max_out = max_out;
    prm.out_pitch = windows_pitch_bytes / 2;
    {
        Range nvtx("bicos_b200::windows_from_disparity");
        CU(launch_windows_from_disparity(prm, prior_type == BICOS_B200_32F, static_cast<cudaStream_t>(stream)));
        h->launches += 1;
    }
    return 0;
}

// checks shared by bicos_b200_remap and bicos_b200_match_rectified
static int validate_remap(int n, int src_rows, int src_cols, size_t src_pitch_bytes, int depth, const float* map_x,
                          const float* map_y, size_t map_pitch_bytes, int rows, int cols) {
    if (depth != BICOS_B200_8U && depth != BICOS_B200_16U)
        return fail(BICOS_B200_ERR_INVALID, "bad input depths, only CV_8UC1 and CV_16UC1 are supported");
    if (n < 1 || n > MAX_IMAGES)
        return fail(BICOS_B200_ERR_INVALID, "remap of %d planes: 1 to %d are supported", n, MAX_IMAGES);
    if (!map_x || !map_y)
        return fail(BICOS_B200_ERR_INVALID, "rectification map is null");
    if (src_rows <= 0 || src_cols <= 0 || rows <= 0 || cols <= 0)
        return fail(BICOS_B200_ERR_INVALID, "empty images");
    if (src_rows > 32767 || src_cols > 32767 || rows > 32767 || cols > 32767)
        return fail(BICOS_B200_ERR_INVALID, "image too large: remap source and output have at most 32767 rows and columns");
    if (src_pitch_bytes < (size_t)src_cols * depth_bytes(depth))
        return fail(BICOS_B200_ERR_INVALID, "source pitch smaller than a row");
    if (map_pitch_bytes < (size_t)cols * sizeof(float) || map_pitch_bytes % sizeof(float) != 0 ||
        reinterpret_cast<uintptr_t>(map_x) % sizeof(float) != 0 || reinterpret_cast<uintptr_t>(map_y) % sizeof(float) != 0)
        return fail(BICOS_B200_ERR_INVALID, "map rows must be 4-byte aligned and hold cols float32 values");
    return 0;
}

int bicos_b200_remap(bicos_b200_handle h, const void* const* src_planes, int n, int src_rows, int src_cols,
                     size_t src_pitch_bytes, int depth, const float* map_x, const float* map_y, size_t map_pitch_bytes,
                     int rows, int cols, void* const* dst_planes, size_t dst_pitch_bytes, void* stream) {
    if (!h || !src_planes || !dst_planes)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    if (int rc = validate_remap(n, src_rows, src_cols, src_pitch_bytes, depth, map_x, map_y, map_pitch_bytes, rows, cols))
        return rc;
    if (dst_pitch_bytes < (size_t)cols * depth_bytes(depth))
        return fail(BICOS_B200_ERR_INVALID, "output pitch smaller than a row");
    DeviceGuard g(h->device);
    RemapParams prm {};
    if (int rc = fill_table(prm.side[0].src, src_planes, n, 0))
        return rc;
    if (int rc = fill_table(prm.side[0].dst, dst_planes, n, 0))
        return rc;
    prm.side[0].map_x = map_x;
    prm.side[0].map_y = map_y;
    prm.n = n;
    prm.src_rows = src_rows;
    prm.src_cols = src_cols;
    prm.rows = rows;
    prm.cols = cols;
    prm.src_pitch = src_pitch_bytes;
    prm.map_pitch = map_pitch_bytes;
    prm.dst_pitch = dst_pitch_bytes;
    CU(launch_remap(prm, 1, depth == BICOS_B200_16U, static_cast<cudaStream_t>(stream)));
    h->launches += 1;
    return 0;
}

int bicos_b200_match_rectified(bicos_b200_handle h, const void* const* planes0, const void* const* planes1, int n,
                               int src_rows, int src_cols, size_t src_pitch_bytes, int depth,
                               const bicos_b200_rectify_maps* maps, int rows, int cols, const bicos_b200_config* cfg,
                               void* disparity, size_t disparity_pitch_bytes, void* corrmap, size_t corrmap_pitch_bytes,
                               void* stream) {
    if (!h)
        return fail(BICOS_B200_ERR_INVALID, "null handle");
    if (!maps)
        return fail(BICOS_B200_ERR_INVALID, "rectification maps are null");
    const size_t pitch = ((size_t)cols * depth_bytes(depth) + 127) & ~(size_t)127; // rectified planes in the workspace
    // everything the match would reject at the rectified size is rejected before the remap is enqueued
    MatchShape sh {};
    if (int rc = validate_match(planes0, planes1, n, rows, cols, pitch, depth, cfg, disparity, sh))
        return rc;
    for (int side = 0; side < 2; ++side)
        if (int rc = validate_remap(n, src_rows, src_cols, src_pitch_bytes, depth, side ? maps->map_x1 : maps->map_x0,
                                    side ? maps->map_y1 : maps->map_y0, maps->map_pitch_bytes, rows, cols))
            return rc;
    DeviceGuard g(h->device);
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    RemapParams prm {};
    if (int rc = fill_table(prm.side[0].src, planes0, n, 0))
        return rc;
    if (int rc = fill_table(prm.side[1].src, planes1, n, 0))
        return rc;
    if (int rc = enter_workspace(h, s)) // the previous match of the handle may still read the rectified planes
        return rc;
    const size_t plane_bytes = pitch * (size_t)rows;
    CU(h->rect.reserve(plane_bytes * 2 * (size_t)n));
    std::vector<const void*> rect0((size_t)n), rect1((size_t)n);
    for (int i = 0; i < n; ++i) {
        rect0[(size_t)i] = static_cast<char*>(h->rect.ptr) + plane_bytes * (size_t)i;
        rect1[(size_t)i] = static_cast<char*>(h->rect.ptr) + plane_bytes * (size_t)(n + i);
    }
    fill_table(prm.side[0].dst, rect0.data(), n, 0);
    fill_table(prm.side[1].dst, rect1.data(), n, 0);
    prm.side[0].map_x = maps->map_x0;
    prm.side[0].map_y = maps->map_y0;
    prm.side[1].map_x = maps->map_x1;
    prm.side[1].map_y = maps->map_y1;
    prm.n = n;
    prm.src_rows = src_rows;
    prm.src_cols = src_cols;
    prm.rows = rows;
    prm.cols = cols;
    prm.src_pitch = src_pitch_bytes;
    prm.map_pitch = maps->map_pitch_bytes;
    prm.dst_pitch = pitch;
    {
        Range nvtx("bicos_b200::remap x2");
        CU(launch_remap(prm, 2, depth == BICOS_B200_16U, s));
        h->launches += 1;
    }
    return match_banded_or_whole(h, rect0.data(), rect1.data(), n, rows, cols, pitch, depth, cfg, disparity, disparity_pitch_bytes,
                                 corrmap, corrmap_pitch_bytes, s);
}

int bicos_b200_reproject(bicos_b200_handle h, const void* disparity, int disparity_type, size_t disparity_pitch_bytes,
                         int rows, int cols, const double q[16], int flags, float* xyz, size_t xyz_pitch_bytes,
                         float* points, int32_t* pixel_index, unsigned long long* counts, void* stream) {
    if (!h || !q || !disparity)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    if (disparity_type != BICOS_B200_16S && disparity_type != BICOS_B200_32F)
        return fail(BICOS_B200_ERR_INVALID, "bad disparity type %d: only int16 (CV_16SC1) and float32 (CV_32FC1)", disparity_type);
    if ((flags & ~BICOS_B200_REPROJECT_ALLOW_NEGATIVE_Z) != 0)
        return fail(BICOS_B200_ERR_INVALID, "unknown reprojection flags %#x", flags);
    if (!xyz && !points)
        return fail(BICOS_B200_ERR_INVALID, "no output: give xyz, points, or both");
    if (points && !counts)
        return fail(BICOS_B200_ERR_INVALID, "points need counts");
    if (pixel_index && !points)
        return fail(BICOS_B200_ERR_INVALID, "pixel_index needs points");
    if (rows < 1 || cols < 1 || rows > 32767 || cols > 32767)
        return fail(BICOS_B200_ERR_INVALID, "disparity of %d x %d: rows and cols must be 1 to 32767", rows, cols);
    const size_t es = disparity_type == BICOS_B200_16S ? 2 : 4;
    if (disparity_pitch_bytes < (size_t)cols * es || disparity_pitch_bytes % es != 0 || reinterpret_cast<uintptr_t>(disparity) % es != 0)
        return fail(BICOS_B200_ERR_INVALID, "disparity rows must be aligned to and hold cols elements");
    if (xyz && (xyz_pitch_bytes < (size_t)cols * 3 * sizeof(float) || xyz_pitch_bytes % sizeof(float) != 0 ||
                reinterpret_cast<uintptr_t>(xyz) % sizeof(float) != 0))
        return fail(BICOS_B200_ERR_INVALID, "xyz rows must be 4-byte aligned and hold cols * 3 float32 values");
    if ((points && reinterpret_cast<uintptr_t>(points) % sizeof(float) != 0) ||
        (pixel_index && reinterpret_cast<uintptr_t>(pixel_index) % sizeof(int32_t) != 0) ||
        (counts && reinterpret_cast<uintptr_t>(counts) % sizeof(unsigned long long) != 0))
        return fail(BICOS_B200_ERR_INVALID, "misaligned points, pixel_index or counts");
    DeviceGuard g(h->device);
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    ReprojectParams prm {};
    prm.disparity = disparity;
    prm.disparity_pitch = disparity_pitch_bytes;
    prm.rows = rows;
    prm.cols = cols;
    for (int k = 0; k < 16; ++k)
        prm.q[k] = q[k];
    prm.allow_negative_z = (flags & BICOS_B200_REPROJECT_ALLOW_NEGATIVE_Z) ? 1 : 0;
    prm.xyz = xyz;
    prm.xyz_pitch = xyz_pitch_bytes;
    prm.points = points;
    prm.pixel_index = pixel_index;
    prm.counts = counts;
    if (int rc = enter_workspace(h, s)) // the previous call of the handle may still use the status words
        return rc;
    if (counts) {
        const size_t work_bytes = sizeof(ReprojectWork) + sizeof(unsigned long long) * (size_t)reproject_tiles(rows, cols);
        CU(h->reproj.reserve(work_bytes));
        CU(cudaMemsetAsync(h->reproj.ptr, 0, work_bytes, s));
        prm.work = static_cast<ReprojectWork*>(h->reproj.ptr);
        prm.status = reinterpret_cast<unsigned long long*>(prm.work + 1);
    }
    {
        Range nvtx("bicos_b200::reproject");
        CU(launch_reproject(prm, disparity_type == BICOS_B200_32F, s));
        h->launches += 1;
    }
    return leave_workspace(h, s);
}

int bicos_b200_filter_speckles(bicos_b200_handle h, void* disparity, int disparity_type, size_t disparity_pitch_bytes, int rows,
                               int cols, double new_value, int max_speckle_size, double max_diff, unsigned long long* counts,
                               void* stream) {
    if (!h || !disparity)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    if (disparity_type != BICOS_B200_16S && disparity_type != BICOS_B200_32F)
        return fail(BICOS_B200_ERR_INVALID, "bad disparity type %d: only int16 (CV_16SC1) and float32 (CV_32FC1)", disparity_type);
    if (rows < 1 || cols < 1 || rows > 32767 || cols > 32767)
        return fail(BICOS_B200_ERR_INVALID, "disparity of %d x %d: rows and cols must be 1 to 32767", rows, cols);
    const size_t es = disparity_type == BICOS_B200_16S ? 2 : 4;
    if (disparity_pitch_bytes < (size_t)cols * es || disparity_pitch_bytes % es != 0 || reinterpret_cast<uintptr_t>(disparity) % es != 0)
        return fail(BICOS_B200_ERR_INVALID, "disparity rows must be aligned to and hold cols elements");
    if (std::isnan(max_diff))
        return fail(BICOS_B200_ERR_INVALID, "max_diff is NaN");
    if (counts && reinterpret_cast<uintptr_t>(counts) % sizeof(unsigned long long) != 0)
        return fail(BICOS_B200_ERR_INVALID, "misaligned counts");
    SpeckleParams prm {};
    if (disparity_type == BICOS_B200_16S) {
        // cvRound: to nearest, half to even (the default rounding mode)
        const double nv = std::nearbyint(new_value), nd = std::nearbyint(max_diff);
        if (!(nv >= -32768.0 && nv <= 32767.0))
            return fail(BICOS_B200_ERR_INVALID, "new_value %g does not round into int16", new_value);
        prm.new_i = (int)nv;
        prm.diff_i = (int)std::fmax(-65535.0, std::fmin(65535.0, nd)); // int16 differences lie within +-65535
    } else {
        prm.new_f = (float)new_value;
        prm.diff_f = (float)max_diff;
    }
    prm.disparity = disparity;
    prm.disparity_pitch = disparity_pitch_bytes;
    prm.rows = rows;
    prm.cols = cols;
    prm.max_size = max_speckle_size;
    prm.counts = counts;
    DeviceGuard g(h->device);
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (int rc = enter_workspace(h, s)) // the previous call of the handle may still use the labels
        return rc;
    const size_t px = (size_t)rows * cols;
    CU(h->speckle.reserve(2 * px * sizeof(int)));
    prm.parent = static_cast<int*>(h->speckle.ptr);
    prm.size = prm.parent + px;
    if (counts)
        CU(cudaMemsetAsync(counts, 0, 2 * sizeof(unsigned long long), s));
    {
        Range nvtx("bicos_b200::filter_speckles");
        CU(launch_speckles(prm, disparity_type == BICOS_B200_32F, s));
        h->launches += 4;
    }
    return leave_workspace(h, s);
}

int bicos_b200_match_rows(bicos_b200_handle h, const void* const* planes0,
                          const void* const* planes1, int n, int rows, int cols, size_t pitch_bytes,
                          int depth, const bicos_b200_config* cfg, int row_begin, int row_end,
                          void* disparity, size_t disparity_pitch_bytes, void* corrmap,
                          size_t corrmap_pitch_bytes, void* stream) {
    if (!h)
        return fail(BICOS_B200_ERR_INVALID, "null handle");
    DeviceGuard g(h->device);
    return do_match(h, planes0, planes1, n, rows, cols, pitch_bytes, depth, cfg, row_begin, row_end, disparity,
                    disparity_pitch_bytes, corrmap, corrmap_pitch_bytes, static_cast<cudaStream_t>(stream));
}

int bicos_b200_match_batch(bicos_b200_handle h, int count, const void* const* const* planes0,
                           const void* const* const* planes1, int n, int rows, int cols, size_t pitch_bytes,
                           int depth, const bicos_b200_config* cfg, void* const* disparity,
                           size_t disparity_pitch_bytes, void* const* corrmap, size_t corrmap_pitch_bytes,
                           void* stream) {
    if (!h)
        return fail(BICOS_B200_ERR_INVALID, "null handle");
    if (count <= 0 || !planes0 || !planes1 || !disparity)
        return fail(BICOS_B200_ERR_INVALID, "empty batch or null argument");
    DeviceGuard g(h->device);
    MatchShape sh {};
    std::vector<Unit> units((size_t)count);
    for (int f = 0; f < count; ++f) {
        if (int rc = validate_match(planes0[f], planes1[f], n, rows, cols, pitch_bytes, depth, cfg, disparity[f], sh))
            return rc;
        sh.disparity_pitch = disparity_pitch_bytes;
        sh.corrmap_pitch = corrmap_pitch_bytes;
        if (int rc = make_unit(units[(size_t)f], planes0[f], planes1[f], sh, 0, rows, disparity[f], corrmap ? corrmap[f] : nullptr))
            return rc;
    }
    Range nvtx("bicos_b200::match_batch");
    if (!h->overlap) {
        for (int f = 0; f < count; ++f)
            if (int rc = do_match(h, planes0[f], planes1[f], n, rows, cols, pitch_bytes, depth, cfg, 0, rows, disparity[f],
                                  disparity_pitch_bytes, corrmap ? corrmap[f] : nullptr, corrmap_pitch_bytes, static_cast<cudaStream_t>(stream)))
                return rc;
        return 0;
    }
    if (int rc = run_pipeline(h, units, sh, static_cast<cudaStream_t>(stream)))
        return rc;
    h->stage_count += count;
    return 0;
}

int bicos_b200_set_overlap(bicos_b200_handle h, int enabled) {
    if (!h)
        return fail(BICOS_B200_ERR_INVALID, "null handle");
    h->overlap = enabled != 0;
    return 0;
}

// dense host planes that lie back to back in one allocation ([n][rows][cols], e.g. one numpy
// array) can be uploaded band-wise with one strided 3-D copy instead of n 2-D copies
static bool planes_contiguous(const void* const* planes, int n, size_t plane_bytes) {
    for (int i = 1; i < n; ++i)
        if (static_cast<const char*>(planes[i]) != static_cast<const char*>(planes[0]) + plane_bytes * i)
            return false;
    return true;
}

static cudaError_t upload_band(const void* const* host_planes, bool contiguous, char* dev_base, int n, int rows,
                               size_t row_bytes, size_t pitch, int rb, int re, cudaStream_t stream) {
    if (contiguous) {
        cudaMemcpy3DParms p {};
        p.srcPtr = make_cudaPitchedPtr(const_cast<void*>(host_planes[0]), row_bytes, row_bytes, (size_t)rows);
        p.srcPos = make_cudaPos(0, (size_t)rb, 0);
        p.dstPtr = make_cudaPitchedPtr(dev_base, pitch, row_bytes, (size_t)rows);
        p.dstPos = make_cudaPos(0, (size_t)rb, 0);
        p.extent = make_cudaExtent(row_bytes, (size_t)(re - rb), (size_t)n);
        p.kind = cudaMemcpyHostToDevice;
        return cudaMemcpy3DAsync(&p, stream);
    }
    for (int i = 0; i < n; ++i) {
        cudaError_t err = cudaMemcpy2DAsync(dev_base + pitch * rows * i + pitch * rb, pitch,
                                            static_cast<const char*>(host_planes[i]) + row_bytes * rb, row_bytes,
                                            row_bytes, (size_t)(re - rb), cudaMemcpyHostToDevice, stream);
        if (err != cudaSuccess)
            return err;
    }
    return cudaSuccess;
}

int bicos_b200_match_host_begin(bicos_b200_handle h, const void* const* host_planes0,
                                const void* const* host_planes1, int n, int rows, int cols, int depth,
                                const bicos_b200_config* cfg, void* host_disparity, void* host_corrmap) {
    if (!h || !host_planes0 || !host_planes1 || !host_disparity)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    if (h->host_pending)
        return fail(BICOS_B200_ERR_INVALID, "a host match is already in flight on this handle: call bicos_b200_match_host_end first");
    if (int rc = validate_common(n, rows, cols, depth, cfg, nullptr))
        return rc;
    for (int i = 0; i < n; ++i)
        if (!host_planes0[i] || !host_planes1[i])
            return fail(BICOS_B200_ERR_INVALID, "image %d is null", i);
    DeviceGuard g(h->device);
    Range nvtx_host("bicos_b200::match_host_begin");

    // Rows are independent, so the image is cut into row bands that flow through three
    // streams: band b+1 uploads while band b is matched and band b-1 downloads. With pinned
    // host memory the copies are plain DMA; pageable memory still works (staged by the driver).
    if (!h->s_in) {
        CU(cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&h->s_compute, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
        for (int b = 0; b < MAX_BANDS; ++b) {
            CU(cudaEventCreateWithFlags(&h->ev_in[b], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&h->ev_done[b], cudaEventDisableTiming));
        }
    }
    // Band boundaries: about 192 rows each (measured best at 2048 columns, 96 .. 768 tried), with
    // a short first band so that the first kernels start early and a short last band so that
    // little work trails the last upload.
    int cut[MAX_BANDS + 1];
    int bands = 0;
    {
        static const int band_rows = [] { // BICOS_B200_HOST_BAND_ROWS: for sweeps of the host pipeline
            const char* v = getenv("BICOS_B200_HOST_BAND_ROWS");
            const int r = v ? atoi(v) : 0;
            return r >= 16 ? r : 192;
        }();
        int inner = rows / band_rows;
        inner = inner < 1 ? 1 : inner > MAX_BANDS - 2 ? MAX_BANDS - 2 : inner;
        const int edge = rows >= 4 * band_rows ? 64 : 0; // only worth it when there are several bands anyway
        cut[bands++] = 0;
        if (edge)
            cut[bands++] = edge;
        for (int b = 1; b < inner; ++b)
            cut[bands++] = edge + (int)((long long)(rows - 2 * edge) * b / inner);
        if (edge)
            cut[bands++] = rows - edge;
        cut[bands] = rows;
    }

    const size_t eb = depth_bytes(depth);
    const size_t row_bytes = (size_t)cols * eb;
    const size_t pitch = (row_bytes + 15) & ~(size_t)15;
    const size_t plane_bytes = pitch * rows;
    const size_t disp_eb = has_thr(cfg) ? 4 : 2;
    const size_t corr_eb = cfg->precision != 0 ? 8 : 4;
    const bool want_corr = host_corrmap && has_thr(cfg);
    int band_rows_max = 1;
    for (int b = 0; b < bands; ++b)
        band_rows_max = cut[b + 1] - cut[b] > band_rows_max ? cut[b + 1] - cut[b] : band_rows_max;
    {
        // reserve everything up front: a reallocation inside the pipeline would stall it
        int K = 0;
        validate_common(n, rows, cols, depth, cfg, &K);
        const size_t dpw = desc_pitch_for(cols, K);
        const size_t px = (size_t)band_rows_max * cols;
        CU(h->stage_in.reserve(plane_bytes * 2 * n));
        CU(h->stage_disp.reserve((size_t)rows * cols * disp_eb));
        if (want_corr)
            CU(h->stage_corr.reserve((size_t)rows * cols * corr_eb));
        CU(h->desc0.reserve(dpw * band_rows_max * sizeof(uint32_t)));
        CU(h->desc1.reserve(dpw * band_rows_max * sizeof(uint32_t)));
        CU(h->keys.reserve(px * sizeof(uint32_t) * 4));
        if (has_thr(cfg) && cfg->subpixel_step >= 0)
            if (int rc = prepare_steps(h, cfg->subpixel_step, h->s_compute))
                return rc;
    }

    std::vector<const void*> dev0(n), dev1(n);
    char* base = static_cast<char*>(h->stage_in.ptr);
    for (int i = 0; i < n; ++i) {
        dev0[i] = base + plane_bytes * i;
        dev1[i] = base + plane_bytes * (n + i);
    }
    const bool contig0 = planes_contiguous(host_planes0, n, row_bytes * rows);
    const bool contig1 = planes_contiguous(host_planes1, n, row_bytes * rows);

    // Pageable caller memory (numpy arrays, malloc: what pybicos' BICOS_Match passes) cannot be
    // handed to the DMA engines; the driver would stage it through a small bounce buffer at about
    // 8 GB/s. Instead a few host threads copy band b into a ring of pinned band buffers while the
    // GPU works on band b-1, and the results come back through pinned images that _end copies out.
    const bool stage_inputs = is_pageable(host_planes0[0]) || is_pageable(host_planes1[0]);
    const bool stage_disp = is_pageable(host_disparity);
    const bool stage_corr = want_corr && is_pageable(host_corrmap);
    const size_t slot_plane = row_bytes * band_rows_max; // one plane's band, dense
    if (stage_inputs)
        for (int k = 0; k < PIN_SLOTS; ++k) {
            CU(h->pin_in[k].reserve(slot_plane * 2 * n));
            if (!h->ev_slot[k])
                CU(cudaEventCreateWithFlags(&h->ev_slot[k], cudaEventDisableTiming | cudaEventBlockingSync));
        }
    if (stage_disp)
        CU(h->pin_disp.reserve((size_t)rows * cols * disp_eb));
    if (stage_corr)
        CU(h->pin_corr.reserve((size_t)rows * cols * corr_eb));
    char* const out_disp = static_cast<char*>(stage_disp ? h->pin_disp.ptr : host_disparity);
    char* const out_corr = static_cast<char*>(stage_corr ? h->pin_corr.ptr : host_corrmap);

    // Diagnostic build only (-DBICOS_B200_HOST_PROBE, tools/e2e_probe.py): the environment variable of the same name
    // takes the kernels ("nocompute") and / or the result downloads ("nod2h") out of the pipeline, to see which part
    // of the host link a many-GPU job loses where (profiles/r02_e2e_probe_n8.jsonl). Compiled out of the product.
#ifdef BICOS_B200_HOST_PROBE
    static const char* probe = getenv("BICOS_B200_HOST_PROBE");
    const bool probe_nocompute = probe && strstr(probe, "nocompute"), probe_nod2h = probe && strstr(probe, "nod2h");
#else
    constexpr bool probe_nocompute = false, probe_nod2h = false;
#endif
    // upload of band b is enqueued right before the match of band b, so the host never runs
    // far ahead of the device with copy submissions while kernels wait to be launched
    auto enqueue = [&]() -> int {
        for (int b = 0; b < bands; ++b) {
            const int rb = cut[b], re = cut[b + 1];
            if (stage_inputs) {
                const int slot = b % PIN_SLOTS;
                if (b >= PIN_SLOTS)
                    CU(cudaEventSynchronize(h->ev_slot[slot])); // its previous upload has left the buffer
                char* const pin = static_cast<char*>(h->pin_in[slot].ptr);
                const size_t band_bytes = row_bytes * (size_t)(re - rb);
                CopyPool::get().parallel_for(2 * n, [&](int i) {
                    const void* const* planes = i < n ? host_planes0 : host_planes1;
                    std::memcpy(pin + slot_plane * i, static_cast<const char*>(planes[i % n]) + row_bytes * rb, band_bytes);
                });
                // pinned slot [2n][band rows][row_bytes] -> device planes [2n][rows][pitch], rows rb..re
                cudaMemcpy3DParms cp {};
                cp.srcPtr = make_cudaPitchedPtr(pin, row_bytes, row_bytes, (size_t)band_rows_max);
                cp.dstPtr = make_cudaPitchedPtr(base, pitch, row_bytes, (size_t)rows);
                cp.dstPos = make_cudaPos(0, (size_t)rb, 0);
                cp.extent = make_cudaExtent(row_bytes, (size_t)(re - rb), (size_t)(2 * n));
                cp.kind = cudaMemcpyHostToDevice;
                CU(cudaMemcpy3DAsync(&cp, h->s_in));
                CU(cudaEventRecord(h->ev_slot[slot], h->s_in));
            } else {
                CU(upload_band(host_planes0, contig0, base, n, rows, row_bytes, pitch, rb, re, h->s_in));
                CU(upload_band(host_planes1, contig1, base + plane_bytes * n, n, rows, row_bytes, pitch, rb, re, h->s_in));
            }
            CU(cudaEventRecord(h->ev_in[b], h->s_in));
            CU(cudaStreamWaitEvent(h->s_compute, h->ev_in[b], 0));
            if (!probe_nocompute)
            if (int rc = do_match(h, dev0.data(), dev1.data(), n, rows, cols, pitch, depth, cfg, rb, re,
                                  h->stage_disp.ptr, (size_t)cols * disp_eb, want_corr ? h->stage_corr.ptr : nullptr,
                                  (size_t)cols * corr_eb, h->s_compute))
                return rc;
            CU(cudaEventRecord(h->ev_done[b], h->s_compute));
            CU(cudaStreamWaitEvent(h->s_out, h->ev_done[b], 0));
            const size_t off = (size_t)rb * cols, cnt = (size_t)(re - rb) * cols;
            if (probe_nod2h)
                continue;
            CU(cudaMemcpyAsync(out_disp + off * disp_eb, static_cast<char*>(h->stage_disp.ptr) + off * disp_eb,
                               cnt * disp_eb, cudaMemcpyDeviceToHost, h->s_out));
            if (want_corr)
                CU(cudaMemcpyAsync(out_corr + off * corr_eb, static_cast<char*>(h->stage_corr.ptr) + off * corr_eb,
                                   cnt * corr_eb, cudaMemcpyDeviceToHost, h->s_out));
        }
        return 0;
    };
    if (int rc = enqueue()) {
        const std::string keep = g_error;
        cudaDeviceSynchronize(); // nothing of a half-enqueued match may still touch the host buffers
        g_error = keep;
        return rc;
    }
    h->user_disp = stage_disp ? host_disparity : nullptr;
    h->user_disp_bytes = (size_t)rows * cols * disp_eb;
    h->user_corr = stage_corr ? host_corrmap : nullptr;
    h->user_corr_bytes = (size_t)rows * cols * corr_eb;
    h->host_pending = true;
    return 0;
}

int bicos_b200_match_host_end(bicos_b200_handle h) {
    if (!h)
        return fail(BICOS_B200_ERR_INVALID, "null handle");
    if (!h->host_pending)
        return 0;
    DeviceGuard g(h->device);
    h->host_pending = false;
    CU(cudaStreamSynchronize(h->s_out));
    CU(cudaStreamSynchronize(h->s_compute));
    if (int rc = check_search_timeout())
        return rc;
    // pageable result buffers: out of the pinned images, a slice per host thread
    struct Piece {
        char* dst;
        const char* src;
        size_t bytes;
    };
    std::vector<Piece> pieces;
    auto add = [&](void* user, const PinnedBuffer& pin, size_t bytes) {
        const size_t step = 1u << 20;
        for (size_t o = 0; user && o < bytes; o += step)
            pieces.push_back({ static_cast<char*>(user) + o, static_cast<const char*>(pin.ptr) + o, bytes - o < step ? bytes - o : step });
    };
    add(h->user_disp, h->pin_disp, h->user_disp_bytes);
    add(h->user_corr, h->pin_corr, h->user_corr_bytes);
    CopyPool::get().parallel_for((int)pieces.size(), [&](int i) { std::memcpy(pieces[i].dst, pieces[i].src, pieces[i].bytes); });
    h->user_disp = h->user_corr = nullptr;
    return 0;
}

int bicos_b200_match_host(bicos_b200_handle h, const void* const* host_planes0,
                          const void* const* host_planes1, int n, int rows, int cols, int depth,
                          const bicos_b200_config* cfg, void* host_disparity, void* host_corrmap) {
    if (int rc = bicos_b200_match_host_begin(h, host_planes0, host_planes1, n, rows, cols, depth, cfg, host_disparity,
                                             host_corrmap))
        return rc;
    return bicos_b200_match_host_end(h);
}

// ---- peer-memory output assembly (one process per GPU) ------------------------------------------

int bicos_b200_shared_alloc(int device, size_t bytes, void** dev_ptr, void* handle_out) {
    if (!dev_ptr || !handle_out || bytes == 0)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == BICOS_B200_IPC_HANDLE_BYTES, "IPC handle size");
    DeviceGuard g(device);
    if (!g.ok)
        return fail(BICOS_B200_ERR_CUDA, "cannot select device %d", device);
    void* p = nullptr;
    CU(cudaMalloc(&p, bytes)); // a dedicated allocation: IPC handles name whole allocations
    cudaIpcMemHandle_t hd;
    const cudaError_t err = cudaIpcGetMemHandle(&hd, p);
    if (err != cudaSuccess) {
        cudaFree(p);
        return cuda_fail(err, "cudaIpcGetMemHandle");
    }
    std::memcpy(handle_out, &hd, sizeof hd);
    *dev_ptr = p;
    return 0;
}

int bicos_b200_shared_open(int device, const void* handle, void** dev_ptr) {
    if (!handle || !dev_ptr)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    DeviceGuard g(device);
    if (!g.ok)
        return fail(BICOS_B200_ERR_CUDA, "cannot select device %d", device);
    cudaIpcMemHandle_t hd;
    std::memcpy(&hd, handle, sizeof hd);
    CU(cudaIpcOpenMemHandle(dev_ptr, hd, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}

int bicos_b200_shared_close(int device, void* dev_ptr) {
    if (!dev_ptr)
        return 0;
    DeviceGuard g(device);
    CU(cudaDeviceSynchronize());
    CU(cudaIpcCloseMemHandle(dev_ptr));
    return 0;
}

int bicos_b200_shared_free(int device, void* dev_ptr) {
    if (!dev_ptr)
        return 0;
    DeviceGuard g(device);
    CU(cudaDeviceSynchronize());
    CU(cudaFree(dev_ptr));
    return 0;
}

int bicos_b200_set_profiling(bicos_b200_handle h, int enabled) {
    if (!h)
        return fail(BICOS_B200_ERR_INVALID, "null handle");
    h->profiling = enabled != 0;
    h->prof_used = 0;
    for (int st = 0; st < N_STAGES; ++st)
        h->stage_ms[st] = 0;
    h->stage_count = 0;
    return 0;
}

int bicos_b200_stage_times(bicos_b200_handle h, double* ms_out, long long* matches_out) {
    if (!h || !ms_out)
        return fail(BICOS_B200_ERR_INVALID, "null argument");
    DeviceGuard g(h->device);
    CU(cudaDeviceSynchronize());
    if (int rc = check_search_timeout())
        return rc;
    if (int rc = prof_collect(h))
        return rc;
    for (int st = 0; st < N_STAGES; ++st)
        ms_out[st] = h->stage_ms[st];
    if (matches_out)
        *matches_out = h->stage_count;
    return 0;
}

int bicos_b200_synchronize(bicos_b200_handle h, void* stream) {
    if (!h)
        return fail(BICOS_B200_ERR_INVALID, "null handle");
    DeviceGuard g(h->device);
    CU(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    return check_search_timeout();
}

long long bicos_b200_kernel_launches(bicos_b200_handle h) {
    return h ? h->launches : 0;
}

int bicos_b200_set_search_engine(int engine) {
    if (engine < BICOS_B200_SEARCH_AUTO || engine > BICOS_B200_SEARCH_TENSOR)
        return fail(BICOS_B200_ERR_INVALID, "search engine %d (0 = auto, 1 = popc, 2 = tensor)", engine);
    set_search_engine(engine);
    return 0;
}

int bicos_b200_get_search_engine(void) {
    return search_engine();
}

const char* bicos_b200_last_search_kernel(void) {
    return last_search_kernel();
}

} // extern "C"
