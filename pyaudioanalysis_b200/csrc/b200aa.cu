// libb200aa.so -- C ABI (include/b200aa.h) over the sm_100a kernels.
// Build: see pyaudioanalysis_b200/build.py (nvcc -gencode arch=compute_100a,code=sm_100a).
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>      // header-only NVTX 3: ranges around the entry points (visible in nsys / ncu timelines)

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200aa.h"
#include "common.cuh"
#include "generic_kernel.cuh"
#include "fast_kernel.cuh"
#include "pair_kernel.cuh"
#include "solo_kernel.cuh"
#include "tables.inl"

using namespace b200aa;

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_cuda_err;
static std::atomic<int64_t> g_launches{0};

static int cuda_fail(cudaError_t e, const char *what)
{
    g_cuda_err = std::string(what) + ": " + cudaGetErrorString(e);
    return B200AA_ERR_CUDA;
}
#define CK(call)                                                     \
    do {                                                             \
        cudaError_t e_ = (call);                                     \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call);          \
    } while (0)
#define CK_LAUNCH(name)                                              \
    do {                                                             \
        g_launches.fetch_add(1, std::memory_order_relaxed);          \
        cudaError_t e_ = cudaGetLastError();                         \
        if (e_ != cudaSuccess) return cuda_fail(e_, name);           \
    } while (0)

struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

extern "C" int b200aa_abi_version(void) { return B200AA_ABI_VERSION; }
extern "C" int64_t b200aa_launch_count(void) { return g_launches.load(); }
extern "C" const char *b200aa_last_cuda_error(void) { return g_cuda_err.c_str(); }

extern "C" const char *b200aa_status_string(int s)
{
    switch (s) {
    case B200AA_OK: return "ok";
    case B200AA_ERR_INVALID: return "invalid argument";
    case B200AA_ERR_TOO_SHORT: return "need at least one array to concatenate";   // the reference's text
    case B200AA_ERR_CHROMA: return "chroma: semitone index >= num_fft (window too short for this sampling rate)";
    case B200AA_ERR_MEL_RANGE: return "mel filterbank: filter edge beyond num_fft";
    case B200AA_ERR_CUDA: return "CUDA error";
    case B200AA_ERR_UNSUPPORTED: return "window too large for the on-chip transform";
    case B200AA_ERR_NO_DEVICE: return "no sm_100 CUDA device";
    default: return "unknown status";
    }
}

extern "C" int b200aa_device_ok(void)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return B200AA_ERR_NO_DEVICE; }
    cudaDeviceProp pr;
    if (cudaGetDeviceProperties(&pr, dev) != cudaSuccess) { cudaGetLastError(); return B200AA_ERR_NO_DEVICE; }
    return pr.major == 10 ? B200AA_OK : B200AA_ERR_NO_DEVICE;
}

// ------------------------------------------------------------------------------------------------
// host tables / counts
// ------------------------------------------------------------------------------------------------
extern "C" int b200aa_host_table(int fs, int window, int which, double *h_out)
{
    if (!h_out || window < 2 || fs <= 0) return B200AA_ERR_INVALID;
    const int K = window / 2;
    std::vector<double> t;
    int rc = B200AA_OK;
    if (which == 0) rc = b200aa_host::build_mel(fs, K, t);
    else if (which == 1) rc = b200aa_host::build_chroma(fs, K, t);
    else if (which == 2) b200aa_host::build_dct(t);
    else return B200AA_ERR_INVALID;
    if (rc != B200AA_OK) return rc;
    std::memcpy(h_out, t.data(), t.size() * sizeof(double));
    return B200AA_OK;
}

extern "C" int64_t b200aa_num_frames(int64_t n, int w, int s)
{
    return (w < 1 || s < 1) ? 0 : b200aa_host::num_frames(n, w, s);
}
extern "C" int64_t b200aa_spectrogram_rows(int64_t n, int w, int s)
{
    if (w < 1 || s < 1) return 0;
    // int((N - w) / s) + 1 with Python's truncation toward zero (ShortTermFeatures.py:413)
    return (n - w) / s + 1;
}
extern "C" int64_t b200aa_chromagram_rows(int64_t n, int w, int s)
{
    if (w < 1 || s < 1) return 0;
    return (n - s - w) / s + 1;     // C division truncates toward zero like int(x / y) (:347)
}
extern "C" int64_t b200aa_mid_windows(int64_t n_frames, int stepr)
{
    return (stepr < 1 || n_frames <= 0) ? 0 : (n_frames + stepr - 1) / stepr;
}

// ------------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------------
struct Transform {           // device tables of one transform length
    int n = 0, Nc = 0, packed = 0;
    std::vector<int> radix;
    float2 *d_tw = nullptr, *d_tw_post = nullptr;
    ~Transform()
    {
        if (d_tw) cudaFree(d_tw);
        if (d_tw_post) cudaFree(d_tw_post);
    }
};

struct b200aa_plan {
    int fs = 0, window = 0, step = 0, K = 0;
    int device = 0, sm_count = 0;
    int force_generic = 0;
    int fast_kind = 0;                  // 0 = none, else index of the specialised kernel
    int tables_status = B200AA_OK;      // B200AA_ERR_CHROMA / _MEL_RANGE when the reference cannot build its tables
    BlobLayout bl{};
    int *d_blob = nullptr;
    std::vector<int> h_blob;
    std::mutex mu;
    std::map<int, std::unique_ptr<Transform>> transforms;   // by transform length
    // workspace of the host-buffer entry points: grow-only device buffers reused across calls (a cudaMalloc /
    // cudaFree pair per call costs more than the kernels for a single clip); calls serialise on host_mu
    std::mutex host_mu;
    void *ws[4] = {nullptr, nullptr, nullptr, nullptr};
    size_t ws_cap[4] = {0, 0, 0, 0};
    FastTables fast{};                  // extra device tables of the specialised kernel
    PairTables pair{};                  // inter-pass twiddles of the warp-autonomous pair kernel (windows 32 * R)
    SoloTables solo{};                  // tables of the warp-autonomous per-frame kernel (windows 882 / 400 / 600)
    int prefer = -1;                    // -1 = automatic, 0 / 1 / 2 / 3 = generic / register-tiled CTA / pair / solo kernel only (testing, A/B)
    // ring of work counters (one per in-flight launch of a persistent kernel).  A slot is handed out again only after
    // the launch that used it last has finished: that launch recorded the slot's event, the next user's stream waits on it.
    // A slot is kSlotBytes wide: the CTA / solo / generic kernels use its first word as their work counter, the pair kernel
    // the whole slot as its per-warp range descriptors (csrc/sched.cuh: 8 bytes per resident warp).
    static constexpr unsigned kSlots = 64;
    static constexpr size_t kSlotBytes = 64 * 1024;
    unsigned char *d_counters = nullptr;
    cudaEvent_t slot_event[kSlots] = {};
    bool slot_used[kSlots] = {};
    unsigned next_slot = 0;
    std::mutex slot_mu;
    static constexpr int kPipe = 3;     // streams of the chunked host pipeline, each with its own clips / records / features buffers
    cudaStream_t pipe_stream[kPipe] = {nullptr, nullptr, nullptr};
    void *pipe_ws[kPipe][3] = {};
    size_t pipe_cap[kPipe][3] = {};
    ~b200aa_plan()
    {
        if (d_blob) cudaFree(d_blob);
        for (void *w : ws) if (w) cudaFree(w);
        for (int k = 0; k < kPipe; ++k) {
            if (pipe_stream[k]) cudaStreamDestroy(pipe_stream[k]);
            for (void *w : pipe_ws[k]) if (w) cudaFree(w);
        }
        fast.release();
        pair.release();
        solo.release();
        if (d_counters) cudaFree(d_counters);
        for (cudaEvent_t e : slot_event) if (e) cudaEventDestroy(e);
    }
};

static int make_transform(int n, std::unique_ptr<Transform> &out)
{
    std::unique_ptr<Transform> t(new Transform);
    t->n = n;
    t->packed = (n % 2 == 0) ? 1 : 0;
    t->Nc = t->packed ? n / 2 : n;
    t->radix = b200aa_host::radix_list(t->Nc);
    if (t->Nc == 1) t->radix.clear();
    if ((int)t->radix.size() > kMaxRadix) return B200AA_ERR_UNSUPPORTED;
    std::vector<float2> tw(t->Nc), tp(t->Nc);
    for (int j = 0; j < t->Nc; ++j) {
        const double a = -2.0 * b200aa_host::kPi * double(j) / double(t->Nc);
        tw[j] = make_float2(float(std::cos(a)), float(std::sin(a)));
        const double b = -2.0 * b200aa_host::kPi * double(j) / double(n);
        tp[j] = make_float2(float(std::cos(b)), float(std::sin(b)));
    }
    CK(cudaMalloc(&t->d_tw, sizeof(float2) * t->Nc));
    CK(cudaMalloc(&t->d_tw_post, sizeof(float2) * t->Nc));
    CK(cudaMemcpy(t->d_tw, tw.data(), sizeof(float2) * t->Nc, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(t->d_tw_post, tp.data(), sizeof(float2) * t->Nc, cudaMemcpyHostToDevice));
    out = std::move(t);
    return B200AA_OK;
}

static int get_transform(b200aa_plan *pl, int n, Transform **out)
{
    std::lock_guard<std::mutex> g(pl->mu);
    auto it = pl->transforms.find(n);
    if (it == pl->transforms.end()) {
        std::unique_ptr<Transform> t;
        int rc = make_transform(n, t);
        if (rc != B200AA_OK) return rc;
        it = pl->transforms.emplace(n, std::move(t)).first;
    }
    *out = it->second.get();
    return B200AA_OK;
}

// pack mel CSR + DCT + chroma entries into one int32 blob
// Returns the status of the feature tables (mfcc_filter_banks runs before the frame loop, :578 / :230-231, the chroma
// scatter fails on frame 0, :290-294); the blob is built either way so that spectrogram() still works.
static int build_blob(int fs, int K, std::vector<int> &blob, BlobLayout &bl)
{
    std::vector<double> mel, chr, dct;
    int rc_mel = b200aa_host::build_mel(fs, K, mel);
    int rc_chr = b200aa_host::build_chroma(fs, K, chr);
    b200aa_host::build_dct(dct);
    std::vector<int> m_start(40, 0), m_count(40, 0), m_off(40, 0);
    std::vector<float> m_w;
    if (rc_mel == B200AA_OK)
        for (int i = 0; i < 40; ++i) {
            int lo = -1, hi = -1;
            for (int k = 0; k < K; ++k)
                if (mel[size_t(i) * K + k] != 0.0) { if (lo < 0) lo = k; hi = k; }
            m_off[i] = (int)m_w.size();
            if (lo >= 0) {
                m_start[i] = lo;
                m_count[i] = hi - lo + 1;
                for (int k = lo; k <= hi; ++k) m_w.push_back(float(mel[size_t(i) * K + k]));
            }
        }
    std::vector<int> c_off(13, 0), c_bin;
    std::vector<float> c_w;
    if (rc_chr == B200AA_OK)
        for (int c = 0; c < 12; ++c) {
            c_off[c] = (int)c_bin.size();
            for (int k = 0; k < K; ++k)
                if (chr[size_t(c) * K + k] != 0.0) { c_bin.push_back(k); c_w.push_back(float(chr[size_t(c) * K + k])); }
            c_off[c + 1] = (int)c_bin.size();
        }
    auto put_i = [&](const std::vector<int> &v) { int at = (int)blob.size(); blob.insert(blob.end(), v.begin(), v.end()); return at; };
    auto put_f = [&](const std::vector<float> &v) {
        int at = (int)blob.size();
        for (float f : v) { int w; std::memcpy(&w, &f, 4); blob.push_back(w); }
        return at;
    };
    blob.clear();
    bl.mel_start = put_i(m_start);
    bl.mel_count = put_i(m_count);
    bl.mel_off = put_i(m_off);
    bl.mel_w = put_f(m_w);
    std::vector<float> dpad(13 * 41, 0.f);
    for (int r = 0; r < 13; ++r)
        for (int n = 0; n < 40; ++n) dpad[r * 41 + n] = float(dct[size_t(r) * 40 + n]);
    bl.dct = put_f(dpad);
    bl.chr_off = put_i(c_off);
    bl.chr_bin = put_i(c_bin);
    bl.chr_w = put_f(c_w);
    {
        std::vector<int> order(40);
        for (int i = 0; i < 40; ++i) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return m_count[a] < m_count[b]; });
        // 16 groups of <= 3 filters with balanced tap totals (longest-processing-time greedy)
        std::vector<int> grp(16 * 3, -1), load(16, 0), cntg(16, 0);
        for (int i = 39; i >= 0; --i) {
            const int f = order[i];
            int best = -1;
            for (int g = 0; g < 16; ++g)
                if (cntg[g] < 3 && (best < 0 || load[g] < load[best])) best = g;
            grp[best * 3 + cntg[best]++] = f;
            load[best] += m_count[f];
        }
        bl.mel_grp = put_i(grp);
    }
    while (blob.size() % 4) blob.push_back(0);
    bl.words = (int)blob.size();
    return (rc_mel != B200AA_OK) ? rc_mel : rc_chr;
}

extern "C" int b200aa_plan_create(b200aa_plan **out, int fs, int window, int step)
{
    if (!out || fs <= 0 || window < 2 || step < 1) return B200AA_ERR_INVALID;
    int rc = b200aa_device_ok();
    if (rc != B200AA_OK) return rc;
    std::unique_ptr<b200aa_plan> pl(new b200aa_plan);
    pl->fs = fs; pl->window = window; pl->step = step; pl->K = window / 2;
    CK(cudaGetDevice(&pl->device));
    CK(cudaDeviceGetAttribute(&pl->sm_count, cudaDevAttrMultiProcessorCount, pl->device));
    // tables that only feature_extraction / chromagram need may be unbuildable (the reference raises
    // there too); spectrogram must still work, so remember the status instead of failing here.
    pl->tables_status = build_blob(fs, pl->K, pl->h_blob, pl->bl);
    CK(cudaMalloc(&pl->d_blob, sizeof(int) * pl->h_blob.size()));
    CK(cudaMemcpy(pl->d_blob, pl->h_blob.data(), sizeof(int) * pl->h_blob.size(), cudaMemcpyHostToDevice));
    Transform *t = nullptr;
    rc = get_transform(pl.get(), window, &t);
    if (rc != B200AA_OK) return rc;
    rc = fast_plan_init(fs, window, step, pl->h_blob, pl->bl, &pl->fast, &pl->fast_kind);
    if (rc != B200AA_OK) return rc;
    int sl_ = 0, sr_ = 0;
    if ((pair_r_for_window(window) || solo_shape_for_window(window, &sl_, &sr_)) && pl->tables_status == B200AA_OK) {
        std::vector<double> mel, chr, dct;
        b200aa_host::build_mel(fs, pl->K, mel);
        b200aa_host::build_chroma(fs, pl->K, chr);
        b200aa_host::build_dct(dct);
        std::vector<int> pblob;
        PairBlobLayout pbl{};
        build_pair_blob(mel, chr, dct, pl->K, pblob, pbl);
        rc = pair_plan_init(window, pblob, pbl, &pl->pair);
        if (rc != B200AA_OK) return cuda_fail(cudaGetLastError(), "pair_plan_init");
        rc = solo_plan_init(window, pblob, pbl, &pl->solo);
        if (rc != B200AA_OK) return cuda_fail(cudaGetLastError(), "solo_plan_init");
    }
    CK(cudaMalloc(&pl->d_counters, b200aa_plan::kSlots * b200aa_plan::kSlotBytes));
    *out = pl.release();
    return B200AA_OK;
}

extern "C" void b200aa_plan_destroy(b200aa_plan *plan) { delete plan; }
// work-counter slot for one launch on stream st (see b200aa_plan::slot_event); call slot_done after the launch
static int slot_acquire(b200aa_plan *pl, cudaStream_t st, unsigned *slot, unsigned int **ctr)
{
    std::lock_guard<std::mutex> g(pl->slot_mu);
    const unsigned s = pl->next_slot++ % b200aa_plan::kSlots;
    if (!pl->slot_event[s]) CK(cudaEventCreateWithFlags(&pl->slot_event[s], cudaEventDisableTiming));
    if (pl->slot_used[s]) CK(cudaStreamWaitEvent(st, pl->slot_event[s], 0));
    *slot = s;
    *ctr = reinterpret_cast<unsigned int *>(pl->d_counters + size_t(s) * b200aa_plan::kSlotBytes);
    return B200AA_OK;
}
static int slot_done(b200aa_plan *pl, cudaStream_t st, unsigned slot)
{
    std::lock_guard<std::mutex> g(pl->slot_mu);
    CK(cudaEventRecord(pl->slot_event[slot], st));
    pl->slot_used[slot] = true;
    return B200AA_OK;
}

static bool use_pair(const b200aa_plan *pl) { return pl->pair.R && !pl->force_generic && (pl->prefer < 0 || pl->prefer == 2); }
static bool use_solo(const b200aa_plan *pl) { return pl->solo.L && !pl->force_generic && (pl->prefer < 0 || pl->prefer == 3); }
static bool use_fast(const b200aa_plan *pl) { return pl->fast_kind && !pl->force_generic && (pl->prefer < 0 || pl->prefer == 1); }
extern "C" int b200aa_plan_kernel_kind(const b200aa_plan *plan)
{
    if (!plan) return 0;
    return use_pair(plan) ? 2 : (use_solo(plan) ? 3 : (use_fast(plan) ? 1 : 0));
}
extern "C" int b200aa_plan_prefer_kernel(b200aa_plan *plan, int kind)
{
    if (!plan || kind < -1 || kind > 3) return B200AA_ERR_INVALID;
    plan->prefer = kind;
    return B200AA_OK;
}
static float *g_pair_dump = nullptr;
extern "C" int b200aa_debug_set_dump(float *d_rows)
{
    g_pair_dump = d_rows;
    return B200AA_OK;
}
extern "C" int b200aa_plan_force_generic(b200aa_plan *plan, int on)
{
    if (!plan) return 0;
    int prev = plan->force_generic;
    plan->force_generic = on ? 1 : 0;
    return prev;
}

// free the grow-only workspaces of the host-buffer entry points (they are re-allocated on demand)
extern "C" int b200aa_plan_trim(b200aa_plan *plan)
{
    if (!plan) return B200AA_ERR_INVALID;
    std::lock_guard<std::mutex> g(plan->host_mu);
    for (int i = 0; i < 4; ++i) {
        if (plan->ws[i]) cudaFree(plan->ws[i]);
        plan->ws[i] = nullptr; plan->ws_cap[i] = 0;
    }
    for (int k = 0; k < b200aa_plan::kPipe; ++k)
        for (int j = 0; j < 3; ++j) {
            if (plan->pipe_ws[k][j]) cudaFree(plan->pipe_ws[k][j]);
            plan->pipe_ws[k][j] = nullptr; plan->pipe_cap[k][j] = 0;
        }
    return B200AA_OK;
}

// a plan's tables live on the device that was current when it was created
static int plan_device_check(const b200aa_plan *pl)
{
    int dev = -1;
    CK(cudaGetDevice(&dev));
    return dev == pl->device ? B200AA_OK : B200AA_ERR_INVALID;
}

// ------------------------------------------------------------------------------------------------
// kernel 0: clip statistics  (signal / 2**15 + dc_normalize, ShortTermFeatures.py:567-570, :14-19)
// accumulators live in the output records: rsv[1..2] (8-byte aligned) = sum (int64 / double), lo/hi = min/max keys
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int float_key(float f)
{
    int b = __float_as_int(f);
    return b >= 0 ? b : b ^ 0x7fffffff;
}
__device__ __forceinline__ float key_float(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

__global__ void stats_init_kernel(b200aa_clip_norm *nm, int64_t n)
{
    int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
    if (i >= n) return;
    unsigned long long *acc = reinterpret_cast<unsigned long long *>(&nm[i].rsv[1]);
    *acc = 0ull;
    reinterpret_cast<int *>(&nm[i].lo)[0] = 0x7fffffff;              // running min key
    reinterpret_cast<int *>(&nm[i].hi)[0] = int(0x80000000u);        // running max key
}

template <int DTYPE>
__global__ void __launch_bounds__(256) stats_accum_kernel(const void *sig, int64_t n_samples, int64_t clip_stride,
                                                           const int64_t *len, b200aa_clip_norm *nm, int chunks)
{
    const int64_t b = blockIdx.y;
    const int64_t L = len ? len[b] : n_samples;
    const int64_t per = (L + chunks - 1) / chunks;
    const int64_t s0 = blockIdx.x * per, s1 = min(L, s0 + per);
    long long isum = 0;
    double dsum = 0.0;
    int kmin = 0x7fffffff, kmax = int(0x80000000u);
    if (DTYPE == B200AA_DTYPE_I16) {
        const short *x = reinterpret_cast<const short *>(sig) + b * clip_stride;
        int mn = 32767, mx = -32768;
        int64_t i = s0 + threadIdx.x;
        // 16-byte vector body when the chunk start is aligned
        const bool al = ((reinterpret_cast<uintptr_t>(x + s0) & 15) == 0);
        if (al) {
            const int4 *v = reinterpret_cast<const int4 *>(x + s0);
            const int64_t nv = (s1 - s0) / 8;
            // four 16-byte loads in flight per thread (the kernel is a pure HBM stream: memory-level parallelism is all it needs)
            int64_t j = threadIdx.x;
            for (; j + 3 * int64_t(blockDim.x) < nv; j += 4 * int64_t(blockDim.x)) {
                int4 q[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) q[t] = __ldg(v + j + t * int64_t(blockDim.x));
                int acc = 0;
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const int w4[4] = {q[t].x, q[t].y, q[t].z, q[t].w};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int a0 = (short)(w4[u] & 0xffff), a1 = w4[u] >> 16;
                        acc += a0 + a1;
                        mn = min(mn, min(a0, a1));
                        mx = max(mx, max(a0, a1));
                    }
                }
                isum += acc;
            }
            for (; j < nv; j += blockDim.x) {
                int acc = 0;
                const int4 q = __ldg(v + j);
                const int w4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int a0 = (short)(w4[u] & 0xffff), a1 = w4[u] >> 16;
                    acc += a0 + a1;
                    mn = min(mn, min(a0, a1));
                    mx = max(mx, max(a0, a1));
                }
                isum += acc;
            }
            i = s0 + nv * 8 + threadIdx.x;
        }
        for (; i < s1; i += blockDim.x) {
            const int a0 = x[i];
            isum += a0;
            mn = min(mn, a0);
            mx = max(mx, a0);
        }
        kmin = mn; kmax = mx;
    } else {
        const float *x = reinterpret_cast<const float *>(sig) + b * clip_stride;
        for (int64_t i = s0 + threadIdx.x; i < s1; i += blockDim.x) {
            const float v = x[i];
            dsum += double(v);
            const int k = float_key(v);
            kmin = min(kmin, k);
            kmax = max(kmax, k);
        }
    }
    // block reduce
    __shared__ long long s_i[8];
    __shared__ double s_d[8];
    __shared__ int s_mn[8], s_mx[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        isum += __shfl_xor_sync(0xffffffffu, isum, o);
        dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
        kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, o));
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
    }
    if (lane == 0) { s_i[warp] = isum; s_d[warp] = dsum; s_mn[warp] = kmin; s_mx[warp] = kmax; }
    __syncthreads();
    if (threadIdx.x == 0 && s1 > s0) {
        for (int w = 1; w < 8; ++w) { isum += s_i[w]; dsum += s_d[w]; kmin = min(kmin, s_mn[w]); kmax = max(kmax, s_mx[w]); }
        if (DTYPE == B200AA_DTYPE_I16)
            atomicAdd(reinterpret_cast<unsigned long long *>(&nm[b].rsv[1]), (unsigned long long)isum);
        else
            atomicAdd(reinterpret_cast<double *>(&nm[b].rsv[1]), dsum);
        atomicMin(reinterpret_cast<int *>(&nm[b].lo), kmin);
        atomicMax(reinterpret_cast<int *>(&nm[b].hi), kmax);
    }
}

template <int DTYPE>
__global__ void stats_finish_kernel(b200aa_clip_norm *nm, int64_t n, int64_t n_samples, const int64_t *len)
{
    int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
    if (i >= n) return;
    const int64_t L = len ? len[i] : n_samples;
    b200aa_clip_norm r = nm[i];
    double mean, mn, mx;
    if (DTYPE == B200AA_DTYPE_I16) {
        const long long s = *reinterpret_cast<const long long *>(&nm[i].rsv[1]);
        mean = L > 0 ? double(s) / double(L) : 0.0;
        mn = double(*reinterpret_cast<const int *>(&r.lo));
        mx = double(*reinterpret_cast<const int *>(&r.hi));
    } else {
        const double s = *reinterpret_cast<const double *>(&nm[i].rsv[1]);
        mean = L > 0 ? s / double(L) : 0.0;
        mn = double(key_float(*reinterpret_cast<const int *>(&r.lo)));
        mx = double(key_float(*reinterpret_cast<const int *>(&r.hi)));
    }
    if (L <= 0) { mn = mx = 0.0; }
    // y = (x/2^15 - mean/2^15) / (max|x/2^15 - mean/2^15| + 1e-10)  ==  (x - mean) / (maxdev + 2^15 * 1e-10)
    const double maxdev = fmax(mx - mean, mean - mn);
    const double a = 1.0 / (maxdev + 32768.0 * 1e-10);
    double m, lo, hi;
    if (DTYPE == B200AA_DTYPE_I16) {
        m = nearbyint(mean);
        lo = floor(mean);
        hi = ceil(mean);
    } else {
        const float mf = float(mean);
        m = double(mf);
        if (double(mf) > mean) { hi = mf; lo = nextafterf(mf, -INFINITY); }
        else if (double(mf) < mean) { lo = mf; hi = nextafterf(mf, INFINITY); }
        else { lo = hi = mf; }
    }
    b200aa_clip_norm o;
    o.a = float(a);
    o.bp = float(a * (m - mean));
    o.m = float(m);
    o.lo = float(lo - m);
    o.hi = float(hi - m);
    o.rsv[0] = o.rsv[1] = o.rsv[2] = 0.f;
    nm[i] = o;
}

extern "C" int b200aa_clip_stats(const void *d_sig, int dtype, int64_t n_clips, int64_t n_samples,
                                 int64_t clip_stride, const int64_t *d_len, b200aa_clip_norm *d_norm, void *stream)
{
    NvtxRange nvtx_("b200aa_clip_stats");
    if (!d_sig || !d_norm || n_clips < 0 || n_samples < 0 || (dtype != 0 && dtype != 1)) return B200AA_ERR_INVALID;
    if (n_clips == 0) return B200AA_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int dev = 0, sms = 148;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int tb = 256;
    stats_init_kernel<<<(unsigned)((n_clips + tb - 1) / tb), tb, 0, st>>>(d_norm, n_clips);
    CK_LAUNCH("stats_init_kernel");
    // enough CTAs to fill the machine, each reading >= 32 KiB
    int64_t want = (int64_t(sms) * 8 + n_clips - 1) / n_clips;
    const int64_t bytes = n_samples * (dtype == 0 ? 2 : 4);
    int64_t cap = (bytes + 32767) / 32768;
    int chunks = (int)std::max<int64_t>(1, std::min<int64_t>(want, cap));
    for (int64_t b0 = 0; b0 < n_clips; b0 += 32768) {
        const int64_t nb = std::min<int64_t>(32768, n_clips - b0);
        dim3 grid(chunks, (unsigned)nb);
        const size_t es = dtype == 0 ? 2 : 4;
        const void *sig = reinterpret_cast<const char *>(d_sig) + size_t(b0) * clip_stride * es;
        const int64_t *ln = d_len ? d_len + b0 : nullptr;
        if (dtype == 0) stats_accum_kernel<0><<<grid, 256, 0, st>>>(sig, n_samples, clip_stride, ln, d_norm + b0, chunks);
        else stats_accum_kernel<1><<<grid, 256, 0, st>>>(sig, n_samples, clip_stride, ln, d_norm + b0, chunks);
        CK_LAUNCH("stats_accum_kernel");
    }
    if (dtype == 0) stats_finish_kernel<0><<<(unsigned)((n_clips + tb - 1) / tb), tb, 0, st>>>(d_norm, n_clips, n_samples, d_len);
    else stats_finish_kernel<1><<<(unsigned)((n_clips + tb - 1) / tb), tb, 0, st>>>(d_norm, n_clips, n_samples, d_len);
    CK_LAUNCH("stats_finish_kernel");
    return B200AA_OK;
}

// ------------------------------------------------------------------------------------------------
// kernel 2: mid-term pooling (MidTermFeatures.py:110-126): one warp per (clip, feature row, window)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mid_pool_kernel(const float *st, int64_t n_clips, int F, int64_t T,
                                                        int64_t t_stride, int ratio, int stepr, int64_t M, float *mid)
{
    const int lane = threadIdx.x & 31;
    const int64_t wid = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
    const int64_t total = n_clips * F * M;
    if (wid >= total) return;
    const int64_t j = wid % M, bf = wid / M;
    const int64_t b = bf / F;
    const int f = int(bf - b * F);
    const int64_t c0 = j * stepr, c1 = min(T, c0 + ratio);
    const float *row = st + (size_t(b) * F + f) * t_stride;
    const int n = int(c1 - c0);
    double s = 0.0;
    for (int64_t c = c0 + lane; c < c1; c += 32) s += double(row[c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const double mean = s / double(n);
    double v = 0.0;
    for (int64_t c = c0 + lane; c < c1; c += 32) { const double d = double(row[c]) - mean; v += d * d; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) {
        float mu = float(mean), sd = float(sqrt(v / double(n)));
        // np.nan_to_num (:126)
        if (isnan(mu)) mu = 0.f;
        if (isnan(sd)) sd = 0.f;
        if (isinf(mu)) mu = mu > 0 ? 3.4028234664e38f : -3.4028234664e38f;
        if (isinf(sd)) sd = 3.4028234664e38f;
        mid[(size_t(b) * 2 * F + f) * M + j] = mu;
        mid[(size_t(b) * 2 * F + F + f) * M + j] = sd;
    }
}

extern "C" int b200aa_mid_pool(const float *d_st, int64_t n_clips, int n_feats, int64_t n_frames, int64_t t_stride,
                               int ratio, int step_ratio, float *d_mid, void *stream)
{
    NvtxRange nvtx_("b200aa_mid_pool");
    if (!d_st || !d_mid || n_clips < 0 || n_feats < 1 || n_frames < 1 || ratio < 1 || step_ratio < 1 || t_stride < n_frames)
        return B200AA_ERR_INVALID;
    const int64_t M = b200aa_mid_windows(n_frames, step_ratio);
    const int64_t warps = n_clips * n_feats * M;
    if (warps == 0) return B200AA_OK;
    const int64_t blocks = (warps * 32 + 255) / 256;
    mid_pool_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_st, n_clips, n_feats, n_frames, t_stride,
                                                                                       ratio, step_ratio, M, d_mid);
    CK_LAUNCH("mid_pool_kernel");
    return B200AA_OK;
}

// long-term average of the mid-term matrix: one warp per (clip, row), fp64 accumulation
__global__ void __launch_bounds__(256) long_term_mean_kernel(const float *mid, int64_t rows_total, int64_t M, float *out)
{
    const int lane = threadIdx.x & 31;
    const int64_t wid = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
    if (wid >= rows_total) return;
    const float *row = mid + size_t(wid) * M;
    double s = 0.0;
    for (int64_t c = lane; c < M; c += 32) s += double(row[c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[wid] = float(s / double(M));
}

extern "C" int b200aa_long_term_mean(const float *d_mid, int64_t n_clips, int n_rows, int64_t n_windows, float *d_out, void *stream)
{
    if (!d_mid || !d_out || n_clips < 0 || n_rows < 1 || n_windows < 1) return B200AA_ERR_INVALID;
    const int64_t rows = n_clips * n_rows;
    if (rows == 0) return B200AA_OK;
    const int64_t blocks = (rows * 32 + 255) / 256;
    long_term_mean_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_mid, rows, n_windows, d_out);
    CK_LAUNCH("long_term_mean_kernel");
    return B200AA_OK;
}

// (mid[b, f, j] - mean[f]) / std[f] -> out[b, j, f]: 32 x 32 tiles through shared memory, both sides coalesced
// (audioSegmentation.py:581-584: one column of the mid-term matrix at a time)
__global__ void normalize_windows_kernel(const float *__restrict__ mid, int n_rows, int64_t n_windows, const float *__restrict__ mean,
                                         const float *__restrict__ sd, float *__restrict__ out)
{
    __shared__ float tile[32][33];
    const int64_t b = blockIdx.z;
    const int64_t j0 = int64_t(blockIdx.x) * 32;
    const int f0 = blockIdx.y * 32;
    const float *src = mid + b * n_rows * n_windows;
    float *dst = out + b * n_rows * n_windows;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int f = f0 + r;
        const int64_t j = j0 + threadIdx.x;
        if (f < n_rows && j < n_windows) tile[r][threadIdx.x] = (src[int64_t(f) * n_windows + j] - mean[f]) / sd[f];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int64_t j = j0 + r;
        const int f = f0 + threadIdx.x;
        if (f < n_rows && j < n_windows) dst[j * n_rows + f] = tile[threadIdx.x][r];
    }
}

extern "C" int b200aa_normalize_windows(const float *d_mid, int64_t n_clips, int n_rows, int64_t n_windows, const float *d_mean,
                                        const float *d_std, float *d_out, void *stream)
{
    if (!d_mid || !d_out || !d_mean || !d_std || n_clips < 0 || n_rows < 1 || n_windows < 0) return B200AA_ERR_INVALID;
    if (n_clips == 0 || n_windows == 0) return B200AA_OK;
    if ((n_rows + 31) / 32 > 65535) return B200AA_ERR_UNSUPPORTED;
    // grid.z holds at most 65 535 clips: larger batches run as slabs of that many, each offset by whole clips
    constexpr int64_t kSlab = 65535;
    const size_t clip_elems = size_t(n_rows) * size_t(n_windows);
    for (int64_t b0 = 0; b0 < n_clips; b0 += kSlab) {
        const int64_t nb = std::min<int64_t>(kSlab, n_clips - b0);
        const dim3 grid((unsigned)((n_windows + 31) / 32), (unsigned)((n_rows + 31) / 32), (unsigned)nb), block(32, 8);
        normalize_windows_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(
            d_mid + size_t(b0) * clip_elems, n_rows, n_windows, d_mean, d_std, d_out + size_t(b0) * clip_elems);
        CK_LAUNCH("normalize_windows_kernel");
    }
    return B200AA_OK;
}

// ------------------------------------------------------------------------------------------------
// kernel 1 launchers
// ------------------------------------------------------------------------------------------------
static void fill_common(StParams &p, const b200aa_plan *pl, const Transform *t, const void *d_sig, int dtype,
                        int64_t n_clips, int64_t n_samples, int64_t clip_stride, const int64_t *d_len,
                        const b200aa_clip_norm *d_norm, float *d_out)
{
    std::memset(&p, 0, sizeof(p));
    p.sig = d_sig; p.len = d_len; p.norm = d_norm; p.out = d_out;
    p.tw = t->d_tw; p.tw_post = t->d_tw_post; p.blob = pl->d_blob; p.bl = pl->bl;
    p.n_clips = n_clips; p.n_samples = n_samples; p.clip_stride = clip_stride;
    p.dtype = dtype; p.window = pl->window; p.fft_n = t->n; p.step = pl->step; p.K = pl->K;
    p.Kp = (pl->K + 3) & ~3;
    p.Nc = t->Nc; p.packed = t->packed;
    p.nrad = (int)t->radix.size();
    for (int i = 0; i < p.nrad; ++i) p.radix[i] = t->radix[i];
}

// choose frames/group and launch the generic kernel
template <int MODE>
static int launch_generic(const b200aa_plan *pl, StParams &p, int64_t rows_max, cudaStream_t st)
{
    int G = 8;
    size_t smem = 0;
    for (; G >= 1; G >>= 1) {
        smem = generic_smem_bytes(G, p.Nc, p.Kp, p.bl.words);
        if (smem <= (G == 8 ? 100u * 1024u : 226u * 1024u)) break;   // 227 KB is the per-CTA opt-in maximum
    }
    const bool big = G < 1;            // one frame does not fit shared memory: window-sized arrays go to global memory
    if (big) {
        G = 1;
        smem = generic_smem_bytes(G, p.Nc, p.Kp, p.bl.words, false);
        if (p.Nc > (1 << 20)) return B200AA_ERR_UNSUPPORTED;          // 2^21-sample windows: beyond any use of the path
    }
    p.G = G;
    // segments: long enough to amortise the 2-frame halo, short enough to balance the SMs
    int64_t seg = rows_max;
    if (MODE == kModeFeatures) {
        const int64_t slots = int64_t(pl->sm_count) * 2;
        int64_t per_clip = std::max<int64_t>(1, (slots * 12 + p.n_clips - 1) / p.n_clips);
        seg = std::max<int64_t>(G * 6 - 2, (rows_max + per_clip - 1) / per_clip);
        seg = std::min<int64_t>(seg, std::max<int64_t>(rows_max, 1));
    } else {
        seg = std::max<int64_t>(G * 4, (rows_max + 63) / 64);
    }
    p.seg_len = seg;
    p.segs_per_clip = std::max<int64_t>(1, (rows_max + seg - 1) / seg);
    p.n_items = p.segs_per_clip * p.n_clips;
    if (p.n_items == 0) return B200AA_OK;
    if (big) {
        auto kern = st_generic_kernel<MODE, true>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
        const int64_t grid = std::min<int64_t>(p.n_items, int64_t(pl->sm_count) * 2);
        p.scratch_stride = generic_big_bytes(G, p.Nc, p.Kp);
        void *scratch = nullptr;
        CK(cudaMallocAsync(&scratch, p.scratch_stride * size_t(grid), st));      // stream-ordered: safe across concurrent launches
        p.scratch = static_cast<unsigned char *>(scratch);
        kern<<<(unsigned)grid, kThreads, smem, st>>>(p);
        const cudaError_t e = cudaGetLastError();
        cudaFreeAsync(scratch, st);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        if (e != cudaSuccess) return cuda_fail(e, "st_generic_kernel (large window)");
        return B200AA_OK;
    }
    auto kern = st_generic_kernel<MODE, false>;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));   // constant: no race between launching threads
    int occ = 1;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kThreads, smem));
    occ = std::max(1, occ);
    const int64_t grid = std::min<int64_t>(p.n_items, int64_t(pl->sm_count) * occ);
    kern<<<(unsigned)grid, kThreads, smem, st>>>(p);
    CK_LAUNCH("st_generic_kernel");
    return B200AA_OK;
}

extern "C" int b200aa_st_features(const b200aa_plan *plan, const void *d_sig, int dtype, int64_t n_clips,
                                  int64_t n_samples, int64_t clip_stride, const int64_t *d_len,
                                  const b200aa_clip_norm *d_norm, int deltas, float *d_out, int64_t t_stride, void *stream)
{
    NvtxRange nvtx_("b200aa_st_features");
    if (!plan || !d_sig || !d_norm || !d_out || n_clips < 0 || (dtype != 0 && dtype != 1) || clip_stride < n_samples)
        return B200AA_ERR_INVALID;
    b200aa_plan *pl = const_cast<b200aa_plan *>(plan);
    // error order of the reference: mel bank (before the loop), no frames (:684), chroma (frame 0)
    if (pl->tables_status == B200AA_ERR_MEL_RANGE) return B200AA_ERR_MEL_RANGE;
    const int64_t T = b200aa_host::num_frames(n_samples, pl->window, pl->step);
    if (T == 0) return B200AA_ERR_TOO_SHORT;
    int rc = pl->tables_status;
    if (rc != B200AA_OK) return rc;
    if ((rc = plan_device_check(pl)) != B200AA_OK) return rc;
    if (t_stride < T) return B200AA_ERR_INVALID;
    if (n_clips == 0) return B200AA_OK;
    Transform *t = nullptr;
    rc = get_transform(pl, pl->window, &t);
    if (rc != B200AA_OK) return rc;
    StParams p;
    fill_common(p, pl, t, d_sig, dtype, n_clips, n_samples, clip_stride, d_len, d_norm, d_out);
    p.t_stride = t_stride; p.deltas = deltas ? 1 : 0; p.n_out = deltas ? 68 : 34; p.mode = kModeFeatures;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (use_pair(pl)) {
        unsigned slot = 0;
        unsigned int *ctr = nullptr;
        if ((rc = slot_acquire(pl, st, &slot, &ctr)) != B200AA_OK) return rc;
        rc = pair_launch_features(pl->pair, p, pl->sm_count, T, reinterpret_cast<unsigned long long *>(ctr), b200aa_plan::kSlotBytes, g_pair_dump, st);
        const int rc2 = slot_done(pl, st, slot);
        if (rc == B200AA_OK) { g_launches.fetch_add(1, std::memory_order_relaxed); return rc2; }
        if (rc != B200AA_ERR_UNSUPPORTED) return rc == B200AA_ERR_CUDA ? cuda_fail(cudaGetLastError(), "pair kernel") : rc;
    }
    if (use_solo(pl)) {
        unsigned slot = 0;
        unsigned int *ctr = nullptr;
        if ((rc = slot_acquire(pl, st, &slot, &ctr)) != B200AA_OK) return rc;
        rc = solo_launch_mode<kModeFeatures>(pl->solo, p, pl->sm_count, T, ctr, b200aa_plan::kSlotBytes, st);
        const int rc2 = slot_done(pl, st, slot);
        if (rc == B200AA_OK) { g_launches.fetch_add(1, std::memory_order_relaxed); return rc2; }
        if (rc != B200AA_ERR_UNSUPPORTED) return rc == B200AA_ERR_CUDA ? cuda_fail(cudaGetLastError(), "solo kernel") : rc;
    }
    if (use_fast(pl)) {
        unsigned slot = 0;
        unsigned int *ctr = nullptr;
        if ((rc = slot_acquire(pl, st, &slot, &ctr)) != B200AA_OK) return rc;
        rc = fast_launch_features(pl->fast_kind, pl->fast, p, pl->sm_count, T, ctr, st);
        const int rc2 = slot_done(pl, st, slot);
        if (rc == B200AA_OK) { g_launches.fetch_add(1, std::memory_order_relaxed); return rc2; }
        if (rc != B200AA_ERR_UNSUPPORTED) return rc == B200AA_ERR_CUDA ? cuda_fail(cudaGetLastError(), "fast kernel") : rc;
    }
    return launch_generic<kModeFeatures>(pl, p, T, st);
}

extern "C" int b200aa_spectrogram(const b200aa_plan *plan, const void *d_sig, int dtype, int64_t n_clips,
                                  int64_t n_samples, int64_t clip_stride, const b200aa_clip_norm *d_norm,
                                  float *d_out, void *stream)
{
    NvtxRange nvtx_("b200aa_spectrogram");
    if (!plan || !d_sig || !d_norm || !d_out || n_clips < 0 || (dtype != 0 && dtype != 1) || clip_stride < n_samples)
        return B200AA_ERR_INVALID;
    b200aa_plan *pl = const_cast<b200aa_plan *>(plan);
    const int w = pl->window, s = pl->step;
    const int64_t R = b200aa_spectrogram_rows(n_samples, w, s);
    if (R <= 0) return B200AA_ERR_TOO_SHORT;      // np.zeros with a non-positive row count / empty result
    if (n_clips == 0) return B200AA_OK;
    int rc = plan_device_check(pl);
    if (rc != B200AA_OK) return rc;
    Transform *t = nullptr;
    rc = get_transform(pl, w, &t);
    if (rc != B200AA_OK) return rc;
    StParams p;
    fill_common(p, pl, t, d_sig, dtype, n_clips, n_samples, clip_stride, nullptr, d_norm, d_out);
    p.mode = kModeSpectrogram;
    p.origin = w; p.row0 = 0; p.rows_total = R; p.rows_launch = R;
    p.rows_valid = std::min<int64_t>(R, b200aa_host::range_len(w, n_samples - w + 1, s));   // :415
    if (use_solo(pl)) {
        cudaStream_t st_ = static_cast<cudaStream_t>(stream);
        unsigned slot = 0;
        unsigned int *ctr = nullptr;
        if ((rc = slot_acquire(pl, st_, &slot, &ctr)) != B200AA_OK) return rc;
        rc = solo_launch_mode<kModeSpectrogram>(pl->solo, p, pl->sm_count, p.rows_launch, ctr, b200aa_plan::kSlotBytes, st_);
        const int rc2 = slot_done(pl, st_, slot);
        if (rc == B200AA_OK) { g_launches.fetch_add(1, std::memory_order_relaxed); return rc2; }
        if (rc != B200AA_ERR_UNSUPPORTED) return rc == B200AA_ERR_CUDA ? cuda_fail(cudaGetLastError(), "solo kernel") : rc;
    }
    if (pl->fast_kind && !pl->force_generic && pl->prefer != 0 && pl->prefer != 3) {
        cudaStream_t st_ = static_cast<cudaStream_t>(stream);
        unsigned slot = 0;
        unsigned int *ctr = nullptr;
        if ((rc = slot_acquire(pl, st_, &slot, &ctr)) != B200AA_OK) return rc;
        rc = fast_launch_rows(pl->fast_kind, kModeSpectrogram, pl->fast, p, pl->sm_count, ctr, st_);
        const int rc2 = slot_done(pl, st_, slot);
        if (rc == B200AA_OK) { g_launches.fetch_add(1, std::memory_order_relaxed); return rc2; }
        if (rc != B200AA_ERR_UNSUPPORTED) return rc == B200AA_ERR_CUDA ? cuda_fail(cudaGetLastError(), "fast kernel") : rc;
    }
    return launch_generic<kModeSpectrogram>(pl, p, R, static_cast<cudaStream_t>(stream));
}

extern "C" int b200aa_chromagram(const b200aa_plan *plan, const void *d_sig, int dtype, int64_t n_clips,
                                 int64_t n_samples, int64_t clip_stride, const b200aa_clip_norm *d_norm,
                                 float *d_out, void *stream)
{
    NvtxRange nvtx_("b200aa_chromagram");
    if (!plan || !d_sig || !d_norm || !d_out || n_clips < 0 || (dtype != 0 && dtype != 1) || clip_stride < n_samples)
        return B200AA_ERR_INVALID;
    b200aa_plan *pl = const_cast<b200aa_plan *>(plan);
    const int w = pl->window, s = pl->step;
    const int64_t R = b200aa_chromagram_rows(n_samples, w, s);
    if (R <= 0 || n_samples - s - w < 0) return B200AA_ERR_TOO_SHORT;
    int rc = pl->tables_status;
    if (rc == B200AA_ERR_CHROMA) return rc;
    if (n_clips == 0) return B200AA_OK;
    if ((rc = plan_device_check(pl)) != B200AA_OK) return rc;
    const int64_t n_it = std::min<int64_t>(R, b200aa_host::range_len(w, n_samples - s, s));        // :349
    // frames that fit entirely: start p = w + i*s with p + w <= N
    int64_t n_full = 0;
    if (n_samples - 2 * int64_t(w) >= 0) n_full = std::min<int64_t>(n_it, (n_samples - 2 * int64_t(w)) / s + 1);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Transform *t = nullptr;
    rc = get_transform(pl, w, &t);
    if (rc != B200AA_OK) return rc;
    StParams p;
    fill_common(p, pl, t, d_sig, dtype, n_clips, n_samples, clip_stride, nullptr, d_norm, d_out);
    p.mode = kModeChromagram;
    p.origin = w; p.row0 = 0; p.rows_total = R; p.rows_launch = R; p.rows_valid = n_full;
    rc = B200AA_ERR_UNSUPPORTED;
    if (use_solo(pl)) {
        unsigned slot = 0;
        unsigned int *ctr = nullptr;
        if ((rc = slot_acquire(pl, st, &slot, &ctr)) != B200AA_OK) return rc;
        rc = solo_launch_mode<kModeChromagram>(pl->solo, p, pl->sm_count, p.rows_launch, ctr, b200aa_plan::kSlotBytes, st);
        if (slot_done(pl, st, slot) != B200AA_OK) return B200AA_ERR_CUDA;
        if (rc == B200AA_OK) g_launches.fetch_add(1, std::memory_order_relaxed);
        else if (rc != B200AA_ERR_UNSUPPORTED) return rc == B200AA_ERR_CUDA ? cuda_fail(cudaGetLastError(), "solo kernel") : rc;
    }
    if (rc == B200AA_ERR_UNSUPPORTED && pl->fast_kind && !pl->force_generic && pl->prefer != 0 && pl->prefer != 3) {
        unsigned slot = 0;
        unsigned int *ctr = nullptr;
        if ((rc = slot_acquire(pl, st, &slot, &ctr)) != B200AA_OK) return rc;
        rc = fast_launch_rows(pl->fast_kind, kModeChromagram, pl->fast, p, pl->sm_count, ctr, st);
        if (slot_done(pl, st, slot) != B200AA_OK) return B200AA_ERR_CUDA;
        if (rc == B200AA_OK) g_launches.fetch_add(1, std::memory_order_relaxed);
        else if (rc != B200AA_ERR_UNSUPPORTED) return rc == B200AA_ERR_CUDA ? cuda_fail(cudaGetLastError(), "fast kernel") : rc;
    }
    if (rc == B200AA_ERR_UNSUPPORTED) rc = launch_generic<kModeChromagram>(pl, p, R, st);
    if (rc != B200AA_OK) return rc;
    // frames clipped at the end of the clip: the reference transforms the n < w samples that are
    // left (ShortTermFeatures.py:352-355); fewer than num_fft samples make its scatter raise.
    for (int64_t i = n_full; i < n_it; ++i) {
        const int64_t start = w + i * s;
        const int64_t n = n_samples - start;
        if (n < pl->K) return B200AA_ERR_INVALID;
        Transform *tc = nullptr;
        rc = get_transform(pl, (int)n, &tc);
        if (rc != B200AA_OK) return rc;
        StParams q;
        fill_common(q, pl, tc, d_sig, dtype, n_clips, n_samples, clip_stride, nullptr, d_norm, d_out);
        q.mode = kModeChromagram;
        q.origin = start; q.row0 = i; q.rows_total = R; q.rows_launch = 1; q.rows_valid = 1;
        rc = launch_generic<kModeChromagram>(pl, q, 1, st);
        if (rc != B200AA_OK) return rc;
    }
    return B200AA_OK;
}

// ------------------------------------------------------------------------------------------------
// host-buffer entry points
// ------------------------------------------------------------------------------------------------
// slot `slot` of the plan's workspace, grown to at least n bytes (caller holds host_mu); nullptr = cudaMalloc failed
static void *workspace(b200aa_plan *pl, int slot, size_t n)
{
    if (pl->ws_cap[slot] < n) {
        if (pl->ws[slot]) cudaFree(pl->ws[slot]);
        pl->ws[slot] = nullptr;
        pl->ws_cap[slot] = 0;
        const size_t want = n + n / 4 + 4096;
        if (cudaMalloc(&pl->ws[slot], want) != cudaSuccess) return nullptr;
        pl->ws_cap[slot] = want;
    }
    return pl->ws[slot];
}

// One host-buffer call: takes the plan's workspace lock, uploads the clips (slot 0) and produces their normalisation
// records (slot 1); the entry points add their own kernels and downloads on the same (legacy default) stream.
struct HostCall {
    b200aa_plan *pl;
    std::unique_lock<std::mutex> hold;
    cudaStream_t st = nullptr;
    void *sig = nullptr;
    b200aa_clip_norm *norm = nullptr;
    explicit HostCall(const b200aa_plan *plan) : pl(const_cast<b200aa_plan *>(plan)), hold(pl->host_mu) {}
    int upload(const void *h_sig, int dtype, int64_t n_clips, int64_t n_samples)
    {
        int rc = plan_device_check(pl);
        if (rc != B200AA_OK) return rc;
        const size_t in_b = size_t(n_clips) * n_samples * (dtype == B200AA_DTYPE_I16 ? 2 : 4);
        sig = workspace(pl, 0, in_b);
        norm = static_cast<b200aa_clip_norm *>(workspace(pl, 1, sizeof(b200aa_clip_norm) * n_clips));
        if (!sig || !norm) return cuda_fail(cudaGetLastError(), "cudaMalloc");
        CK(cudaMemcpyAsync(sig, h_sig, in_b, cudaMemcpyHostToDevice, st));
        return b200aa_clip_stats(sig, dtype, n_clips, n_samples, n_samples, nullptr, norm, st);
    }
    float *result(int slot, size_t bytes) { return static_cast<float *>(workspace(pl, slot, bytes)); }
    int download(void *h_dst, const void *d_src, size_t bytes)
    {
        CK(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, st));
        return B200AA_OK;
    }
    int finish()
    {
        CK(cudaStreamSynchronize(st));
        return B200AA_OK;
    }
};

// Chunked, multi-stream form of b200aa_st_features_host for batches of many clips: every chunk's upload, kernels and
// download are queued on one of three streams, so the PCIe transfers of neighbouring chunks overlap the kernels (pinned
// host memory -- b200aa_host_alloc -- makes the copies truly asynchronous; pageable memory still works, the copies
// then serialise in the driver).
static int st_features_host_pipelined(b200aa_plan *pl, const void *h_sig, int dtype, int64_t n_clips, int64_t n_samples,
                                      int deltas, float *h_out, int64_t T, int64_t chunk)
{
    std::lock_guard<std::mutex> hold(pl->host_mu);
    int rc = plan_device_check(pl);
    if (rc != B200AA_OK) return rc;
    const size_t es = dtype == B200AA_DTYPE_I16 ? 2 : 4;
    const size_t F = deltas ? 68 : 34;
    const size_t need[3] = {size_t(chunk) * n_samples * es, sizeof(b200aa_clip_norm) * size_t(chunk), size_t(chunk) * F * T * 4};
    for (int k = 0; k < b200aa_plan::kPipe; ++k) {
        if (!pl->pipe_stream[k]) CK(cudaStreamCreateWithFlags(&pl->pipe_stream[k], cudaStreamNonBlocking));
        for (int j = 0; j < 3; ++j)
            if (pl->pipe_cap[k][j] < need[j]) {
                if (pl->pipe_ws[k][j]) cudaFree(pl->pipe_ws[k][j]);
                pl->pipe_ws[k][j] = nullptr;
                pl->pipe_cap[k][j] = 0;
                CK(cudaMalloc(&pl->pipe_ws[k][j], need[j]));
                pl->pipe_cap[k][j] = need[j];
            }
    }
    int64_t c = 0;
    for (int64_t a = 0; a < n_clips && rc == B200AA_OK; a += chunk, ++c) {
        const int k = int(c % b200aa_plan::kPipe);
        const int64_t n = std::min<int64_t>(chunk, n_clips - a);
        cudaStream_t st = pl->pipe_stream[k];      // stream order also protects the buffers: chunk c + kPipe waits for chunk c
        void *sig = pl->pipe_ws[k][0];
        b200aa_clip_norm *norm = static_cast<b200aa_clip_norm *>(pl->pipe_ws[k][1]);
        float *out = static_cast<float *>(pl->pipe_ws[k][2]);
        cudaError_t e = cudaMemcpyAsync(sig, static_cast<const char *>(h_sig) + size_t(a) * n_samples * es, size_t(n) * n_samples * es,
                                        cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMemcpyAsync (clips)"); break; }
        rc = b200aa_clip_stats(sig, dtype, n, n_samples, n_samples, nullptr, norm, st);
        if (rc != B200AA_OK) break;
        rc = b200aa_st_features(pl, sig, dtype, n, n_samples, n_samples, nullptr, norm, deltas, out, T, st);
        if (rc != B200AA_OK) break;
        e = cudaMemcpyAsync(h_out + size_t(a) * F * T, out, size_t(n) * F * T * 4, cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemcpyAsync (features)");
    }
    for (int k = 0; k < b200aa_plan::kPipe; ++k) {         // drain every stream, also after an error
        const cudaError_t e = cudaStreamSynchronize(pl->pipe_stream[k]);
        if (e != cudaSuccess && rc == B200AA_OK) rc = cuda_fail(e, "cudaStreamSynchronize");
    }
    return rc;
}

extern "C" int b200aa_st_features_host(const b200aa_plan *plan, const void *h_sig, int dtype, int64_t n_clips,
                                       int64_t n_samples, int deltas, float *h_out)
{
    NvtxRange nvtx_("b200aa_st_features_host");
    if (!plan || !h_sig || !h_out || n_clips < 1 || (dtype != 0 && dtype != 1)) return B200AA_ERR_INVALID;
    if (plan->tables_status == B200AA_ERR_MEL_RANGE) return B200AA_ERR_MEL_RANGE;
    const int64_t T = b200aa_host::num_frames(n_samples, plan->window, plan->step);
    if (T == 0) return B200AA_ERR_TOO_SHORT;
    if (plan->tables_status != B200AA_OK) return plan->tables_status;
    {   // chunks of ~32 MB of samples; batches of fewer than two chunks take the single-stream path below
        const int64_t chunk = std::max<int64_t>(1, (int64_t(32) << 20) / (n_samples * (dtype == B200AA_DTYPE_I16 ? 2 : 4)));
        if (n_clips >= 2 * chunk)
            return st_features_host_pipelined(const_cast<b200aa_plan *>(plan), h_sig, dtype, n_clips, n_samples, deltas, h_out, T, chunk);
    }
    const size_t out_b = size_t(n_clips) * (deltas ? 68 : 34) * T * 4;
    HostCall hc(plan);
    int rc = hc.upload(h_sig, dtype, n_clips, n_samples);
    if (rc) return rc;
    float *out = hc.result(2, out_b);
    if (!out) return cuda_fail(cudaGetLastError(), "cudaMalloc");
    rc = b200aa_st_features(plan, hc.sig, dtype, n_clips, n_samples, n_samples, nullptr, hc.norm, deltas, out, T, hc.st);
    if (rc) return rc;
    if ((rc = hc.download(h_out, out, out_b))) return rc;
    return hc.finish();
}

extern "C" int b200aa_spectrogram_host(const b200aa_plan *plan, const void *h_sig, int dtype, int64_t n_samples, float *h_out)
{
    if (!plan || !h_sig || !h_out || (dtype != 0 && dtype != 1)) return B200AA_ERR_INVALID;
    const int64_t R = b200aa_spectrogram_rows(n_samples, plan->window, plan->step);
    if (R <= 0) return B200AA_ERR_TOO_SHORT;
    const size_t out_b = size_t(R) * plan->K * 4;
    HostCall hc(plan);
    int rc = hc.upload(h_sig, dtype, 1, n_samples);
    if (rc) return rc;
    float *out = hc.result(2, out_b);
    if (!out) return cuda_fail(cudaGetLastError(), "cudaMalloc");
    rc = b200aa_spectrogram(plan, hc.sig, dtype, 1, n_samples, n_samples, hc.norm, out, hc.st);
    if (rc) return rc;
    if ((rc = hc.download(h_out, out, out_b))) return rc;
    return hc.finish();
}

extern "C" int b200aa_chromagram_host(const b200aa_plan *plan, const void *h_sig, int dtype, int64_t n_samples, float *h_out)
{
    if (!plan || !h_sig || !h_out || (dtype != 0 && dtype != 1)) return B200AA_ERR_INVALID;
    const int64_t R = b200aa_chromagram_rows(n_samples, plan->window, plan->step);
    if (R <= 0 || n_samples - plan->step - plan->window < 0) return B200AA_ERR_TOO_SHORT;
    if (plan->tables_status == B200AA_ERR_CHROMA) return B200AA_ERR_CHROMA;
    const size_t out_b = size_t(R) * 12 * 4;
    HostCall hc(plan);
    int rc = hc.upload(h_sig, dtype, 1, n_samples);
    if (rc) return rc;
    float *out = hc.result(2, out_b);
    if (!out) return cuda_fail(cudaGetLastError(), "cudaMalloc");
    rc = b200aa_chromagram(plan, hc.sig, dtype, 1, n_samples, n_samples, hc.norm, out, hc.st);
    if (rc) return rc;
    if ((rc = hc.download(h_out, out, out_b))) return rc;
    return hc.finish();
}

extern "C" int b200aa_mid_features_host(const b200aa_plan *plan, const void *h_sig, int dtype, int64_t n_samples,
                                        int ratio, int step_ratio, float *h_mid, float *h_st)
{
    NvtxRange nvtx_("b200aa_mid_features_host");
    if (!plan || !h_sig || !h_mid || ratio < 1 || step_ratio < 1 || (dtype != 0 && dtype != 1)) return B200AA_ERR_INVALID;
    if (plan->tables_status == B200AA_ERR_MEL_RANGE) return B200AA_ERR_MEL_RANGE;
    const int64_t T = b200aa_host::num_frames(n_samples, plan->window, plan->step);
    if (T == 0) return B200AA_ERR_TOO_SHORT;
    if (plan->tables_status != B200AA_OK) return plan->tables_status;
    const int64_t M = b200aa_mid_windows(T, step_ratio);
    const size_t st_b = size_t(68) * T * 4, mid_b = size_t(136) * M * 4;
    HostCall hc(plan);
    int rc = hc.upload(h_sig, dtype, 1, n_samples);
    if (rc) return rc;
    float *stf = hc.result(2, st_b), *mid = hc.result(3, mid_b);
    if (!stf || !mid) return cuda_fail(cudaGetLastError(), "cudaMalloc");
    rc = b200aa_st_features(plan, hc.sig, dtype, 1, n_samples, n_samples, nullptr, hc.norm, 1, stf, T, hc.st);
    if (rc) return rc;
    rc = b200aa_mid_pool(stf, 1, 68, T, T, ratio, step_ratio, mid, hc.st);
    if (rc) return rc;
    if ((rc = hc.download(h_mid, mid, mid_b))) return rc;
    if (h_st && (rc = hc.download(h_st, stf, st_b))) return rc;
    return hc.finish();
}

// ------------------------------------------------------------------------------------------------
// pinned host buffers (full-speed, truly asynchronous H2D / D2H copies for the host entry points)
// ------------------------------------------------------------------------------------------------
extern "C" int b200aa_host_alloc(void **h_out, size_t bytes)
{
    if (!h_out) return B200AA_ERR_INVALID;
    *h_out = nullptr;
    if (bytes == 0) return B200AA_OK;
    // pages are placed by the calling thread's NUMA policy: bind the thread to the GPU's node first
    CK(cudaHostAlloc(h_out, bytes, cudaHostAllocPortable));
    return B200AA_OK;
}
extern "C" int b200aa_host_free(void *h_ptr)
{
    if (h_ptr) CK(cudaFreeHost(h_ptr));
    return B200AA_OK;
}

// ------------------------------------------------------------------------------------------------
// peer-mapped gather target (SURVEY 8e): rank 0 owns one [n_clips_total, F, T] buffer, every other rank of the
// box maps it (CUDA IPC over NVLink) and its feature kernel stores straight into its slice -- the gather is
// fused into the tile store, no collective kernel, no SMs on the root.
// ------------------------------------------------------------------------------------------------
static_assert(sizeof(cudaIpcMemHandle_t) == B200AA_IPC_HANDLE_BYTES, "handle size");
extern "C" int b200aa_peer_buffer_create(size_t bytes, void **d_out, unsigned char *handle_out)
{
    if (!d_out || !handle_out || bytes == 0) return B200AA_ERR_INVALID;
    CK(cudaMalloc(d_out, bytes));
    cudaIpcMemHandle_t h;
    const cudaError_t e = cudaIpcGetMemHandle(&h, *d_out);
    if (e != cudaSuccess) { cudaFree(*d_out); *d_out = nullptr; return cuda_fail(e, "cudaIpcGetMemHandle"); }
    std::memcpy(handle_out, &h, sizeof(h));
    return B200AA_OK;
}
extern "C" int b200aa_peer_buffer_open(const unsigned char *handle, void **d_out)
{
    if (!handle || !d_out) return B200AA_ERR_INVALID;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    CK(cudaIpcOpenMemHandle(d_out, h, cudaIpcMemLazyEnablePeerAccess));
    return B200AA_OK;
}
extern "C" int b200aa_peer_copy(void *d_dst, const void *d_src, size_t bytes, void *stream)
{
    if (!d_dst || !d_src) return B200AA_ERR_INVALID;
    if (bytes == 0) return B200AA_OK;
    // unified addressing: the copy engines move the block over NVLink, no SM on either side is involved
    CK(cudaMemcpyAsync(d_dst, d_src, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
    return B200AA_OK;
}
extern "C" int b200aa_peer_buffer_close(void *d_ptr, int owner)
{
    if (!d_ptr) return B200AA_OK;
    if (owner) CK(cudaFree(d_ptr));
    else CK(cudaIpcCloseMemHandle(d_ptr));
    return B200AA_OK;
}
