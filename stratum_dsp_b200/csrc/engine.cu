// Host engine + C ABI (include/stratum_b200.h) of the B200 analysis path.
//
// Execution model: a batch is cut into WAVES of tracks whose work areas fit the device arena
// (spectrograms are the bulk: 64 MB for the 2048/512 STFT — 254 MB at frame_size 8192 — and 254 MB for the 8192/512 key STFT
// of a 3-minute track).  Every stage of the reference's analyze_audio (lib.rs:86-1635) is one or a few
// kernels launched over the whole wave; per-track state lives in a TrackDev record on the device.
// The only host round trip inside a wave is the escalation decision (lib.rs:412-459): the records
// are read back, the tracks that need the multi-resolution pass are given arena slots for their
// hop-256 / hop-1024 spectrograms and processed as a compacted sub-batch.
// There is no CPU fallback: without a usable CUDA device every compute entry point fails.
#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <future>
#include <memory>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "key_rows.cuh"

namespace sb {

static inline uint64_t align_up(uint64_t x, uint64_t a) { return (x + a - 1) / a * a; }

// ---- errors ---------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
static void set_error(const std::string& s) { g_last_error = s; }

#define CUDA_OK(expr)                                                                                 \
    do {                                                                                              \
        cudaError_t e_ = (expr);                                                                      \
        if (e_ != cudaSuccess) {                                                                      \
            set_error(std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " #expr);           \
            return STRATUM_PROCESSING_ERROR;                                                          \
        }                                                                                             \
    } while (0)

// ---- launch accounting / stage timing ----------------------------------------------------------------
static std::atomic<uint64_t> g_launches{0};
static std::atomic<int> g_timing{0};
static std::mutex g_stage_mu;
static std::map<std::string, double> g_stage_ms;
static std::vector<std::string> g_stage_order;

void count_launch(const char*) { g_launches.fetch_add(1, std::memory_order_relaxed); }

// Device time of a group of launches, accumulated per stage name.  Events are only recorded here;
// they are resolved after the wave's final stream synchronisation, so timing adds no host sync.
struct PendingStage {
    const char* name;
    cudaEvent_t a, b;
};
static thread_local std::vector<PendingStage> g_pending;

struct StageTimer {
    cudaStream_t s;
    const char* name;
    cudaEvent_t a = nullptr, b = nullptr;
    StageTimer(cudaStream_t s_, const char* n) : s(s_), name(n) {
        if (g_timing.load()) {
            cudaEventCreate(&a);
            cudaEventCreate(&b);
            cudaEventRecord(a, s);
        }
    }
    ~StageTimer() {
        if (!a) return;
        cudaEventRecord(b, s);
        g_pending.push_back(PendingStage{name, a, b});
    }
};

static void resolve_stage_times(std::vector<PendingStage>& pending) {  // call once the wave that recorded them has completed
    if (pending.empty()) return;
    std::lock_guard<std::mutex> lk(g_stage_mu);
    for (PendingStage& p : pending) {
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            if (!g_stage_ms.count(p.name)) g_stage_order.push_back(p.name);
            g_stage_ms[p.name] += ms;
        }
        cudaEventDestroy(p.a);
        cudaEventDestroy(p.b);
    }
    pending.clear();
}

// Host-side time during which the device has nothing queued (planning, the escalation round trip, result gathering):
// reported next to the device stages as "host_*" when stage timing is on.
struct HostSpan {
    const char* name;
    std::chrono::steady_clock::time_point t0;
    bool on;
    explicit HostSpan(const char* n) : name(n), t0(std::chrono::steady_clock::now()), on(g_timing.load() != 0) {}
    void stop() {
        if (!on) return;
        on = false;
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        std::lock_guard<std::mutex> lk(g_stage_mu);
        if (!g_stage_ms.count(name)) g_stage_order.push_back(name);
        g_stage_ms[name] += ms;
    }
    ~HostSpan() { stop(); }
};

static std::atomic<uint64_t> g_last_call_us{0};
static std::atomic<uint32_t> g_last_call_waves{0};
static std::atomic<uint64_t> g_h2d_bytes{0}, g_d2h_bytes{0};  // host<->device traffic of this process (results, staging)  // device time of the most recent batch call (all waves), microseconds

// ---- debug capture (single-track calls) -----------------------------------------------------------------
static std::atomic<int> g_debug{0};
static std::mutex g_debug_mu;
static std::map<std::string, std::vector<float>> g_debug_arrays;

// Grow-only pinned host buffer (asynchronous copy source / target).
struct PinnedBuf {
    void* p = nullptr;
    size_t cap = 0;
    void* need(size_t bytes) {
        if (bytes > cap) {
            if (p) cudaFreeHost(p);
            p = nullptr;
            cap = 0;
            const size_t n = bytes + bytes / 2 + 4096;
            if (cudaHostAlloc(&p, n, cudaHostAllocDefault) != cudaSuccess) {
                p = nullptr;
                return nullptr;
            }
            cap = n;
        }
        return p;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

// Grow-only device buffer.
template <class T>
static bool grow_device(T*& p, size_t& cap, size_t need) {
    if (need <= cap) return true;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    if (cudaMalloc((void**)&p, need) != cudaSuccess) return false;
    cap = need;
    return true;
}

// One long-lived helper thread per device (the sample uploads of host batches): tasks run in order.
class Worker {
public:
    Worker() : th_([this] { run(); }) {}
    ~Worker() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            quit_ = true;
        }
        cv_.notify_all();
        if (th_.joinable()) th_.join();
    }
    std::future<bool> post(std::function<bool()> f) {
        std::packaged_task<bool()> task(std::move(f));
        std::future<bool> fut = task.get_future();
        {
            std::lock_guard<std::mutex> lk(mu_);
            q_.push_back(std::move(task));
        }
        cv_.notify_one();
        return fut;
    }

private:
    void run() {
        for (;;) {
            std::packaged_task<bool()> task;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [this] { return quit_ || !q_.empty(); });
                if (q_.empty()) return;
                task = std::move(q_.front());
                q_.pop_front();
            }
            task();
        }
    }
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<std::packaged_task<bool()>> q_;
    bool quit_ = false;
    std::thread th_;
};

// A wave whose launches are queued and whose results have not been gathered yet.  Two slots per device context: while wave k
// runs, the host gathers wave k-1 and plans wave k+1 (DESIGN §3).  The read-back targets are pinned, so the final copies are
// asynchronous and the stream keeps running into the next wave.
struct WaveJob {
    bool active = false;
    int nt = 0;
    std::vector<uint32_t> idx;
    std::vector<std::string> track_err;  // message of a failure found while planning a track (unsupported sample rate ...)
    PinnedBuf h_tracks, h_oa, h_ia, h_small;
    uint64_t oa_n = 0, ia_n = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;  // device time of the wave
    StratumResult* out = nullptr;
    std::vector<PendingStage> stages;
    bool debug_single = false;
    DevCfg dcfg{};
};

// ---- per-device context ------------------------------------------------------------------------------
struct DeviceCtx {
    int device = -1;
    bool ready = false;
    cudaStream_t stream = nullptr;
    cudaStream_t key_stream = nullptr;  // the key path of a wave runs beside the tempo path
    Tables tab{};
    std::vector<void*> owned;                 // table allocations
    std::map<uint32_t, float2*> tw_tables;    // size -> TW table (Stockham twiddles, oracle/so_fft.cpp)
    std::map<uint32_t, const float*> hann_tables;  // frame size -> Hann window of the generic STFT
    std::map<std::array<float, 3>, const float*> bpm_tabs;  // (min_bpm, max_bpm, bpm_resolution) -> hypothesis table of a fine BPM grid
    std::vector<SrTables> sr_host;
    std::vector<StratumConfig> sr_cfg;        // configuration each sr_host entry was built for (the tables depend on it)
    SrTables* d_srtab = nullptr;
    static constexpr int MAX_SR = 32;
    float* fa = nullptr;
    size_t fa_cap = 0;  // floats
    float* oa = nullptr;
    size_t oa_cap = 0;
    int32_t* ia = nullptr;
    size_t ia_cap = 0;
    TrackDev* d_tracks = nullptr;
    int32_t* d_sr_index = nullptr;
    int32_t* d_list = nullptr;
    float* d_gain = nullptr;
    size_t tr_cap = 0;
    float* d_stage = nullptr;  // two staging buffers for host-sample batches (double-buffered upload)
    cudaStream_t copy_stream = nullptr;
    size_t stage_cap = 0;  // bytes
    float* d_conv = nullptr;  // mono f32 buffer the PCM16 chunks are converted into
    size_t conv_cap = 0;   // bytes
    char* d_meta = nullptr;   // per-chunk offset / channel tables of the PCM16 path (two sets)
    size_t meta_cap = 0;
    PinnedBuf h_meta[2];      // their pinned host images
    char* d_loud = nullptr;   // loudness work area of one chunk (track records, results, cascade states, energies, per-segment powers)
    size_t loud_cap = 0;
    PinnedBuf loud_rec[2], loud_out[2];  // pinned track records / results of two chunks (chunk k+1 is queued before chunk k is read)
    PinnedBuf loud_blk[2];    // momentary and short-term powers of the same two chunks (calls with albums only)
    PinnedBuf loud_ser[2];    // the requested loudness series of the same two chunks (series calls only)
    char* d_album = nullptr;  // album phase: album records, pooled powers, selection scratch, results
    size_t album_cap = 0;
    cudaEvent_t loud_ev[2] = {nullptr, nullptr};
    cudaStream_t loud_stream = nullptr;  // loudness passes of stratum_b200_analyze_loudness_pcm, queued beside the analysis waves
    int32_t* d_count = nullptr;  // escalated tracks of the wave being queued (escalation_compact_kernel)
    PinnedBuf h_count;
    cudaEvent_t ev_legacy = nullptr;  // legacy estimator finished on the key stream
    WaveJob jobs[2];          // two wave slots (one queued ahead of the gather)
    std::unique_ptr<Worker> uploader;
    std::recursive_mutex mu;  // one call at a time per device; held for a whole batch call (upload, conversion, analysis)
};

static std::mutex g_ctx_mu;
static std::map<int, DeviceCtx*> g_ctx;

template <class T>
static T* dev_upload(DeviceCtx& c, const std::vector<T>& v) {
    T* p = nullptr;
    if (cudaMalloc(&p, v.size() * sizeof(T)) != cudaSuccess) return nullptr;
    cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    c.owned.push_back(p);
    return p;
}

static std::vector<float2> make_tw(uint32_t M) {  // TW[t] = (cos, -sin)(2 pi t / M) in double, rounded once
    std::vector<float2> tw(M);
    for (uint32_t t = 0; t < M; ++t) {
        const double a = 2.0 * M_PI * (double)t / (double)M;
        tw[t] = make_float2((float)cos(a), (float)(-sin(a)));
    }
    return tw;
}

// Per-pass compact tables for the STFT kernels: for every radix-4 pass with sub-size S = 4, 16, ..., M/4 the
// values TW_M[(k*r) * M/(4S)] (r = 1..3, k < S) stored at [S - 4 + (r-1)*S + k] — the same floats as make_tw.
static std::vector<float2> make_pass_tw(uint32_t M) {
    const std::vector<float2> tw = make_tw(M);
    std::vector<float2> t(M - 4);
    for (uint32_t S = 4; S < M; S *= 4)
        for (uint32_t r = 1; r <= 3; ++r)
            for (uint32_t k = 0; k < S; ++k) t[S - 4 + (r - 1) * S + k] = tw[(uint64_t)(k * r) * (M / (4 * S))];
    return t;
}

static std::vector<float> make_hann(uint32_t n) {  // chroma/extractor.rs:318-323, f32
    std::vector<float> w(n);
    const float pi = 3.14159265358979323846f;
    for (uint32_t i = 0; i < n; ++i) {
        const float x = 2.0f * pi * (float)i / (float)(n - 1);
        w[i] = 0.5f * (1.0f - cosf(x));
    }
    return w;
}

static void make_key_templates(std::vector<float>& major, std::vector<float>& minor, int template_set) {  // key/templates.rs:64-143 (K-K), 145-222 (Temperley)
    const float kk_maj[12] = {6.35f, 2.23f, 3.48f, 2.33f, 4.38f, 4.09f, 2.52f, 5.19f, 2.39f, 3.66f, 2.29f, 2.88f};
    const float kk_min[12] = {6.33f, 2.68f, 3.52f, 5.38f, 2.60f, 3.53f, 2.54f, 4.75f, 3.98f, 2.69f, 3.34f, 3.17f};
    const float tp_maj[12] = {5.0f, 2.0f, 3.5f, 2.0f, 4.5f, 4.0f, 2.0f, 4.5f, 2.0f, 3.5f, 1.5f, 4.0f};
    const float tp_min[12] = {5.0f, 2.0f, 3.5f, 5.0f, 2.0f, 3.5f, 2.0f, 4.5f, 3.5f, 2.0f, 4.0f, 3.5f};
    const float* cmaj = template_set == 1 ? tp_maj : kk_maj;
    const float* cmin = template_set == 1 ? tp_min : kk_min;
    major.assign(144, 0.0f);
    minor.assign(144, 0.0f);
    for (int k = 0; k < 12; ++k) {
        for (int s = 0; s < 12; ++s) {
            major[k * 12 + s] = cmaj[(s + 12 - k) % 12];
            minor[k * 12 + s] = cmin[(s + 12 - k) % 12];
        }
        for (std::vector<float>* v : {&major, &minor}) {
            float ss = 0.0f;
            for (int i = 0; i < 12; ++i) ss += (*v)[k * 12 + i] * (*v)[k * 12 + i];
            const float n = sqrtf(ss);
            if (n > 1e-12f)
                for (int i = 0; i < 12; ++i) (*v)[k * 12 + i] /= n;
        }
    }
}

static const float2* get_tw(DeviceCtx& c, uint32_t M) {
    auto it = c.tw_tables.find(M);
    if (it != c.tw_tables.end()) return it->second;
    float2* p = dev_upload(c, make_tw(M));
    c.tw_tables[M] = p;
    return p;
}

// Mel fold schedule for par_feat_kernel: the bands' entry lists cut into at most 64 chunks of near-equal length (two per lane), a
// band's chunks consecutive in `pos` order so that one lane per band can add their partial sums in order afterwards.  Layout of ck[256]:
// [0..64) first entry, [64..128) end entry, [128..192) position of the chunk's partial sum, [192..233) first position of each band.
// Slots are sorted by length (longest first: the first 32 go to the lanes' first round); idle slots are empty and point at positions
// no band reads.  mel_off = n_mels + 1 entry offsets (n_mels <= 40).
static void mel_fold_schedule(const int32_t* mel_off, uint32_t nm, int32_t* ck) {
    for (int i = 0; i < 256; ++i) ck[i] = 0;
    uint32_t C = 1;
    for (;; ++C) {
        uint32_t k = 0;
        for (uint32_t m = 0; m < nm; ++m) k += ((uint32_t)(mel_off[m + 1] - mel_off[m]) + C - 1) / C;
        if (k <= 64) break;
    }
    struct Chunk { int32_t a, e, pos; };
    std::vector<Chunk> chunks;
    int32_t pos = 0;
    for (uint32_t m = 0; m < nm; ++m) {
        ck[192 + m] = pos;
        const uint32_t n = (uint32_t)(mel_off[m + 1] - mel_off[m]);
        const uint32_t k = (n + C - 1) / C;
        int32_t a = mel_off[m];
        for (uint32_t j = 0; j < k; ++j) {
            const int32_t len = (int32_t)(n / k + (j < n % k ? 1 : 0));
            chunks.push_back({a, a + len, pos++});
            a += len;
        }
    }
    for (uint32_t m = nm; m <= 40; ++m) ck[192 + m] = pos;
    std::stable_sort(chunks.begin(), chunks.end(), [](const Chunk& x, const Chunk& y) { return x.e - x.a > y.e - y.a; });
    for (size_t i = 0; i < 64; ++i) {
        const Chunk ch = i < chunks.size() ? chunks[i] : Chunk{0, 0, (int32_t)std::min<size_t>(i, 63)};  // idle slots write a partial nobody reads (positions >= the chunk count)
        ck[i] = ch.a;
        ck[64 + i] = ch.e;
        ck[128 + i] = ch.pos;
    }
}

// tables of the generic STFT for frame size n (a power of two); win == nullptr on allocation failure
static GenStft get_gen_stft(DeviceCtx& c, uint32_t n) {
    GenStft g{};
    auto it = c.hann_tables.find(n);
    if (it == c.hann_tables.end()) it = c.hann_tables.emplace(n, dev_upload(c, make_hann(n))).first;
    g.win = it->second;
    g.tw = get_tw(c, n / 2);
    g.rw = get_tw(c, n);
    g.n = (g.win && g.tw && g.rw) ? n : 0;
    return g;
}

// The BPM hypotheses of the reference's grid loops, `bpm = min_bpm; while bpm <= limit { ..; bpm += bpm_resolution }` in f32:
// limit = max_bpm in the autocorrelation tempogram (tempogram_autocorr.rs:79-178), max_bpm + 1e-10 in the comb filterbank
// (comb_filter.rs:96-215).  The count and the values come from the accumulation, not from (max - min) / res: 40..240 at 0.1 gives
// 2000 hypotheses, and at 0.01 the last values are 5 steps away from min + i * res.  Writes the first min(count, cap) values and
// returns the count, or -1 beyond BPM_GRID_MAX hypotheses.  That includes every grid whose accumulation stalls (bpm_resolution
// below half an ulp of bpm), on which the reference never terminates.
static int bpm_grid(float min_bpm, float limit, float res, float* out, int cap) {
    int n = 0;
    for (float bpm = min_bpm; bpm <= limit; bpm = bpm + res) {
        if (n == BPM_GRID_MAX) return -1;
        if (n < cap) out[n] = bpm;
        ++n;
    }
    return n;
}

// Hypothesis table of a fine BPM grid (the comb filterbank's loop: it covers the tempogram's), uploaded once per grid.
static const float* get_bpm_tab(DeviceCtx& c, const DevCfg& d) {
    const std::array<float, 3> key{d.min_bpm, d.max_bpm, d.bpm_resolution};
    auto it = c.bpm_tabs.find(key);
    if (it != c.bpm_tabs.end()) return it->second;
    std::vector<float> tab(std::max(d.n_bpm, d.n_comb));
    bpm_grid(d.min_bpm, d.max_bpm + 1e-10f, d.bpm_resolution, tab.data(), (int)tab.size());
    const float* p = dev_upload(c, tab);
    if (p) c.bpm_tabs[key] = p;
    return p;
}

static int ctx_init(DeviceCtx& c, int device) {
    CUDA_OK(cudaSetDevice(device));
    c.device = device;
    CUDA_OK(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    CUDA_OK(cudaStreamCreateWithFlags(&c.key_stream, cudaStreamNonBlocking));
    c.tab.tw1024 = get_tw(c, 1024);
    c.tab.tw4096 = get_tw(c, 4096);
    {
        const std::vector<float2> p1 = make_pass_tw(1024), p4 = make_pass_tw(4096);
        c.tab.ptw1024 = dev_upload(c, p1);
        c.tab.ptw4096 = dev_upload(c, p4);
        stft_upload_constants(p1.data(), p4.data());
    }
    c.tab.rw2048 = get_tw(c, 2048);  // RW_N[k] = TW_N[k], k <= N/2
    c.tab.rw8192 = get_tw(c, 8192);
    {   // mirror symmetry of the real-split table (k_stft.cu: stft_key12_kernel reads one entry per bin pair when it holds)
        const std::vector<float2> rw = make_tw(8192);
        bool sym = true;
        for (uint32_t k = 1; k < 2048 && sym; ++k) sym = rw[4096 - k].x == -rw[k].x && rw[4096 - k].y == rw[k].y;
        c.tab.rw8192_sym = sym ? 1 : 0;
    }
    {
        const std::vector<float2> rw = make_tw(2048);
        bool sym = true;
        for (uint32_t k = 1; k < 512 && sym; ++k) sym = rw[1024 - k].x == -rw[k].x && rw[1024 - k].y == rw[k].y;
        c.tab.rw2048_sym = sym ? 1 : 0;
    }
    c.tab.win2048 = dev_upload(c, make_hann(2048));
    c.tab.win8192 = dev_upload(c, make_hann(8192));
    std::vector<float> mj, mn;
    make_key_templates(mj, mn, 0);
    c.tab.key_major = dev_upload(c, mj);
    c.tab.key_minor = dev_upload(c, mn);
    make_key_templates(mj, mn, 1);
    c.tab.key_major_tp = dev_upload(c, mj);
    c.tab.key_minor_tp = dev_upload(c, mn);
    CUDA_OK(cudaMalloc(&c.d_srtab, sizeof(SrTables) * DeviceCtx::MAX_SR));
    CUDA_OK(cudaMalloc(&c.d_count, sizeof(int32_t) * 4));
    CUDA_OK(cudaEventCreateWithFlags(&c.ev_legacy, cudaEventDisableTiming));
    if (!c.tab.tw1024 || !c.tab.tw4096 || !c.tab.ptw1024 || !c.tab.ptw4096 || !c.tab.rw2048 || !c.tab.rw8192 || !c.tab.win2048 || !c.tab.win8192 || !c.tab.key_major || !c.tab.key_minor ||
        !c.tab.key_major_tp || !c.tab.key_minor_tp) {
        set_error("device table allocation failed");
        return STRATUM_PROCESSING_ERROR;
    }
    c.ready = true;
    return STRATUM_OK;
}

static DeviceCtx* get_ctx(int device, int* status) {
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        set_error("no CUDA device is usable (stratum_b200 has no CPU fallback)");
        *status = STRATUM_PROCESSING_ERROR;
        return nullptr;
    }
    if (device < 0) {
        if (cudaGetDevice(&device) != cudaSuccess) device = 0;
    }
    if (device >= n) {
        set_error("device id out of range");
        *status = STRATUM_INVALID_INPUT;
        return nullptr;
    }
    DeviceCtx*& c = g_ctx[device];
    if (!c) c = new DeviceCtx();
    if (!c->ready) {
        const int st = ctx_init(*c, device);
        if (st != STRATUM_OK) {
            *status = st;
            return nullptr;
        }
    }
    *status = STRATUM_OK;
    return c;
}

// ---- per-sample-rate tables ------------------------------------------------------------------------------
static long f32_as_isize(float x) {
    if (!(x == x)) return 0;
    if (x >= 9.2233715e18f) return INT64_MAX;
    if (x <= -9.2233715e18f) return INT64_MIN;
    return (long)x;
}
static uint32_t hz_to_bin(float hz, float res, uint32_t n_bins) {  // period/tempogram.rs:279-289
    if (!std::isfinite(hz) || hz <= 0.0f || !std::isfinite(res) || res <= 0.0f) return 0;
    long b = f32_as_isize(roundf(hz / res));
    long hi = (long)n_bins - 1;
    if (hi < 0) hi = 0;
    return (uint32_t)std::max<long>(0, std::min<long>(b, hi));
}

// Bins b in [1, key_bins - 2] with fmin <= b * res <= fmax, the peak-search range of frame_to_hpcp (chroma/extractor.rs:584-591);
// lo > hi = empty.
static void hpcp_band_bins(uint32_t sr, uint32_t key_frame, float fmin, float fmax, uint32_t* lo_out, uint32_t* hi_out) {
    const uint32_t key_bins = key_frame / 2 + 1;
    const float res = (float)sr / (float)key_frame;
    uint32_t lo = 1, hi = 0;
    if (fmax > fmin) {
        lo = 0;
        for (uint32_t b = 1; b + 1 < key_bins; ++b) {
            const float f = (float)b * res;
            if (f < fmin) continue;
            if (f > fmax) break;
            if (lo == 0) lo = b;
            hi = b;
        }
        if (lo == 0) {
            lo = 1;
            hi = 0;
        }
    }
    *lo_out = lo;
    *hi_out = hi;
}

// Columns of the compact masked band (k_key.cu, key_compact): the HPCP peak search reads one bin either side of its band(s); the
// first column is rounded down to a multiple of 32 bins so that a warp of the mask kernel stores one full 128-byte line.
static void compact_band(uint32_t sr, const StratumConfig& cfg, uint32_t key_frame, uint32_t* lo_out, uint32_t* stride_out) {
    const uint32_t key_bins = key_frame / 2 + 1;
    const float nyq = (float)sr / 2.0f;
    uint32_t lo, hi;
    hpcp_band_bins(sr, key_frame, fmaxf(100.0f, 20.0f), fminf(5000.0f, nyq), &lo, &hi);
    if (cfg.enable_key_hpcp_bass_blend) {
        uint32_t bl, bh;
        hpcp_band_bins(sr, key_frame, fmaxf(cfg.key_hpcp_bass_fmin_hz, 20.0f), fminf(cfg.key_hpcp_bass_fmax_hz, nyq), &bl, &bh);
        if (bl <= bh) {
            if (lo > hi) { lo = bl; hi = bh; }
            else { lo = std::min(lo, bl); hi = std::max(hi, bh); }
        }
    }
    if (lo > hi) {
        *lo_out = 0;
        *stride_out = 32;
        return;
    }
    const uint32_t first = (lo - 1) & ~31u;
    const uint32_t end = std::min(hi + 2, key_bins);  // one past the last column read
    *lo_out = first;
    *stride_out = (uint32_t)align_up(end - first, 32);
    // one stride for every sample rate whose band fits (>= 39.2 kHz with 8192-point key frames): mask_kernel<.., BS = 960> then addresses
    // the band rows with immediates; 44.1 kHz needs 960 anyway, 48 kHz would need 864
    if (key_frame == 8192 && *stride_out <= 960) *stride_out = 960;
}

static bool key_compact_mode(const StratumConfig& c) {  // see DevCfg::key_compact
    static const bool off = getenv("STRATUM_B200_KEY_COMPACT") && atoi(getenv("STRATUM_B200_KEY_COMPACT")) == 0;  // A/B switch for measurements
    if (off) return false;
    const bool mask_runs = !c.enable_key_hpss_harmonic && (c.enable_key_harmonic_mask || (c.enable_key_spectrogram_time_smoothing && c.key_spectrogram_smooth_margin > 0));
    return mask_runs && c.enable_key_hpcp && !c.enable_key_log_frequency && !c.enable_key_beat_synchronous && !c.enable_key_hpcp_whitening &&
           !c.enable_key_tuning_compensation;
}

static int sr_slot(DeviceCtx& c, uint32_t sr, const StratumConfig& cfg, int* slot_out) {
    for (size_t i = 0; i < c.sr_host.size(); ++i)
        if (c.sr_host[i].sr == sr && memcmp(&c.sr_cfg[i], &cfg, sizeof cfg) == 0) {
            *slot_out = (int)i;
            return STRATUM_OK;
        }
    if ((int)c.sr_host.size() >= DeviceCtx::MAX_SR) {
        set_error("too many distinct (sample rate, configuration) pairs in one batch (max 32)");
        return STRATUM_NOT_IMPLEMENTED;
    }
    SrTables st{};
    st.sr = sr;
    const uint32_t key_frame = cfg.enable_key_stft_override ? std::max<uint32_t>(cfg.key_stft_frame_size, 256) : cfg.frame_size;  // lib.rs:984-989
    const uint32_t key_bins = key_frame / 2 + 1;
    const uint32_t n_bins = cfg.frame_size / 2 + 1;  // tempo-path STFT bins (the novelty curves' spectrogram)
    const float freq_res = (float)sr / (float)cfg.frame_size;
    uint32_t vm = 1u;  // full
    // band edges — period/tempogram.rs:356-372
    const uint32_t b0 = 1;
    const uint32_t b_low = std::max(hz_to_bin(cfg.tempogram_band_low_max_hz, freq_res, n_bins), b0);
    const uint32_t b_mid = std::max(hz_to_bin(cfg.tempogram_band_mid_max_hz, freq_res, n_bins), b_low + 1);
    uint32_t b_hi = cfg.tempogram_band_high_max_hz > 0.0f ? std::max(hz_to_bin(cfg.tempogram_band_high_max_hz, freq_res, n_bins), b_mid + 1) : n_bins;
    b_hi = std::min(b_hi, n_bins);
    st.b0 = b0;
    st.b_low = std::min(b_low, n_bins);
    st.b_mid = std::min(b_mid, n_bins);
    st.b_hi = b_hi;
    if (cfg.enable_tempogram_band_fusion) {
        const uint32_t s[3] = {st.b0, st.b_low, st.b_mid}, e[3] = {st.b_low, st.b_mid, st.b_hi};
        const float w[3] = {cfg.tempogram_band_w_low, cfg.tempogram_band_w_mid, cfg.tempogram_band_w_high};
        for (int b = 0; b < 3; ++b)
            if (std::isfinite(w[b]) && w[b] > 0.0f && e[b] > s[b] + 1) vm |= 1u << (1 + b);
    }
    // mel filterbank — period/novelty.rs:72-190.  Stored per band as the entries the reference's per-bin
    // contribution lists yield for that band in ascending-bin order: rising slope (l+1..c), then falling slope
    // (c..r-1) — the centre bin contributes twice with weight 1, exactly as the two loops of novelty.rs:150-175 do.
    std::vector<int32_t> mel_off(1, 0), mel_bin;
    std::vector<float> mel_w;
    st.n_mels = 0;
    if (cfg.enable_tempogram_mel_novelty) {
        const uint32_t n_mels = std::max<uint32_t>(cfg.tempogram_mel_n_mels, 4);
        if (n_mels > 40) {
            set_error("tempogram_mel_n_mels > 40 is not supported");
            return STRATUM_NOT_IMPLEMENTED;
        }
        auto mel_of = [](float hz) { return 2595.0f * log10f(1.0f + hz / 700.0f); };
        auto inv_mel = [](float m) { return 700.0f * (powf(10.0f, m / 2595.0f) - 1.0f); };
        const float nyq = (float)sr * 0.5f;
        const float fmin = fminf(fmaxf(cfg.tempogram_mel_fmin_hz, 0.0f), fmaxf(nyq, 1.0f));
        float fmax = cfg.tempogram_mel_fmax_hz;
        if (!(std::isfinite(fmax) && fmax > 0.0f)) fmax = nyq;
        {
            const float lo = fmin + 1.0f;
            if (fmax < lo) fmax = lo;
            if (fmax > nyq) fmax = nyq;
        }
        const float res = (float)sr / (float)cfg.frame_size;
        const float mmin = mel_of(fmin), mmax = mel_of(fmax);
        const float step = (mmax - mmin) / (float)(n_mels + 1);
        std::vector<uint32_t> pts(n_mels + 2);
        for (uint32_t i = 0; i < n_mels + 2; ++i) {
            const float hz = inv_mel(mmin + step * (float)i);
            long b = f32_as_isize(roundf(hz / res));
            b = std::max<long>(0, std::min<long>(b, (long)n_bins - 1));
            pts[i] = (uint32_t)b;
        }
        for (size_t i = 1; i < pts.size(); ++i)
            if (pts[i] <= pts[i - 1]) pts[i] = std::min(pts[i - 1] + 1, n_bins - 1);
        for (uint32_t m = 0; m < n_mels; ++m) {
            const uint32_t l = pts[m], cc = pts[m + 1], r = pts[m + 2];
            if (l < cc && cc < r) {
                for (uint32_t b = l; b <= cc; ++b) {
                    const float w = (b == l) ? 0.0f : ((float)b - (float)l) / ((float)cc - (float)l);
                    if (w > 0.0f) { mel_bin.push_back((int32_t)b); mel_w.push_back(w); }
                }
                for (uint32_t b = cc; b <= r; ++b) {
                    const float w = (b == r) ? 0.0f : ((float)r - (float)b) / ((float)r - (float)cc);
                    if (w > 0.0f) { mel_bin.push_back((int32_t)b); mel_w.push_back(w); }
                }
            }
            mel_off.push_back((int32_t)mel_bin.size());
        }
        st.n_mels = n_mels;
        vm |= 1u << 4;
    }
    mel_off.resize(42, mel_off.back());
    if (mel_bin.empty()) { mel_bin.push_back(0); mel_w.push_back(0.0f); }
    st.variant_mask = vm;
    {
        std::vector<int32_t> ck(256, 0);
        mel_fold_schedule(mel_off.data(), st.n_mels, ck.data());
        st.mel_chunks = dev_upload(c, ck);
    }
    st.mel_off = dev_upload(c, mel_off);
    st.mel_bin = dev_upload(c, mel_bin);
    st.mel_w = dev_upload(c, mel_w);
    // HPCP band in key-STFT bins — chroma/extractor.rs:584-591 (b from 1 to n_bins-2)
    hpcp_band_bins(sr, key_frame, fmaxf(100.0f, 20.0f), fminf(5000.0f, (float)sr / 2.0f), &st.key_bin_lo, &st.key_bin_hi);
    {   // bands and tables of the optional key-path variants (SURVEY §8a a39), key-STFT bins
        const float res = (float)sr / (float)key_frame;
        const float nyq = (float)sr / 2.0f;
        // bass-band HPCP: same peak loop as above on [bass_fmin, bass_fmax] (extractor.rs:1206-1220 -> 551-556, 584-591)
        st.bass_fmin = fmaxf(cfg.key_hpcp_bass_fmin_hz, 20.0f);
        st.bass_fmax = fminf(cfg.key_hpcp_bass_fmax_hz, nyq);
        hpcp_band_bins(sr, key_frame, st.bass_fmin, st.bass_fmax, &st.bass_bin_lo, &st.bass_bin_hi);
        st.white_n = std::min<uint32_t>(std::max(st.key_bin_hi, st.bass_bin_hi) + 2, key_bins);
        // tuning estimator band (extractor.rs:100-121): all bins with fmin <= f <= fmax
        {
            const float fmin = fmaxf(80.0f, 20.0f);
            const float fmax = fminf(fmaxf(2000.0f, fmin + 1.0f), nyq);  // clamp(fmin + 1, nyq)
            st.tune_bin_lo = 1;
            st.tune_bin_hi = 0;
            bool first = true;
            for (uint32_t b = 0; b < key_bins; ++b) {
                const float f = (float)b * res;
                if (f < fmin) continue;
                if (f > fmax) break;
                if (first) { st.tune_bin_lo = b; first = false; }
                st.tune_bin_hi = b;
            }
        }
        // median-HPSS band (extractor.rs:1408-1420)
        {
            const float fmin = fmaxf(100.0f, 20.0f);
            const float fmax = fminf(fmaxf(5000.0f, fmin + 1.0f), nyq);
            long bs = (long)floorf(fmin / res), be = (long)ceilf(fmax / res);
            bs = std::min<long>(std::max<long>(bs, 0), (long)key_bins);
            be = std::min<long>(std::max<long>(be, 0), (long)key_bins);
            st.hpss_b0 = (uint32_t)bs;
            st.hpss_band = be > bs ? (uint32_t)(be - bs) : 0u;
        }
        // log-frequency resampling (extractor.rs:733-803): per semitone bin, the (linear bin, weight) entries in ascending
        // linear-bin order — the order in which the reference adds them
        {
            const float fmin = fmaxf(100.0f, 20.0f), fmax = fminf(5000.0f, nyq - 1.0f);
            const float smin = 12.0f * log2f(fmin / 440.0f) + 57.0f, smax = 12.0f * log2f(fmax / 440.0f) + 57.0f;
            const long bmin = (long)floorf(smin), bmax = (long)ceilf(smax);
            const long nsl = bmax - bmin + 1;
            const uint32_t n_semi = nsl > 0 ? (uint32_t)nsl : 0u;
            st.log_n = n_semi;
            st.log_offset = (int32_t)floorf(12.0f * log2f(100.0f / 440.0f) + 57.0f);  // lib.rs:1076-1079
            std::vector<std::vector<std::pair<int32_t, float>>> per(n_semi);
            for (uint32_t b = 0; b < key_bins && n_semi > 0; ++b) {
                const float f = (float)b * res;
                if (f < fmin || f >= fmax || f >= nyq) continue;
                const float semitone = 12.0f * log2f(f / 440.0f) + 57.0f;
                const float x = semitone - (float)bmin;
                const float fl = floorf(x), ce = ceilf(x);
                const uint32_t lo = fl > 0.0f ? (uint32_t)fl : 0u;
                const uint32_t hi = std::min<uint32_t>(ce > 0.0f ? (uint32_t)ce : 0u, n_semi - 1);
                if (lo < n_semi) {
                    const float wh = x - (float)lo, wl = 1.0f - wh;
                    per[lo].push_back({(int32_t)b, wl});
                    if (hi != lo && hi < n_semi) per[hi].push_back({(int32_t)b, wh});
                }
            }
            std::vector<int32_t> off(n_semi + 1, 0), bins;
            std::vector<float> ws;
            for (uint32_t q = 0; q < n_semi; ++q) {
                for (auto& e : per[q]) {
                    bins.push_back(e.first);
                    ws.push_back(e.second);
                }
                off[q + 1] = (int32_t)bins.size();
            }
            if (bins.empty()) { bins.push_back(0); ws.push_back(0.0f); }
            if (cfg.enable_key_log_frequency && n_semi > 128) {
                set_error("log-frequency key spectrogram with more than 128 semitone bins is not supported");
                return STRATUM_NOT_IMPLEMENTED;
            }
            st.log_off = dev_upload(c, off);
            st.log_bin = dev_upload(c, bins);
            st.log_w = dev_upload(c, ws);
        }
    }
    {   // KWeightingFilter::new — normalization.rs:127-155 (single RBJ high-pass biquad), f32 like the reference
        const float pi = 3.14159265358979323846f;
        const float w0 = 2.0f * pi * 1681.9745f / (float)sr;
        const float cw = cosf(w0), sw = sinf(w0);
        const float alpha = sw / 2.0f * sqrtf(1.0f / 0.707f);
        const float B0 = (1.0f + cw) / 2.0f, B1 = -(1.0f + cw), B2 = (1.0f + cw) / 2.0f;
        const float a0 = 1.0f + alpha, A1 = -2.0f * cw, A2 = 1.0f - alpha;
        st.kw_b0 = B0 / a0;
        st.kw_b1 = B1 / a0;
        st.kw_b2 = B2 / a0;
        st.kw_a1 = A1 / a0;
        st.kw_a2 = A2 / a0;
        const float blk = (float)sr * 400.0f / 1000.0f;  // normalization.rs:198
        st.lufs_block = blk > 0.0f ? (uint32_t)blk : 0u;
    }
    {   // chroma folding (extractor.rs:393-487): the bin -> pitch-class weights do not depend on the frame, so they are
        // tabulated per pitch class in ascending-bin order (the order in which the reference adds them)
        std::vector<int32_t> off(13, 0), bins;
        std::vector<float> ws;
        std::vector<std::vector<std::pair<int32_t, float>>> per(12);
        const float res = (float)sr / (float)key_frame;
        uint32_t lo = 1, hi = 0;
        bool first = true;
        for (uint32_t b = 0; b < key_bins; ++b) {
            const float freq = (float)b * res;
            if (freq < 100.0f) continue;
            if (freq > fminf(5000.0f, (float)sr / 2.0f)) break;
            if (freq >= (float)sr / 2.0f) break;
            if (first) { lo = b; first = false; }
            hi = b;
            const float semitone = 12.0f * log2f(freq / 440.0f) + 57.0f - 0.0f;
            if (cfg.soft_chroma_mapping) {
                float spc = fmodf(semitone, 12.0f);
                if (spc < 0.0f) spc += 12.0f;
                float ppc = fmodf(roundf(spc), 12.0f);
                if (ppc < 0.0f) ppc += 12.0f;
                const int primary = (int)ppc;
                for (int o = -1; o <= 1; ++o) {
                    const int tc = ((primary + o) % 12 + 12) % 12;
                    float dist = fabsf(spc - (float)tc);
                    dist = fminf(dist, 12.0f - dist);
                    const float sigma = fmaxf(cfg.soft_mapping_sigma, 1e-6f);
                    per[tc].push_back({(int32_t)b, expf(-dist * dist / (2.0f * sigma * sigma))});
                }
            } else {
                int cls = (int)roundf(semitone) % 12;
                if (cls < 0) cls += 12;
                per[cls].push_back({(int32_t)b, 1.0f});
            }
        }
        for (int tc = 0; tc < 12; ++tc) {
            for (auto& e : per[tc]) {
                bins.push_back(e.first);
                ws.push_back(e.second);
            }
            off[tc + 1] = (int32_t)bins.size();
        }
        if (bins.empty()) { bins.push_back(0); ws.push_back(0.0f); }
        // The HPCP front end handles any band (2048 peak slots cover a whole 8192-point row).  Plain chroma folding, its tuned and
        // beat-synchronous forms, HPCP whitening and the median-HPSS key mask keep per-frame tables of 1024 band bins, which the
        // 100..5000 Hz band exceeds when sr / key_frame < 4.79 Hz (below 39.2 kHz with the default 8192-point key STFT).
        const bool fixed_tables = !cfg.enable_key_hpcp || cfg.enable_key_beat_synchronous || cfg.enable_key_tuning_compensation || cfg.enable_key_hpcp_whitening ||
                                  cfg.enable_key_hpss_harmonic;
        if (fixed_tables && hi >= lo && hi - lo + 1 > 1024) {
            char msg[256];
            snprintf(msg, sizeof msg,
                     "sample rate %u Hz is not supported with this key configuration: the 100..5000 Hz band spans %u key-STFT bins (max 1024; the default HPCP key path has no such limit)",
                     sr, hi - lo + 1);
            set_error(msg);
            return STRATUM_NOT_IMPLEMENTED;
        }
        st.fold_lo = lo;
        st.fold_hi = hi;
        st.fold_off = dev_upload(c, off);
        st.fold_bin = dev_upload(c, bins);
        st.fold_w = dev_upload(c, ws);
    }
    c.sr_host.push_back(st);
    c.sr_cfg.push_back(cfg);
    *slot_out = (int)c.sr_host.size() - 1;
    if (cudaMemcpy(c.d_srtab, c.sr_host.data(), sizeof(SrTables) * c.sr_host.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
        set_error("sr table upload failed");
        return STRATUM_PROCESSING_ERROR;
    }
    return STRATUM_OK;
}

// ---- configuration -----------------------------------------------------------------------------------------
static void config_default(StratumConfig* c) {  // src/config.rs:594-744
    memset(c, 0, sizeof *c);
    c->abi_version = STRATUM_B200_ABI_VERSION;
    c->min_amplitude_db = -40.0f;
    c->normalization = STRATUM_NORM_PEAK;
    c->enable_normalization = 1;
    c->enable_silence_trimming = 1;
    c->enable_onset_consensus = 1;
    c->onset_threshold_percentile = 0.80f;
    c->onset_consensus_tolerance_ms = 50;
    for (int i = 0; i < 4; ++i) c->onset_consensus_weights[i] = 0.25f;
    c->enable_legacy_bpm_guardrails = 1;
    c->enable_tempogram_multi_resolution = 1;
    c->tempogram_multi_res_top_k = 25;
    c->tempogram_multi_res_w512 = 0.45f;
    c->tempogram_multi_res_w256 = 0.35f;
    c->tempogram_multi_res_w1024 = 0.20f;
    c->tempogram_multi_res_structural_discount = 0.85f;
    c->tempogram_multi_res_double_time_512_factor = 0.92f;
    c->tempogram_multi_res_margin_threshold = 0.08f;
    c->enable_tempogram_band_fusion = 1;
    c->tempogram_band_low_max_hz = 200.0f;
    c->tempogram_band_mid_max_hz = 2000.0f;
    c->tempogram_band_high_max_hz = 8000.0f;
    c->tempogram_band_w_full = 0.40f;
    c->tempogram_band_w_low = 0.25f;
    c->tempogram_band_w_mid = 0.20f;
    c->tempogram_band_w_high = 0.15f;
    c->tempogram_band_seed_only = 1;
    c->tempogram_band_support_threshold = 0.25f;
    c->tempogram_band_consensus_bonus = 0.08f;
    c->tempogram_novelty_w_spectral = 0.30f;
    c->tempogram_novelty_w_energy = 0.35f;
    c->tempogram_novelty_w_hfc = 0.35f;
    c->tempogram_novelty_local_mean_window = 16;
    c->tempogram_novelty_smooth_window = 5;
    c->enable_tempogram_mel_novelty = 1;
    c->tempogram_mel_n_mels = 40;
    c->tempogram_mel_fmin_hz = 30.0f;
    c->tempogram_mel_fmax_hz = 8000.0f;
    c->tempogram_mel_max_filter_bins = 2;
    c->tempogram_mel_weight = 0.15f;
    c->tempogram_superflux_max_filter_bins = 4;
    c->tempogram_candidates_top_n = 10;
    c->legacy_bpm_preferred_min = 72.0f;
    c->legacy_bpm_preferred_max = 168.0f;
    c->legacy_bpm_soft_min = 60.0f;
    c->legacy_bpm_soft_max = 210.0f;
    c->legacy_bpm_conf_mul_preferred = 1.30f;
    c->legacy_bpm_conf_mul_soft = 0.70f;
    c->legacy_bpm_conf_mul_extreme = 0.01f;
    c->min_bpm = 40.0f;
    c->max_bpm = 240.0f;
    c->bpm_resolution = 1.0f;
    c->frame_size = 2048;
    c->hop_size = 512;
    c->soft_mapping_sigma = 0.5f;
    c->key_spectrogram_smooth_margin = 12;
    c->enable_key_frame_weighting = 1;
    c->key_min_tonalness = 0.0f;
    c->key_tonalness_power = 2.0f;
    c->key_energy_power = 0.50f;
    c->enable_key_harmonic_mask = 1;
    c->key_harmonic_mask_power = 2.0f;
    c->enable_key_stft_override = 1;
    c->key_stft_frame_size = 8192;
    c->key_stft_hop_size = 512;
    c->enable_key_segment_voting = 1;
    c->key_segment_len_frames = 1024;
    c->key_segment_hop_frames = 512;
    c->key_segment_min_clarity = 0.20f;
    c->enable_key_hpcp = 1;
    c->key_hpcp_peaks_per_frame = 24;
    c->key_hpcp_num_harmonics = 4;
    c->key_hpcp_harmonic_decay = 0.60f;
    c->key_hpcp_mag_power = 0.50f;
    c->chroma_sharpening_power = 1.0f;
    c->hpss_margin = 10;
    c->soft_chroma_mapping = 1;
    c->enable_key_spectrogram_time_smoothing = 1;
    c->key_template_set = 0;
    c->key_edge_trim_fraction = 0.15f;
    c->key_mode_third_ratio_margin = 0.0f;
    c->key_mode_flip_min_score_ratio = 0.60f;
    c->key_minor_leading_tone_bonus_weight = 0.2f;
    c->key_ensemble_kk_weight = 0.5f;
    c->key_ensemble_temperley_weight = 0.5f;
    c->key_multi_scale_n_lengths = 3;
    c->key_multi_scale_lengths[0] = 120;
    c->key_multi_scale_lengths[1] = 360;
    c->key_multi_scale_lengths[2] = 720;
    c->key_multi_scale_hop = 60;
    c->key_multi_scale_min_clarity = 0.20f;
    c->key_multi_scale_n_weights = 0;
    c->key_median_segment_length_frames = 480;
    c->key_median_segment_hop_frames = 120;
    c->key_median_min_segments = 3;
    c->key_tuning_max_abs_semitones = 0.08f;
    c->key_tuning_frame_step = 20;
    c->key_tuning_peak_rel_threshold = 0.35f;
    c->key_hpss_frame_step = 4;
    c->key_hpss_time_margin = 8;
    c->key_hpss_freq_margin = 8;
    c->key_hpss_mask_power = 2.0f;
    c->key_hpcp_whitening_smooth_bins = 31;
    c->key_hpcp_bass_fmin_hz = 55.0f;
    c->key_hpcp_bass_fmax_hz = 300.0f;
    c->key_hpcp_bass_weight = 0.35f;
}

// Rejects configurations whose branch is not built (SURVEY §8a a39) instead of silently ignoring them.
static int config_validate(const StratumConfig& c) {
    auto ni = [](const char* what) {
        set_error(std::string("not implemented in the B200 path: ") + what);
        return (int)STRATUM_NOT_IMPLEMENTED;
    };
    if (c.abi_version != STRATUM_B200_ABI_VERSION) {
        set_error("StratumConfig.abi_version mismatch");
        return STRATUM_INVALID_INPUT;
    }
    if (c.enable_normalization && (c.normalization < STRATUM_NORM_PEAK || c.normalization > STRATUM_NORM_LOUDNESS)) {
        set_error("unknown normalization method");
        return STRATUM_INVALID_INPUT;
    }
    if ((c.enable_hpss_onsets || c.enable_tempogram_percussive_fallback) && c.hpss_margin > 10) return ni("hpss_margin > 10");
    if (c.emit_tempogram_candidates && c.tempogram_candidates_top_n > 200) return ni("tempogram_candidates_top_n > 200");
    if (!tempo_frame_supported(c.frame_size)) return ni("frame_size other than 2048, 4096 or 8192");
    if (c.hop_size == 0) {
        set_error("Hop size must be > 0");
        return STRATUM_INVALID_INPUT;
    }
    if (c.hop_size < 32 || c.hop_size > 16384) return ni("hop_size outside 32..16384");  // (work areas are sized by the frame count)
    if (c.enable_key_stft_override) {  // any power of two from 256 (lib.rs:986 clamps below) to 8192; 2048 and 8192 have fused kernels
        const uint32_t kf = std::max<uint32_t>(c.key_stft_frame_size, 256);
        if ((kf & (kf - 1)) != 0 || kf > 8192) return ni("key_stft_frame_size that is not a power of two between 256 and 8192");
    }
    if (c.key_spectrogram_smooth_margin > 15) return ni("key_spectrogram_smooth_margin > 15");
    if (c.key_hpcp_peaks_per_frame > 32) return ni("key_hpcp_peaks_per_frame > 32");
    if (c.key_hpcp_num_harmonics > 8) return ni("key_hpcp_num_harmonics > 8");
    if (c.tempogram_superflux_max_filter_bins > 8) return ni("tempogram_superflux_max_filter_bins > 8");
    if (c.tempogram_multi_res_top_k > 32) return ni("tempogram_multi_res_top_k > 32");
    // enable_key_median is accepted and has no effect, as in the reference: analyze_audio never reads it (lib.rs imports no detect_key_median)
    if (c.enable_key_hpss_harmonic && (c.key_hpss_time_margin > 10 || c.key_hpss_freq_margin > 10)) return ni("key_hpss_time_margin / key_hpss_freq_margin > 10");
    if (c.enable_key_hpcp_whitening && c.key_hpcp_whitening_smooth_bins > 63) return ni("key_hpcp_whitening_smooth_bins > 63");
    if (c.key_template_set != 0 && c.key_template_set != 1) {
        set_error("unknown key_template_set");
        return STRATUM_INVALID_INPUT;
    }
    if (c.key_multi_scale_n_lengths > 8 || c.key_multi_scale_n_weights > 8) return ni("more than 8 multi-scale lengths / weights");
    if (!(c.min_bpm > 0.0f) || !(c.max_bpm > c.min_bpm) || !(c.bpm_resolution > 0.0f)) {
        set_error("Invalid BPM range");
        return STRATUM_INVALID_INPUT;
    }
    // the comb filterbank's loop bound is the larger one, so its count bounds both grids
    if (bpm_grid(c.min_bpm, c.max_bpm + 1e-10f, c.bpm_resolution, nullptr, 0) < 0)
        return ni(("more than " + std::to_string(BPM_GRID_MAX) + " BPM hypotheses (bpm_resolution too fine for the BPM range)").c_str());
    if (!(c.onset_threshold_percentile >= 0.0f && c.onset_threshold_percentile <= 1.0f)) {
        set_error("Threshold percentile must be in [0, 1]");
        return STRATUM_INVALID_INPUT;
    }
    if (c.onset_consensus_tolerance_ms == 0) {
        set_error("Tolerance must be > 0");
        return STRATUM_INVALID_INPUT;
    }
    return STRATUM_OK;
}

static DevCfg make_devcfg(const StratumConfig& c) {
    DevCfg d{};
    d.min_bpm = c.min_bpm;
    d.max_bpm = c.max_bpm;
    d.bpm_resolution = c.bpm_resolution;
    d.n_bpm = (uint32_t)std::max(bpm_grid(c.min_bpm, c.max_bpm, c.bpm_resolution, nullptr, 0), 0);
    d.n_comb = (uint32_t)std::max(bpm_grid(c.min_bpm, c.max_bpm + 1e-10f, c.bpm_resolution, nullptr, 0), 0);
    d.ac_stride = std::max<uint32_t>(AC_CAP, d.n_bpm);
    d.bpm_tab = nullptr;  // device table: Session::open, for grids of more than AC_CAP hypotheses
    d.silence_thr_linear = powf(10.0f, c.min_amplitude_db / 20.0f);
    d.silence_min_ms = 500;
    d.energy_thr_mul = powf(10.0f, -20.0f / 20.0f);
    d.target_peak = powf(10.0f, (0.0f - 1.0f) / 20.0f);
    d.rms_target = powf(10.0f, ((-14.0f + 3.0f) - 1.0f) / 20.0f);  // normalize(.., target_lufs = -14, headroom = 1): normalization.rs:532, 345
    d.normalization = c.normalization;
    d.enable_normalization = c.enable_normalization;
    d.enable_trim = c.enable_silence_trimming;
    d.enable_consensus = c.enable_onset_consensus;
    d.onset_pct = c.onset_threshold_percentile;
    d.consensus_tol_ms = c.onset_consensus_tolerance_ms;
    for (int i = 0; i < 4; ++i) d.cons_w[i] = c.onset_consensus_weights[i];
    d.hpss_onsets = c.enable_hpss_onsets;
    d.perc_fallback = c.enable_tempogram_percussive_fallback && c.enable_tempogram_multi_resolution && !c.force_legacy_bpm;
    d.hpss_margin = c.hpss_margin;
    d.sf_k = c.tempogram_superflux_max_filter_bins;
    d.mel_k = c.tempogram_mel_max_filter_bins;
    d.nov_ws = c.tempogram_novelty_w_spectral;
    d.nov_we = c.tempogram_novelty_w_energy;
    d.nov_wh = c.tempogram_novelty_w_hfc;
    d.nov_lmw = c.tempogram_novelty_local_mean_window;
    d.nov_smw = c.tempogram_novelty_smooth_window;
    d.band_fusion = c.enable_tempogram_band_fusion;
    d.mel_enabled = c.enable_tempogram_mel_novelty;
    d.seed_only = c.tempogram_band_seed_only;
    d.w_full = c.tempogram_band_w_full;
    d.w_low = c.tempogram_band_w_low;
    d.w_mid = c.tempogram_band_w_mid;
    d.w_high = c.tempogram_band_w_high;
    d.w_mel = c.tempogram_mel_weight;
    d.support_thr = c.tempogram_band_support_threshold;
    d.consensus_bonus = c.tempogram_band_consensus_bonus;
    // lib.rs:382-385 / multi_resolution.rs:230-234
    const uint32_t base_top_n = std::max(std::max(c.tempogram_candidates_top_n, c.tempogram_multi_res_top_k), 10u);
    d.base_top_n = c.enable_tempogram_multi_resolution ? base_top_n : (c.emit_tempogram_candidates ? c.tempogram_candidates_top_n : 0);  // lib.rs:378-410, 714-737
    d.emit_cands = c.emit_tempogram_candidates;
    d.mr_top_k = std::max(c.tempogram_multi_res_top_k, 1u);
    d.mr_aux_k = std::min(std::max(d.mr_top_k * 4, 25u), 200u);
    d.mr_w512 = c.tempogram_multi_res_w512;
    d.mr_w256 = c.tempogram_multi_res_w256;
    d.mr_w1024 = c.tempogram_multi_res_w1024;
    d.mr_dt = c.tempogram_multi_res_double_time_512_factor;
    d.mr_margin = c.tempogram_multi_res_margin_threshold;
    d.mr_human_prior = c.tempogram_multi_res_use_human_prior;
    d.mr_enabled = c.enable_tempogram_multi_resolution;
    d.force_legacy = c.force_legacy_bpm;
    d.legacy_guardrails = c.enable_legacy_bpm_guardrails;
    d.bpm_fusion = c.enable_bpm_fusion;
    d.lg_pmin = c.legacy_bpm_preferred_min;
    d.lg_pmax = c.legacy_bpm_preferred_max;
    d.lg_smin = c.legacy_bpm_soft_min;
    d.lg_smax = c.legacy_bpm_soft_max;
    d.lg_mp = c.legacy_bpm_conf_mul_preferred;
    d.lg_ms = c.legacy_bpm_conf_mul_soft;
    d.lg_me = c.legacy_bpm_conf_mul_extreme;
    d.key_margin = c.key_spectrogram_smooth_margin;
    d.key_mask_power = c.key_harmonic_mask_power;
    d.key_mask = c.enable_key_harmonic_mask;
    d.key_smooth_only = !c.enable_key_harmonic_mask && c.enable_key_spectrogram_time_smoothing && c.key_spectrogram_smooth_margin > 0;
    d.key_hpcp = c.enable_key_hpcp;
    d.key_compact = key_compact_mode(c);
    d.chroma_sharpen = c.chroma_sharpening_power;
    d.key_weighting = c.enable_key_frame_weighting;
    d.key_voting = c.enable_key_segment_voting;
    d.key_min_tonal = c.key_min_tonalness;
    d.key_tonal_pow = c.key_tonalness_power;
    d.key_energy_pow = c.key_energy_power;
    d.key_seg_len = c.key_segment_len_frames;
    d.key_seg_hop = c.key_segment_hop_frames;
    d.key_seg_min_clarity = c.key_segment_min_clarity;
    d.hpcp_peaks = c.key_hpcp_peaks_per_frame;
    d.hpcp_harm = c.key_hpcp_num_harmonics;
    d.hpcp_decay = c.key_hpcp_harmonic_decay;
    d.hpcp_pow = c.key_hpcp_mag_power;
    d.hpcp_sigma = c.soft_mapping_sigma;
    d.hop = c.hop_size;
    d.frame = c.frame_size;
    d.bins = c.frame_size / 2 + 1;
    d.bs = c.hop_size == 512 ? 0 : SLOT_BASE_ALT;  // the base path shares slot 0 with the multi-resolution pass only at hop 512
    d.key_frame = c.enable_key_stft_override ? std::max<uint32_t>(c.key_stft_frame_size, 256) : c.frame_size;  // lib.rs:984-995
    d.key_hop = c.enable_key_stft_override ? std::max<uint32_t>(c.key_stft_hop_size, 1) : c.hop_size;
    d.key_bins = d.key_frame / 2 + 1;
    d.key_stride = key_compact_mode(c) ? (d.key_bins + 7) / 8 * 8 : d.key_bins;  // compact mode: only the STFT writes and the mask reads these rows
    d.key_mode = c.enable_key_ensemble ? KEY_ROWS_ENSEMBLE : (c.enable_key_multi_scale ? KEY_ROWS_MULTI_SCALE : KEY_ROWS_VOTE);
    d.key_template_set = c.key_template_set;
    d.key_edge_trim = c.enable_key_edge_trim;
    d.key_edge_frac = c.key_edge_trim_fraction;
    d.key_heur = c.enable_key_mode_heuristic || c.enable_key_minor_harmonic_bonus;
    d.key_third_margin = c.key_mode_third_ratio_margin;
    d.key_flip_ratio = c.enable_key_mode_heuristic ? c.key_mode_flip_min_score_ratio : 0.0f;
    d.key_minor_bonus = c.enable_key_minor_harmonic_bonus;
    d.key_minor_bonus_w = c.key_minor_leading_tone_bonus_weight;
    d.key_ens_kk = c.key_ensemble_kk_weight;
    d.key_ens_tp = c.key_ensemble_temperley_weight;
    d.ms_n = std::min<uint32_t>(c.key_multi_scale_n_lengths, 8);
    d.ms_nw = std::min<uint32_t>(c.key_multi_scale_n_weights, 8);
    for (int i = 0; i < 8; ++i) {
        d.ms_len[i] = c.key_multi_scale_lengths[i];
        d.ms_w[i] = c.key_multi_scale_weights[i];
    }
    d.ms_hop = c.key_multi_scale_hop;
    d.ms_min_clarity = c.key_multi_scale_min_clarity;
    d.key_tuning = c.enable_key_tuning_compensation;
    d.tune_max_abs = c.key_tuning_max_abs_semitones;
    d.tune_thr = c.key_tuning_peak_rel_threshold;
    d.tune_step = c.key_tuning_frame_step;
    d.key_whiten = c.enable_key_hpcp_whitening && c.key_hpcp_whitening_smooth_bins >= 3;
    d.whiten_half = (std::max<uint32_t>(c.key_hpcp_whitening_smooth_bins, 3) | 1u) / 2;
    d.key_bass_blend = c.enable_key_hpcp_bass_blend;
    d.bass_weight = c.key_hpcp_bass_weight;
    d.key_log_freq = c.enable_key_log_frequency;
    d.key_beat_sync = c.enable_key_beat_synchronous;
    d.key_soft_mapping = c.soft_chroma_mapping;
    d.key_hpss = c.enable_key_hpss_harmonic;
    d.khpss_step = c.key_hpss_frame_step;
    d.khpss_tm = c.key_hpss_time_margin;
    d.khpss_fm = c.key_hpss_freq_margin;
    d.khpss_power = c.key_hpss_mask_power;
    return d;
}

// ---- arena planning -----------------------------------------------------------------------------------------
struct Bump {
    uint64_t pos = 0;
    uint64_t take(uint64_t n, uint64_t al = 32) {
        pos = align_up(pos, al);
        const uint64_t p = pos;
        pos += n;
        return p;
    }
};

static void plan_hop(Bump& fa, HopLayout& H, uint32_t fcap, uint32_t hop, const DevCfg& kd, bool with_spec = true) {
    H.fmax = fcap;
    H.hop = hop;
    H.fft_cap = std::max<uint32_t>(next_pow2_u32(fcap > 1 ? fcap - 1 : 1), 4);
    H.spec = with_spec ? fa.take((uint64_t)fcap * kd.bins) : 0;
    H.frame = fa.take((uint64_t)FRAME_Q * fcap);
    H.pair = fa.take((uint64_t)PAIR_Q * fcap);
    H.nov = fa.take((uint64_t)MAX_VARIANTS * fcap);
    H.tgfft = fa.take((uint64_t)MAX_VARIANTS * (H.fft_cap / 2 + 1));
    H.tgac = fa.take((uint64_t)MAX_VARIANTS * kd.ac_stride);
    H.tgwork = fa.take((uint64_t)MAX_VARIANTS * 2 * H.fft_cap);
    H.tgtw = nullptr;
    H.pad_ = 0;
}

// Base (always needed) work areas of one track.
static void plan_track(Bump& fa, Bump& oa, Bump& ia, TrackDev& T, const StratumConfig& cfg, const DevCfg& kd) {
    const uint64_t n = T.n;
    const uint32_t F512 = frames_of(n, kd.frame, 512), F256 = frames_of(n, kd.frame, 256), F1024 = frames_of(n, kd.frame, 1024);
    const uint32_t Fk = frames_of(n, kd.key_frame, kd.key_hop);
    const uint32_t Fsil = n >= kd.frame ? frames_of(n, kd.frame, kd.frame / 2) : 1;
    const uint32_t Fb = frames_of(n, kd.frame, kd.hop);  // frames of the base path (= F512 at the default hop_size)
    T.fall = std::max(std::max(std::max(F256, F512), std::max(F1024, 1u)), Fb);
    T.fkmax = Fk;
    plan_hop(fa, T.hop[0], std::max(F512, 1u), 512, kd);
    T.cands[0] = fa.take((uint64_t)MAX_CANDS * 4);
    if (kd.bs != 0) {  // hop_size other than 512: the base path gets a slot of its own
        plan_hop(fa, T.hop[SLOT_BASE_ALT], std::max(Fb, 1u), kd.hop, kd);
        T.cands[SLOT_BASE_ALT] = fa.take((uint64_t)MAX_CANDS * 4);
    }
    T.sil_rms = fa.take(Fsil + 1);
    T.erms = fa.take(std::max(F512, Fb) + 2);
    T.scratch = fa.take((uint64_t)12 * T.fall);
    T.keyspec = fa.take((uint64_t)Fk * kd.key_stride + 8, 32);
    T.keymask = T.keyspec;  // the mask is applied in place (or, key_compact: only its HPCP band is kept, in kband)
    if (kd.key_compact) {
        compact_band(T.sr, cfg, kd.key_frame, &T.kband_lo, &T.kband_stride);
        T.kband = fa.take((uint64_t)Fk * T.kband_stride + 32, 32);
        T.kprefix = fa.take((uint64_t)MASK_SEG_MAX * kd.key_stride, 32);
        T.kepart_stride = (uint32_t)align_up(Fk + 1, 32);
        T.kepart = fa.take((uint64_t)((kd.key_bins + 31) / 32) * T.kepart_stride, 32);  // one row per warp of the mask kernel
    }
    T.chroma = fa.take((uint64_t)Fk * 12 + 12);
    T.chroma2 = fa.take((uint64_t)Fk * 12 + 12);
    T.kenergy = fa.take(Fk + 1);
    T.kweights = fa.take(Fk + 1);
    // score rows (key_rows.cuh); the row count is monotone in the frame count, so the untrimmed Fk bounds every trimmed / edge-trimmed slice
    if (cfg.enable_key_hpcp_whitening && cfg.enable_key_hpcp && !cfg.enable_key_log_frequency) {  // whitened magnitudes of the peak bands
        T.kwhite_stride = 1056;  // >= white_n (the 100..5000 Hz band is at most 1024 key-STFT bins wide at the accepted sample rates)
        T.kwhite = fa.take((uint64_t)Fk * T.kwhite_stride + 8);
    }
    if (cfg.enable_key_hpss_harmonic) {  // harmonic soft mask on the time-downsampled band
        const uint32_t step = std::max<uint32_t>(cfg.key_hpss_frame_step, 1);
        T.khpss_mask = fa.take((uint64_t)((Fk + step - 1) / step + 1) * 1032);
    }
    if (cfg.enable_key_tuning_compensation) {  // per-track chroma-folding lists (tuned mapping)
        T.kfold_w = fa.take((uint64_t)12 * 1024);
        T.kfold_bin = ia.take((uint64_t)12 * 1024 + 16);
    }
    T.seg_cap = key_rows(Fk, kd).nrows + 1;
    T.seg_scores = fa.take((uint64_t)T.seg_cap * 24);
    T.seg_avg = fa.take((uint64_t)T.seg_cap * 13);
    T.seg_rank = fa.take((uint64_t)T.seg_cap * 28);
    // onsets: each detector yields at most every other flux sample
    const uint32_t on_cap = std::max(F512, Fb) / 2 + 8;
    T.on_energy = ia.take(on_cap);
    T.on_spectral = ia.take(on_cap);
    T.on_hfc = ia.take(on_cap);
    T.on_merged = 0;
    T.on_hpss = 0;
    const bool hpss = cfg.enable_hpss_onsets || cfg.enable_tempogram_percussive_fallback;
    if (hpss) {  // HPSS work areas (onset/hpss.rs): two ping-pong pairs of F x bins and the feature slot of the percussive part
        T.on_hpss = ia.take(on_cap);
        for (int q = 0; q < 2; ++q) {
            T.hpss_h[q] = fa.take((uint64_t)std::max(Fb, 1u) * kd.bins);
            T.hpss_p[q] = fa.take((uint64_t)std::max(Fb, 1u) * kd.bins);
        }
        plan_hop(fa, T.hop[SLOT_PERC], std::max(Fb, 1u), kd.hop, kd, false);
        T.cands[SLOT_PERC] = fa.take((uint64_t)MAX_CANDS * 4);
    }
    T.on_final = ia.take((uint64_t)(hpss ? 4 : 3) * on_cap);
    // beat tracker: bpm <= 300 -> at most 5 beat frames per second
    const double dur = (double)n / (double)std::max(T.sr, 1u);
    T.hmm_cap = (uint32_t)std::ceil(dur * 5.0) + 8;
    T.beat_cap = 3 * T.hmm_cap + 64;
    T.onsets_s = fa.take((uint64_t)3 * on_cap);
    T.hmm_em = fa.take(T.hmm_cap);
    T.beats_tmp = fa.take((uint64_t)3 * T.beat_cap);
    T.hmm_frames = ia.take(T.hmm_cap);
    T.hmm_bp = ia.take(T.hmm_cap);
    T.hmm_path = ia.take(T.hmm_cap);
    T.beats = oa.take(T.beat_cap);
    T.downbeats = oa.take(T.beat_cap);
    T.cand_out = cfg.emit_tempogram_candidates ? oa.take((uint64_t)5 * MAX_TOPC) : 0;
    T.n_cand_out = -1;
    // legacy ACF: next_pow2(2 * (max_frame + 1)), max_frame <= n / 512
    T.lg_fft = next_pow2_u32((uint32_t)(2 * (n / kd.hop + 1)));
    T.lg_work = fa.take((uint64_t)4 * T.lg_fft);
    T.lg_comb = fa.take(std::max(kd.n_comb, 1u));
    T.lg_tw = nullptr;
    T.lg_pad = 0;
    T.lufs_nb = T.lufs_block = 0;
    T.lufs_z = T.lufs_s = T.lufs_e = 0;
    if (cfg.enable_normalization && cfg.normalization == STRATUM_NORM_LOUDNESS && n > 0) {
        const float blk = (float)T.sr * 400.0f / 1000.0f;  // normalization.rs:198
        T.lufs_block = blk >= 1.0f ? (uint32_t)blk : 0u;
        if (T.lufs_block) {
            T.lufs_nb = (uint32_t)((n + T.lufs_block - 1) / T.lufs_block);
            T.lufs_z = fa.take(2 * (uint64_t)T.lufs_nb + 2);
            T.lufs_s = fa.take(2 * (uint64_t)T.lufs_nb + 2);
            T.lufs_e = fa.take((uint64_t)T.lufs_nb + 1);
        }
    }
}

static void plan_escalation(Bump& fa, TrackDev& T, const DevCfg& kd) {
    plan_hop(fa, T.hop[1], std::max(frames_of(T.n, kd.frame, 256), 1u), 256, kd);
    T.cands[1] = fa.take((uint64_t)MAX_CANDS * 4);
    plan_hop(fa, T.hop[2], std::max(frames_of(T.n, kd.frame, 1024), 1u), 1024, kd);
    T.cands[2] = fa.take((uint64_t)MAX_CANDS * 4);
}

static int ensure_capacity(DeviceCtx& c, size_t fa_need, size_t oa_need, size_t ia_need, size_t tracks) {
    auto grow = [&](void** p, size_t* cap, size_t need, size_t elt) -> int {
        if (need <= *cap) return STRATUM_OK;
        if (*p) cudaFree(*p);
        *p = nullptr;
        *cap = 0;
        CUDA_OK(cudaMalloc(p, need * elt));
        *cap = need;
        return STRATUM_OK;
    };
    int st;
    if ((st = grow((void**)&c.fa, &c.fa_cap, fa_need, 4))) return st;
    if ((st = grow((void**)&c.oa, &c.oa_cap, oa_need, 4))) return st;
    if ((st = grow((void**)&c.ia, &c.ia_cap, ia_need, 4))) return st;
    if (tracks > c.tr_cap) {
        if (c.d_tracks) cudaFree(c.d_tracks);
        if (c.d_sr_index) cudaFree(c.d_sr_index);
        if (c.d_list) cudaFree(c.d_list);
        if (c.d_gain) cudaFree(c.d_gain);
        c.d_gain = nullptr;
        c.d_tracks = nullptr;
        c.d_sr_index = c.d_list = nullptr;
        c.tr_cap = 0;
        CUDA_OK(cudaMalloc(&c.d_tracks, tracks * sizeof(TrackDev)));
        CUDA_OK(cudaMalloc(&c.d_sr_index, tracks * sizeof(int32_t)));
        CUDA_OK(cudaMalloc(&c.d_list, tracks * sizeof(int32_t)));
        CUDA_OK(cudaMalloc(&c.d_gain, tracks * sizeof(float)));
        c.tr_cap = tracks;
    }
    return STRATUM_OK;
}

static const char* error_message(int code) {
    switch (code) {
        case 1: return "Empty audio samples";                         // lib.rs:100-104
        case 2: return "Invalid sample rate";                         // lib.rs:106-110
        case 3: return "Audio is entirely silent after trimming";     // lib.rs:143-147
        case 4: return "Signal too short for autocorrelation";        // period/autocorrelation.rs:131-135 via lib.rs:315
        case 5: return "Track longer than 2^31 samples is not supported";
        default: return "processing error";
    }
}

static void fill_result(const TrackDev& T, const float* oa_host, const int32_t* ia_host, float ms_per_track, const char* custom_err, StratumResult* r) {
    memset(r, 0, sizeof *r);
    r->status = T.status;
    r->tempogram_multi_res_triggered = r->tempogram_multi_res_used = -1;
    r->tempogram_percussive_triggered = r->tempogram_percussive_used = -1;
    r->time_sig_beats_per_bar = 4;
    r->n_tempogram_candidates = -1;
    if (T.status != 0) {
        snprintf(r->error, sizeof r->error, "%s", custom_err ? custom_err : error_message(T.err_code));
        return;
    }
    r->bpm = T.bpm;
    r->bpm_confidence = T.bpm_confidence;
    r->key_is_minor = T.key >= 12;
    r->key_index = (uint32_t)(T.key % 12);
    r->key_confidence = T.key_confidence;
    r->key_clarity = T.key_clarity;
    r->grid_stability = T.grid_stability;
    auto copy_f = [&](uint64_t off, uint32_t n) -> float* {
        if (n == 0) return nullptr;
        float* p = (float*)malloc(sizeof(float) * n);
        memcpy(p, oa_host + off, sizeof(float) * n);
        return p;
    };
    r->beats = copy_f(T.beats, T.n_beats);
    r->n_beats = T.n_beats;
    r->downbeats = copy_f(T.downbeats, T.n_downbeats);
    r->n_downbeats = T.n_downbeats;
    r->bars = copy_f(T.downbeats, T.n_downbeats);  // bars = downbeats.clone() (beat_tracking/mod.rs:316)
    r->n_bars = T.n_downbeats;
    r->duration_seconds = (float)T.m / (float)T.sr;
    r->sample_rate = T.sr;
    r->processing_time_ms = ms_per_track;
    r->onset_method_consensus = T.onset_method_consensus;
    // warnings / flags — lib.rs:1567-1589
    if (T.bpm == 0.0f) r->warnings |= STRATUM_WARN_BPM_FAILED;
    if (T.grid_stability < 0.5f) r->warnings |= STRATUM_WARN_LOW_GRID_STABILITY;
    if (T.key_confidence < 0.3f) r->warnings |= STRATUM_WARN_LOW_KEY_CONFIDENCE;
    if (T.key_clarity < 0.2f) {
        r->warnings |= STRATUM_WARN_LOW_KEY_CLARITY;
        r->flags |= STRATUM_FLAG_WEAK_TONALITY;
    }
    r->tempogram_multi_res_triggered = T.mr_triggered;
    r->tempogram_multi_res_used = T.mr_used;
    r->tempogram_percussive_triggered = T.perc_triggered;
    r->tempogram_percussive_used = T.perc_used;
    r->trim_start = T.trim_start;
    r->trim_end = T.trim_end;
    r->n_onsets = T.n_on_final;
    if (T.n_on_final) {
        r->onsets = (int64_t*)malloc(sizeof(int64_t) * T.n_on_final);
        for (uint32_t i = 0; i < T.n_on_final; ++i) r->onsets[i] = ia_host[T.on_final + i];
    }
    r->n_hmm_beat_frames = T.n_hmm_frames;
    if (T.n_hmm_frames) {
        r->hmm_beat_frames = (int32_t*)malloc(sizeof(int32_t) * T.n_hmm_frames);
        memcpy(r->hmm_beat_frames, ia_host + T.hmm_frames, sizeof(int32_t) * T.n_hmm_frames);
    }
    r->time_sig_beats_per_bar = T.time_sig;
    r->beats_refined = T.beats_refined;
    r->n_tempogram_candidates = T.n_cand_out;
    if (T.n_cand_out > 0) {
        r->tempogram_candidates = (StratumTempoCandidate*)malloc(sizeof(StratumTempoCandidate) * T.n_cand_out);
        for (int32_t i = 0; i < T.n_cand_out; ++i) {
            const float* o = oa_host + T.cand_out + 5 * (size_t)i;
            r->tempogram_candidates[i] = StratumTempoCandidate{o[0], o[1], o[2], o[3], o[4] != 0.0f ? 1 : 0};
        }
    }
}

static void debug_put(const char* name, const float* d, size_t n, cudaStream_t s) {
    std::vector<float> h(n);
    if (n) cudaMemcpyAsync(h.data(), d, n * sizeof(float), cudaMemcpyDeviceToHost, s);
    cudaStreamSynchronize(s);
    std::lock_guard<std::mutex> lk(g_debug_mu);
    g_debug_arrays[name] = std::move(h);
}
static void debug_put_i(const char* name, const int32_t* d, size_t n, cudaStream_t s) {
    std::vector<int32_t> h(n);
    if (n) cudaMemcpyAsync(h.data(), d, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s);
    cudaStreamSynchronize(s);
    std::vector<float> f(h.begin(), h.end());
    std::lock_guard<std::mutex> lk(g_debug_mu);
    g_debug_arrays[name] = std::move(f);
}

static uint64_t esc_floats(uint64_t n, const DevCfg& kd) {
    TrackDev T{};
    T.n = n;
    Bump b;
    plan_escalation(b, T, kd);
    return align_up(b.pos, 64);
}

// ---- one wave ----------------------------------------------------------------------------------------------------
struct WavePlan {
    std::vector<uint32_t> idx;  // track indices of the batch in this wave
    uint64_t fa_base = 0, oa = 0, ia = 0;
    uint64_t esc_each_max = 0;  // largest escalation footprint of a track in the wave
};

// stream `waiter` continues only after everything queued on `signaller` so far
static void stream_wait(cudaStream_t waiter, cudaStream_t signaller) {
    cudaEvent_t e;
    if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return;
    cudaEventRecord(e, signaller);
    cudaStreamWaitEvent(waiter, e, 0);
    cudaEventDestroy(e);  // released once the record has completed
}

// On an error return from the middle of a wave: let both streams drain (queued kernels still reference the arenas and the
// host buffers of this call) and drop the stage-timer events of the launches made so far.
struct WaveAbortGuard {
    DeviceCtx& c;
    bool armed = true;
    explicit WaveAbortGuard(DeviceCtx& c_) : c(c_) {}
    ~WaveAbortGuard() {
        if (!armed) return;
        cudaStreamSynchronize(c.stream);
        cudaStreamSynchronize(c.key_stream);
        for (PendingStage& p : g_pending) {
            cudaEventDestroy(p.a);
            cudaEventDestroy(p.b);
        }
        g_pending.clear();
    }
};

static void debug_dump_wave(DeviceCtx& c, const WaveJob& job);

// Queues every launch of one wave and its final read-back.  `mid` runs on the host once the first part of the wave (everything up
// to the escalation gate) is queued and before the host waits for the escalated-track count — the one point inside a wave where
// the host needs a device value; the caller gathers the previous wave and starts the next upload there.
static int wave_begin(DeviceCtx& c, const float* d_samples, const uint64_t* sample_off, const uint64_t* lens, const uint32_t* srs, const WavePlan& wp,
                      const StratumConfig& cfg, const DevCfg& dcfg, size_t fa_budget, StratumResult* out, WaveJob& job, const std::function<int()>& mid) {
    const int nt = (int)wp.idx.size();
    HostSpan span_plan("host_plan");
    job.nt = nt;
    job.idx = wp.idx;
    job.out = out;
    job.dcfg = dcfg;
    job.track_err.assign(nt, std::string());
    job.debug_single = g_debug.load() && nt == 1;
    TrackDev* tracks = static_cast<TrackDev*>(job.h_tracks.need(sizeof(TrackDev) * nt));
    if (!tracks) {
        set_error("pinned host allocation failed");
        return STRATUM_PROCESSING_ERROR;
    }
    int32_t* sr_index = static_cast<int32_t*>(job.h_small.need(sizeof(int32_t) * nt));  // pinned: a pageable source would make the copy wait for the stream
    if (!sr_index) {
        set_error("pinned host allocation failed");
        return STRATUM_PROCESSING_ERROR;
    }
    memset(sr_index, 0, sizeof(int32_t) * nt);
    Bump fa, oa, ia;
    WaveCtx w{};
    w.stream = c.stream;
    w.samples = d_samples;
    w.n_tracks = nt;
    w.tab = c.tab;
    w.cfg = dcfg;
    w.max_key_peaks = 1;
    if (dcfg.key_frame != 2048 && dcfg.key_frame != 8192) {
        w.gen_key = get_gen_stft(c, dcfg.key_frame);
        if (w.gen_key.n == 0) {
            set_error("table allocation failed");
            return STRATUM_PROCESSING_ERROR;
        }
    }
    if (dcfg.frame == 4096) {  // the tempo-path STFT takes the generic kernel at this size (k_stft.cu: launch_stft_hop)
        w.gen_tempo = get_gen_stft(c, dcfg.frame);
        if (w.gen_tempo.n == 0) {
            set_error("table allocation failed");
            return STRATUM_PROCESSING_ERROR;
        }
    }
    bool kband_seen = false;
    const bool mr_on = dcfg.mr_enabled && !dcfg.force_legacy;
    for (int i = 0; i < nt; ++i) {
        TrackDev& T = tracks[i];
        memset(&T, 0, sizeof T);
        const uint32_t gi = wp.idx[i];
        T.off = sample_off[gi];
        T.n = lens[gi];
        T.sr = srs[gi];
        T.status = 0;
        T.mr_triggered = T.mr_used = T.perc_triggered = T.perc_used = -1;
        if (T.n == 0) { T.status = STRATUM_INVALID_INPUT; T.err_code = 1; }
        else if (T.sr == 0) { T.status = STRATUM_INVALID_INPUT; T.err_code = 2; }
        else if (T.n >= (1ull << 31)) { T.status = STRATUM_NOT_IMPLEMENTED; T.err_code = 5; }
        if (T.status == 0) {
            int slot = 0;
            const int st = sr_slot(c, T.sr, cfg, &slot);
            if (st == STRATUM_OK) {
                sr_index[i] = slot;
                const SrTables& S = c.sr_host[slot];
                w.max_key_peaks = std::max(w.max_key_peaks, S.key_bin_hi >= S.key_bin_lo ? (S.key_bin_hi - S.key_bin_lo + 2) / 2 : 0u);
                w.max_key_peaks = std::max(w.max_key_peaks, S.bass_bin_hi >= S.bass_bin_lo ? (S.bass_bin_hi - S.bass_bin_lo + 2) / 2 : 0u);
            } else {  // this track fails with the table builder's message; the rest of the wave carries on (analyze_batch.rs:293-322)
                T.status = st;
                T.err_code = 6;
                job.track_err[i] = g_last_error;
            }
        }
        if (T.status != 0) {
            T.n = 0;
            T.sr = T.sr ? T.sr : 1;
        }
        plan_track(fa, oa, ia, T, cfg, dcfg);
        if (T.status == 0 && T.kband_stride != w.kband_stride_common) w.kband_stride_common = kband_seen ? 0u : T.kband_stride;
        if (T.status == 0) kband_seen = true;
        T.hop[0].tgtw = get_tw(c, T.hop[0].fft_cap);
        if (dcfg.bs != 0) T.hop[SLOT_BASE_ALT].tgtw = get_tw(c, T.hop[SLOT_BASE_ALT].fft_cap);
        if (dcfg.hpss_onsets || dcfg.perc_fallback) T.hop[SLOT_PERC].tgtw = get_tw(c, T.hop[SLOT_PERC].fft_cap);
        T.lg_tw = get_tw(c, T.lg_fft);
        if (mr_on) {  // escalation work areas, relative to the start of whichever arena slot escalation_compact_kernel assigns
            Bump b;
            plan_escalation(b, T, dcfg);
            T.hop[1].tgtw = get_tw(c, T.hop[1].fft_cap);
            T.hop[2].tgtw = get_tw(c, T.hop[2].fft_cap);
        }
        if (!T.hop[0].tgtw || !T.hop[dcfg.bs].tgtw || !T.lg_tw || (mr_on && (!T.hop[1].tgtw || !T.hop[2].tgtw))) {
            set_error("twiddle table allocation failed");
            return STRATUM_PROCESSING_ERROR;
        }
        const uint32_t Fsil = T.n >= dcfg.frame ? frames_of(T.n, dcfg.frame, dcfg.frame / 2) : (T.n > 0 ? 1 : 0);
        T.Fsil = Fsil;
        // provisional (untrimmed) frame counts; trim_kernel rewrites them
        T.m = T.n;
        T.trim_start = 0;
        T.trim_end = T.n;
        w.max_F[0] = std::max(w.max_F[0], frames_of(T.n, dcfg.frame, 512));
        w.max_F[1] = std::max(w.max_F[1], frames_of(T.n, dcfg.frame, 256));
        w.max_F[2] = std::max(w.max_F[2], frames_of(T.n, dcfg.frame, 1024));
        w.max_F[SLOT_BASE_ALT] = std::max(w.max_F[SLOT_BASE_ALT], frames_of(T.n, dcfg.frame, dcfg.hop));
        w.max_F[SLOT_PERC] = w.max_F[dcfg.bs];
        w.max_Fk = std::max(w.max_Fk, frames_of(T.n, dcfg.key_frame, dcfg.key_hop));
        w.max_Fsil = std::max(w.max_Fsil, Fsil);
        w.max_n = std::max<uint64_t>(w.max_n, T.n);
        w.max_beat_cap = std::max(w.max_beat_cap, T.beat_cap);
        w.max_seg_cap = std::max(w.max_seg_cap, T.seg_cap);
        w.max_lg_fft = std::max(w.max_lg_fft, T.lg_fft);
        w.max_lufs_nb = std::max(w.max_lufs_nb, T.lufs_nb);
    }
    const uint64_t fa_base_end = align_up(fa.pos, 64);
    // escalation pool: whatever is left of the budget (at least one track's worth)
    uint64_t esc_each = 0;
    for (int i = 0; i < nt; ++i) esc_each = std::max<uint64_t>(esc_each, esc_floats(tracks[i].n, dcfg));
    uint64_t esc_slots = 0;
    if (mr_on) {
        const uint64_t room = fa_budget > fa_base_end ? fa_budget - fa_base_end : 0;
        esc_slots = esc_each ? std::min<uint64_t>(std::max<uint64_t>(room / esc_each, 1), (uint64_t)nt) : 0;
    }
    const uint64_t fa_total = fa_base_end + esc_slots * esc_each;
    int st = ensure_capacity(c, fa_total + 64, oa.pos + 64, ia.pos + 64, nt);
    if (st != STRATUM_OK) return st;
    job.oa_n = oa.pos;
    job.ia_n = ia.pos;
    float* oa_host = static_cast<float*>(job.h_oa.need(sizeof(float) * (oa.pos + 1)));
    int32_t* ia_host = static_cast<int32_t*>(job.h_ia.need(sizeof(int32_t) * (ia.pos + 1)));
    if (!oa_host || !ia_host) {
        set_error("pinned host allocation failed");
        return STRATUM_PROCESSING_ERROR;
    }
    if (!job.ev0 && (cudaEventCreate(&job.ev0) != cudaSuccess || cudaEventCreate(&job.ev1) != cudaSuccess)) {
        set_error("event creation failed");
        return STRATUM_PROCESSING_ERROR;
    }
    w.fa = c.fa;
    w.oa = c.oa;
    w.ia = c.ia;
    w.tracks = c.d_tracks;
    w.srtab = c.d_srtab;
    w.sr_index = c.d_sr_index;
    cudaStream_t s = c.stream;
    WaveAbortGuard guard(c);
    cudaEventRecord(job.ev0, s);
    CUDA_OK(cudaMemcpyAsync(c.d_tracks, tracks, sizeof(TrackDev) * nt, cudaMemcpyHostToDevice, s));
    CUDA_OK(cudaMemcpyAsync(c.d_sr_index, sr_index, sizeof(int32_t) * nt, cudaMemcpyHostToDevice, s));
    span_plan.stop();
    {
        StageTimer t(s, "preprocess");
        launch_peak(w);
        const float* d_gain = nullptr;
        if (dcfg.enable_normalization && dcfg.normalization == STRATUM_NORM_LOUDNESS) {
            // normalize_lufs (normalization.rs:401-484): gate, mean, log10 and the dB -> linear powf are evaluated on
            // the host (same libm as the reference's platform) from the device's block energies and peaks
            std::vector<TrackDev> rb(nt);
            CUDA_OK(cudaMemcpyAsync(rb.data(), c.d_tracks, sizeof(TrackDev) * nt, cudaMemcpyDeviceToHost, s));
            std::vector<std::vector<float>> en(nt);
            for (int i = 0; i < nt; ++i) {
                en[i].resize(tracks[i].lufs_nb);  // layout fields are host-planned
                if (tracks[i].lufs_nb && tracks[i].status == 0)
                    CUDA_OK(cudaMemcpyAsync(en[i].data(), c.fa + tracks[i].lufs_e, sizeof(float) * tracks[i].lufs_nb, cudaMemcpyDeviceToHost, s));
            }
            CUDA_OK(cudaStreamSynchronize(s));
            std::vector<float> gains(nt, 1.0f);
            const float gate = powf(10.0f, (-70.0f + 0.691f) / 10.0f);
            const float target_peak = powf(10.0f, (0.0f - 1.0f) / 20.0f);
            for (int i = 0; i < nt; ++i) {
                if (rb[i].status != 0) continue;
                const float peak = rb[i].peak;
                float acc = 0.0f;
                size_t cnt = 0;
                for (float e : en[i])
                    if (e > gate) {
                        acc += e;
                        ++cnt;
                    }
                float g = 1.0f;
                if (cnt == 0) {  // all blocks gated: fall back to peak normalisation (:417-424)
                    if (peak > 1e-10f) g = fminf(target_peak / peak, 1.0f / peak);
                } else {
                    const float mean = acc / (float)cnt;
                    const float lufs = -0.691f + 10.0f * log10f(mean);
                    g = powf(10.0f, (-14.0f - lufs) / 20.0f);
                    if (peak * g > target_peak) g = target_peak / peak;
                }
                gains[i] = g;
            }
            CUDA_OK(cudaMemcpyAsync(c.d_gain, gains.data(), sizeof(float) * nt, cudaMemcpyHostToDevice, s));
            CUDA_OK(cudaStreamSynchronize(s));  // `gains` is a stack-owned buffer
            d_gain = c.d_gain;
        }
        launch_gain(w, d_gain);
        launch_silence_trim(w);
    }
    // The key path (8192-point STFT -> harmonic mask -> HPCP -> vote) only needs the trimmed, normalised samples, so it
    // can run on its own stream beside the onset / tempo / beat path.  Measured on B200 (256 x 3-min tracks): 925
    // tracks/s with the two paths overlapped vs 970 one after the other — both are bound by the same SM resources
    // (issue slots, L1/shared pipe), so overlap only adds cache pressure.  Off unless STRATUM_B200_DUAL_STREAM is set.
    static const bool dual_stream = getenv("STRATUM_B200_DUAL_STREAM") != nullptr;
    const bool split = dual_stream && !job.debug_single && !dcfg.key_beat_sync;  // beat-synchronous chroma reads the beat grid
    // Late split (default): the key path and the legacy estimator are independent of the tempo path's tail, whose kernels are
    // small latency-bound grids (one CTA or warp per track: legacy ACF/comb, the hop-256/1024 tempograms and their fusion,
    // the final BPM, the beat tracker — about 45 ms of a 980 ms step).  The legacy estimator starts on the second stream as
    // soon as the consensus onsets exist; the key path is forked there after the last heavy tempo kernel (the multi-resolution
    // features), so those tails run beside the key STFT instead of in front of it.  Unlike the early split above, no two
    // bandwidth- or issue-heavy kernels ever overlap.
    static const bool no_late_split = getenv("STRATUM_B200_NO_LATE_SPLIT") != nullptr;
    const bool late = !split && !no_late_split && !job.debug_single && !dcfg.key_beat_sync;
    bool key_forked = false;
    auto run_key_path = [&](cudaStream_t ks) {
        WaveCtx wk = w;
        wk.stream = ks;
        { StageTimer t(ks, "stft_8192_key"); launch_stft_key(wk); }
        if (job.debug_single) {
            TrackDev T;
            cudaMemcpyAsync(&T, c.d_tracks, sizeof(TrackDev), cudaMemcpyDeviceToHost, ks);
            cudaStreamSynchronize(ks);
            const uint32_t nk = std::min<uint32_t>(T.Fk, 64);
            debug_put("key.spec_head", c.fa + T.keyspec, (size_t)nk * dcfg.key_stride, ks);  // rows of key_stride floats
        }
        { StageTimer t(ks, "key_mask"); launch_key_mask(wk); }
        { StageTimer t(ks, "key_hpcp"); launch_key_hpcp(wk); }
        { StageTimer t(ks, "key_vote"); launch_key_vote(wk); }
    };
    auto fork_key_path = [&]() {  // late split: everything the key path needs (gain, trim) was produced long ago on s
        if (!late || key_forked) return;
        key_forked = true;
        stream_wait(c.key_stream, s);
        run_key_path(c.key_stream);
    };
    if (split) {
        stream_wait(c.key_stream, s);
        run_key_path(c.key_stream);
    }
    if (late) {  // the energy-flux detector (a latency-bound add chain per frame) only feeds the consensus: beside the STFT
        stream_wait(c.key_stream, s);
        WaveCtx we = w;
        we.stream = c.key_stream;
        { StageTimer t(c.key_stream, "onsets_energy"); launch_energy_onsets(we); }
    } else {
        StageTimer t(s, "onsets_energy");
        launch_energy_onsets(w);
    }
    const int bs = dcfg.bs;  // the base path's slot
    { StageTimer t(s, "stft_2048_hop512"); launch_stft_hop(w, bs, nullptr, nt); }
    { StageTimer t(s, "spec_features"); launch_spec_features(w, bs, nullptr, nt); }
    if (dcfg.hpss_onsets) {  // lib.rs:222-235: onsets of the percussive component as the fourth detector
        StageTimer t(s, "hpss");
        launch_hpss(w, nullptr, nt);
        launch_seq_features(w, SLOT_PERC, nullptr, nt);
        launch_hpss_onsets(w);
    }
    if (late) stream_wait(s, c.key_stream);  // energy onsets
    { StageTimer t(s, "onsets_consensus"); launch_spectral_onsets_consensus(w); }
    const bool want_tempogram = !dcfg.force_legacy;
    if (want_tempogram) {
        StageTimer t(s, "tempogram");
        launch_tempogram(w, bs, nullptr, nt);
        launch_escalation_gate(w);
        if (dcfg.mr_enabled) launch_escalation_compact(w, c.d_list, c.d_count, fa_base_end, esc_each, (uint32_t)esc_slots);
    }
    bool legacy_on_key_stream = false;
    if (late) {  // needs the consensus onsets only; its result is read by final_bpm
        stream_wait(c.key_stream, s);
        WaveCtx wl = w;
        wl.stream = c.key_stream;
        { StageTimer t(c.key_stream, "legacy_bpm"); launch_legacy_bpm(wl); }
        cudaEventRecord(c.ev_legacy, c.key_stream);
        legacy_on_key_stream = true;
    } else {
        StageTimer t(s, "legacy_bpm");
        launch_legacy_bpm(w);
    }
    bool mid_done = false;
    auto run_mid = [&]() -> int {
        if (mid_done) return STRATUM_OK;
        mid_done = true;
        return mid ? mid() : (int)STRATUM_OK;
    };
    std::vector<TrackDev> gate_rb;  // records as of the gate (percussive fallback / debug only)
    if (want_tempogram && dcfg.mr_enabled) {
        // the only device value the host needs inside a wave: how many tracks escalate (sizes the multi-resolution grids)
        int32_t* h_count = static_cast<int32_t*>(c.h_count.need(sizeof(int32_t) * 4));
        if (!h_count) {
            set_error("pinned host allocation failed");
            return STRATUM_PROCESSING_ERROR;
        }
        CUDA_OK(cudaMemcpyAsync(h_count, c.d_count, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        if (dcfg.perc_fallback || job.debug_single) {
            gate_rb.resize(nt);
            CUDA_OK(cudaMemcpyAsync(gate_rb.data(), c.d_tracks, sizeof(TrackDev) * nt, cudaMemcpyDeviceToHost, s));
        }
        if ((st = run_mid()) != STRATUM_OK) return st;
        {
            HostSpan span_esc("host_escalation");  // time the host waits for the count with nothing else to do
            CUDA_OK(cudaStreamSynchronize(s));
        }
        const size_t n_esc = (size_t)std::max(0, std::min(h_count[0], nt));
        g_d2h_bytes.fetch_add(sizeof(int32_t));
        for (size_t p0 = 0; p0 < n_esc; p0 += esc_slots) {
            const size_t p1 = std::min(n_esc, p0 + (size_t)esc_slots);
            const int nl = (int)(p1 - p0);
            const int32_t* lst = c.d_list + p0;
            {
                StageTimer t(s, "stft_multires");
                if (bs != 0) launch_stft_hop(w, 0, lst, nl);  // hop_size is not 512: the pass needs its own hop-512 spectrogram (lib.rs:493-509)
                launch_stft_hop(w, 1, lst, nl);
                launch_stft_hop(w, 2, lst, nl);
            }
            {
                StageTimer t(s, "multires_features");
                if (bs != 0) launch_spec_features(w, 0, lst, nl);
                launch_spec_features(w, 1, lst, nl);
                launch_spec_features(w, 2, lst, nl);
            }
            if (late && p1 == n_esc) fork_key_path();  // last heavy kernel of the tempo path is queued: the key path starts behind it
            {
                StageTimer t(s, "multires_tempogram");
                if (bs != 0) launch_tempogram(w, 0, lst, nl);
                launch_tempogram(w, 1, lst, nl);
                launch_tempogram(w, 2, lst, nl);
                launch_multires_fusion(w, lst, nl);
            }
            if (job.debug_single) {
                TrackDev T;
                cudaMemcpyAsync(&T, c.d_tracks, sizeof(TrackDev), cudaMemcpyDeviceToHost, s);
                cudaStreamSynchronize(s);
                for (int h = 1; h < 3; ++h) {
                    const uint32_t L = T.F[h] > 0 ? T.F[h] - 1 : 0;
                    const std::string tag = h == 1 ? "h256." : "h1024.";
                    debug_put((tag + "nov.full").c_str(), c.fa + T.hop[h].nov, L, s);
                    debug_put((tag + "tg.fft.full").c_str(), c.fa + T.hop[h].tgfft, T.hop[h].fft_cap / 2 + 1, s);
                    debug_put((tag + "tg.ac.full").c_str(), c.fa + T.hop[h].tgac, dcfg.n_bpm, s);
                    debug_put((tag + "cands").c_str(), c.fa + T.cands[h], (size_t)MAX_CANDS * 4, s);
                }
            }
        }
    }
    if (want_tempogram && dcfg.mr_enabled && dcfg.perc_fallback) {
        // percussive tempogram fallback (lib.rs:587-683) for the tracks the gate put in the low-tempo trap; gate_rb was
        // read back after the gate, so perc_triggered is valid on the host
        std::vector<int32_t> pl;
        for (int i = 0; i < nt; ++i)
            if (gate_rb[i].status == 0 && gate_rb[i].perc_triggered == 1) pl.push_back(i);
        if (!pl.empty()) {
            StageTimer t(s, "percussive_fallback");
            const int nl = (int)pl.size();
            CUDA_OK(cudaMemcpyAsync(c.d_list, pl.data(), sizeof(int32_t) * nl, cudaMemcpyHostToDevice, s));
            if (!dcfg.hpss_onsets) launch_hpss(w, c.d_list, nl);
            launch_spec_features(w, SLOT_PERC, c.d_list, nl);
            launch_tempogram(w, SLOT_PERC, c.d_list, nl);
            launch_perc_accept(w, c.d_list, nl);
            CUDA_OK(cudaStreamSynchronize(s));  // `pl` is a stack-owned buffer
        }
    }
    if (late && !key_forked) fork_key_path();  // nothing escalated (or multi-resolution off): fork here
    if (legacy_on_key_stream) cudaStreamWaitEvent(s, c.ev_legacy, 0);  // not the whole key stream: the key path is queued behind the legacy estimator
    { StageTimer t(s, "final_bpm"); launch_final_bpm(w); launch_emit_candidates(w); }
    { StageTimer t(s, "beats"); launch_beat_tracking(w); }
    if (split || late) stream_wait(s, c.key_stream);
    else run_key_path(s);
    CUDA_OK(cudaMemcpyAsync(tracks, c.d_tracks, sizeof(TrackDev) * nt, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaMemcpyAsync(oa_host, c.oa, sizeof(float) * oa.pos, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaMemcpyAsync(ia_host, c.ia, sizeof(int32_t) * ia.pos, cudaMemcpyDeviceToHost, s));
    g_d2h_bytes.fetch_add(sizeof(TrackDev) * nt + sizeof(float) * oa.pos + sizeof(int32_t) * ia.pos);
    g_h2d_bytes.fetch_add((sizeof(TrackDev) + sizeof(int32_t)) * nt);
    cudaEventRecord(job.ev1, s);
    job.stages.swap(g_pending);
    g_pending.clear();
    guard.armed = false;
    job.active = true;
    return run_mid();  // waves without an escalation wait gather the previous wave here
}

// Waits for a queued wave and gathers its results.
static int wave_end(DeviceCtx& c, WaveJob& job, double* wave_ms) {
    if (!job.active) return STRATUM_OK;
    job.active = false;
    const cudaError_t e = cudaEventSynchronize(job.ev1);
    HostSpan span_gather("host_gather");
    resolve_stage_times(job.stages);
    if (e != cudaSuccess) {
        set_error(std::string("CUDA error: ") + cudaGetErrorString(e) + " while waiting for a wave");
        return STRATUM_PROCESSING_ERROR;
    }
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, job.ev0, job.ev1);
    if (wave_ms) *wave_ms += ms;
    const TrackDev* tracks = static_cast<const TrackDev*>(job.h_tracks.p);
    const float* oa_host = static_cast<const float*>(job.h_oa.p);
    const int32_t* ia_host = static_cast<const int32_t*>(job.h_ia.p);
    for (int i = 0; i < job.nt; ++i)
        fill_result(tracks[i], oa_host, ia_host, ms / (float)job.nt, job.track_err[i].empty() ? nullptr : job.track_err[i].c_str(), &job.out[job.idx[i]]);
    if (job.debug_single) debug_dump_wave(c, job);
    return STRATUM_OK;
}

static void debug_dump_wave(DeviceCtx& c, const WaveJob& job) {
    cudaStream_t s = c.stream;
    const DevCfg& dcfg = job.dcfg;
    const TrackDev& T = static_cast<const TrackDev*>(job.h_tracks.p)[0];
    if (T.status != 0) return;
    const int bs = dcfg.bs;
    const HopLayout& H = T.hop[bs];
    const uint32_t F = T.F[bs], L = F > 0 ? F - 1 : 0;
    const uint64_t fm = H.fmax;
    debug_put("gain", &c.d_tracks[0].gain, 1, s);
    debug_put("spec512_head", c.fa + H.spec, (size_t)std::min<uint32_t>(F, 64) * dcfg.bins, s);
    debug_put("onset.spectral_flux", c.fa + H.pair + 0 * fm, L, s);
    debug_put("frame.hfc", c.fa + H.frame + 2 * fm, F, s);
    debug_put("frame.energy", c.fa + H.frame + 1 * fm, F, s);
    debug_put("pair.superflux", c.fa + H.pair + 1 * fm, L, s);
    debug_put("pair.mel", c.fa + H.pair + 5 * fm, L, s);
    debug_put_i("onset.energy", c.ia + T.on_energy, T.n_on_energy, s);
    debug_put_i("onset.spectral", c.ia + T.on_spectral, T.n_on_spectral, s);
    debug_put_i("onset.hfc", c.ia + T.on_hfc, T.n_on_hfc, s);
    if (dcfg.hpss_onsets) debug_put_i("onset.hpss", c.ia + T.on_hpss, T.n_on_hpss, s);
    if (T.hpss_ready) {
        debug_put("hpss.perc_head", c.fa + T.hop[SLOT_PERC].spec, (size_t)std::min<uint32_t>(F, 64) * dcfg.bins, s);
        float pe[4] = {T.est[SLOT_PERC].bpm, T.est[SLOT_PERC].confidence, (float)T.est[SLOT_PERC].agreement, (float)T.est[SLOT_PERC].ok};
        std::lock_guard<std::mutex> lk(g_debug_mu);
        g_debug_arrays["perc.est"] = std::vector<float>(pe, pe + 4);
    }
    const char* vn[5] = {"base.nov.full", "base.nov.low", "base.nov.mid", "base.nov.high", "base.nov.mel"};
    for (int v = 0; v < 5; ++v) debug_put(vn[v], c.fa + H.nov + (uint64_t)v * fm, L, s);
    debug_put("base.tg.fft.full", c.fa + H.tgfft, H.fft_cap / 2 + 1, s);
    debug_put("base.tg.ac.full", c.fa + H.tgac, dcfg.n_bpm, s);
    if (T.n_on_final >= 2) debug_put("legacy.comb_raw", c.fa + T.lg_comb, dcfg.n_comb, s);  // hypothesis order; not computed with fewer onsets
    debug_put("base.cands", c.fa + T.cands[bs], (size_t)MAX_CANDS * 4, s);
    float est[12] = {T.est[bs].bpm, T.est[bs].confidence, (float)T.est[bs].agreement, (float)T.est[bs].ok, (float)T.est[bs].n_cands,
                     T.legacy.bpm, T.legacy.confidence, (float)T.legacy.ok, (float)T.escalate, T.est[1].bpm, T.est[2].bpm, 0.0f};
    {
        std::lock_guard<std::mutex> lk(g_debug_mu);
        g_debug_arrays["base.est"] = std::vector<float>(est, est + 12);
    }
    debug_put("key.hpcp_raw", c.fa + T.chroma, (size_t)T.Fk * 12, s);
    debug_put("key.hpcp_smooth", c.fa + T.chroma2, (size_t)T.Fk * 12, s);
    debug_put("key.energy", c.fa + T.kenergy, T.Fk, s);
    debug_put("key.weights", c.fa + T.kweights, T.Fk, s);
    debug_put("key.seg_scores", c.fa + T.seg_scores, (size_t)T.seg_cap * 24, s);
    if (dcfg.key_compact) debug_put("key.band_head", c.fa + T.kband, (size_t)std::min<uint32_t>(T.Fk, 64) * T.kband_stride, s);
    else debug_put("key.mask_head", c.fa + T.keyspec, (size_t)std::min<uint32_t>(T.Fk, 64) * dcfg.key_bins, s);
    debug_put_i("hmm.path", c.ia + T.hmm_path, T.hmm_T, s);
}

// Footprint (floats) of a track's base work areas.
static uint64_t track_floats(uint64_t n, uint32_t sr, const StratumConfig& cfg, const DevCfg& kd) {
    TrackDev T{};
    T.n = n;
    T.sr = sr ? sr : 1;
    Bump fa, oa, ia;
    plan_track(fa, oa, ia, T, cfg, kd);
    return align_up(fa.pos, 64) + 64;
}

// Wave packing (host logic, unit-tested through stratum_b200_debug_plan_waves): tracks are taken in order until the wave
// reaches its sample target or the arena budget.  The target balances the remaining samples over ceil(remaining / cap)
// waves, so a batch slightly larger than the cap does not end in a tiny (latency-bound) wave.
struct WaveLimits {
    uint64_t budget_floats;     // float arena budget; raised when a single track alone exceeds it
    uint32_t wave_max;          // track-count cap (<= 65535: a wave's tracks are gridDim.y of most launches)
    uint64_t wave_max_samples;  // sample cap (~0 = none)
};

constexpr uint32_t WAVE_MAX_TRACKS = 65535;
constexpr uint64_t WAVE_CAP_SAMPLES = (uint64_t)208 * 7938000;  // device-resident wave cap: 208 three-minute tracks (see Session::open)

static void pack_wave(uint32_t& i, uint32_t n_tracks, const uint64_t* lens, const uint32_t* srs, const StratumConfig& cfg, const DevCfg& kd, WaveLimits& L,
                      WavePlan& wp) {
    uint64_t used = 0, esc_max = 0, wave_samples = 0, remaining = 0;
    for (uint32_t q = i; q < n_tracks; ++q) remaining += lens[q];
    uint64_t wave_target = L.wave_max_samples;
    if (L.wave_max_samples != ~0ull && remaining > 0) {
        const uint64_t nw = (remaining + L.wave_max_samples - 1) / L.wave_max_samples;
        wave_target = (remaining + nw - 1) / nw;
    }
    while (i < n_tracks && wp.idx.size() < std::min(L.wave_max, WAVE_MAX_TRACKS)) {
        if (!wp.idx.empty() && wave_samples + lens[i] / 2 > wave_target) break;
        const uint64_t need = track_floats(lens[i], srs[i], cfg, kd);
        const uint64_t esc = esc_floats(lens[i], kd);
        const uint64_t esc_new = std::max(esc_max, esc);
        // keep room for escalating about a quarter of the wave at a time (at least one track)
        const uint64_t esc_room = esc_new * std::max<uint64_t>(1, (wp.idx.size() + 4) / 4);
        if (!wp.idx.empty() && used + need + esc_room > L.budget_floats) break;
        wave_samples += lens[i];
        used += need;
        esc_max = esc_new;
        wp.idx.push_back(i);
        ++i;
    }
    if (used + esc_max > L.budget_floats && wp.idx.size() == 1) L.budget_floats = used + esc_max;  // a single track larger than the budget: let cudaMalloc decide
}

// One batch call on one device: waves are queued one ahead of the gather (wave k+1 is planned and its first half queued while
// wave k runs; the host blocks only for the escalated-track count of the wave it is queueing and for finished results).
// The caller holds ctx.mu for the whole session.
struct Session {
    DeviceCtx& c;
    const StratumConfig& cfg;
    DevCfg dcfg;
    WaveLimits lim{};
    int cur = 0;  // job slot of the next wave
    double waves_ms = 0.0;
    uint32_t n_waves = 0;
    cudaEvent_t call_a = nullptr, call_b = nullptr;
    bool opened = false;

    Session(DeviceCtx& ctx, const StratumConfig& cf) : c(ctx), cfg(cf), dcfg(make_devcfg(cf)) {}
    ~Session() {
        if (call_a) cudaEventDestroy(call_a);
        if (call_b) cudaEventDestroy(call_b);
    }

    int open() {
        CUDA_OK(cudaSetDevice(c.device));
        // per-sample-rate tables are built for one configuration; a call with another one starts a fresh set when the
        // table is getting full (slots are only referenced by the waves of one session, and none is in flight here)
        if (!c.sr_cfg.empty() && c.sr_host.size() > DeviceCtx::MAX_SR / 2 && memcmp(&c.sr_cfg.back(), &cfg, sizeof cfg) != 0) {
            c.sr_host.clear();
            c.sr_cfg.clear();
        }
        size_t free_b = 0, total_b = 0;
        CUDA_OK(cudaMemGetInfo(&free_b, &total_b));
        // budget: what is free now plus what our own arena already holds, minus head room
        uint64_t budget_floats = (uint64_t)((double)(free_b + c.fa_cap * 4) * 0.90) / 4;
        // waves of a few hundred tracks already fill the GPU; a larger arena buys nothing and starves the caller (and our
        // own staging buffers) of memory, so the default is capped at 100 GB
        double cap_gb = 100.0;
        if (const char* e = getenv("STRATUM_B200_ARENA_GB")) cap_gb = atof(e);
        budget_floats = std::min<uint64_t>(budget_floats, (uint64_t)(cap_gb * 1e9 / 4));
        // wave size (three-minute tracks), device-resident batch of 1024, round 2 kernels (r02p): 103 -> 1322 tracks/s, 128 -> 1338, 171 -> 1355,
        // 205 -> 1355, 256 -> 1358; round 1 had 128-160 fastest.  The cap is expressed in samples so that batches of short tracks still
        // fill the device; 208 cuts the 1024-track batch into five even waves.  (Host batches are cut by the upload chunks instead: 128.)
        uint32_t wave_max = WAVE_MAX_TRACKS;
        uint64_t wave_max_samples = WAVE_CAP_SAMPLES;
        if (const char* e = getenv("STRATUM_B200_WAVE_MAX_TRACKS")) {
            wave_max = (uint32_t)std::min<long>(std::max(1, atoi(e)), (long)WAVE_MAX_TRACKS);
            wave_max_samples = ~0ull;
        }
        lim = WaveLimits{budget_floats, wave_max, wave_max_samples};
        if (dcfg.n_bpm > (uint32_t)AC_CAP || dcfg.n_comb > (uint32_t)AC_CAP) {  // fine BPM grid: its kernels read the hypotheses from a table
            dcfg.bpm_tab = get_bpm_tab(c, dcfg);
            if (!dcfg.bpm_tab) {
                set_error("BPM grid table allocation failed");
                return STRATUM_PROCESSING_ERROR;
            }
        }
        CUDA_OK(cudaEventCreate(&call_a));
        CUDA_OK(cudaEventCreate(&call_b));
        cudaEventRecord(call_a, c.stream);
        opened = true;
        return STRATUM_OK;
    }

    // Queues the waves of one device-resident group of tracks (track q = d_samples[offs[q] .. offs[q] + lens[q])).  On return the
    // group's last wave may still be running; every earlier wave of the session has been gathered.  `after_prev` runs once, as soon
    // as the waves that were in flight at entry are gathered (their sample buffer is free from then on).
    int submit(const float* d_samples, const uint64_t* offs, const uint64_t* lens, const uint32_t* srs, uint32_t n, StratumResult* out,
               const std::function<void()>& after_prev) {
        uint32_t i = 0;
        bool fired = false;
        int st = STRATUM_OK;
        while (i < n && st == STRATUM_OK) {
            WavePlan wp;
            {
                HostSpan span_pack("host_wave_pack");
                pack_wave(i, n, lens, srs, cfg, dcfg, lim, wp);
            }
            WaveJob& job = c.jobs[cur];
            WaveJob& prev = c.jobs[cur ^ 1];
            auto mid = [&]() -> int {
                const int s2 = wave_end(c, prev, &waves_ms);
                if (!fired) {
                    fired = true;
                    if (after_prev) after_prev();
                }
                return s2;
            };
            st = wave_begin(c, d_samples, offs, lens, srs, wp, cfg, dcfg, lim.budget_floats, out, job, mid);
            if (st != STRATUM_OK) {
                std::string keep = g_last_error;
                wave_end(c, prev, nullptr);  // a wave_begin that failed before its mid point leaves the previous wave queued
                wave_end(c, job, nullptr);
                set_error(keep);
                break;
            }
            ++n_waves;
            cur ^= 1;
            if (job.debug_single) st = wave_end(c, job, &waves_ms);  // the debug dumps read the arena: no wave may follow before them
        }
        if (!fired && st == STRATUM_OK) {
            st = wave_end(c, c.jobs[cur ^ 1], &waves_ms);
            if (after_prev) after_prev();
        }
        return st;
    }

    int drain() {
        const int s1 = wave_end(c, c.jobs[cur], &waves_ms);
        const int s2 = wave_end(c, c.jobs[cur ^ 1], &waves_ms);
        return s1 != STRATUM_OK ? s1 : s2;
    }

    void close() {  // device time of the whole call, inter-wave gaps included
        if (!opened) return;
        cudaEventRecord(call_b, c.stream);
        cudaEventSynchronize(call_b);
        float whole_ms = 0.0f;
        double call_ms = waves_ms;
        if (cudaEventElapsedTime(&whole_ms, call_a, call_b) == cudaSuccess) call_ms = whole_ms;
        g_last_call_us.store((uint64_t)(call_ms * 1000.0));
        g_last_call_waves.store(n_waves);
    }
};

static int analyze_device(DeviceCtx* ctx, const float* d_samples, const uint64_t* offsets, const uint32_t* srs, uint32_t n_tracks, const StratumConfig& cfg,
                          StratumResult* out) {
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    Session S(*ctx, cfg);
    int st = S.open();
    if (st != STRATUM_OK) return st;
    std::vector<uint64_t> lens(n_tracks), offs(n_tracks);
    for (uint32_t i = 0; i < n_tracks; ++i) {
        offs[i] = offsets[i];
        lens[i] = offsets[i + 1] - offsets[i];
    }
    st = S.submit(d_samples, offs.data(), lens.data(), srs, n_tracks, out, nullptr);
    const int st2 = S.drain();
    S.close();
    return st != STRATUM_OK ? st : st2;
}

}  // namespace sb

// =================================================== C ABI ===================================================
using namespace sb;

extern "C" {

void stratum_b200_config_default(StratumConfig* cfg) {
    if (cfg) config_default(cfg);
}

int32_t stratum_b200_analyze_batch_device(const float* d_samples, const uint64_t* offsets, const uint32_t* sample_rates, uint32_t n_tracks,
                                          const StratumConfig* cfg, int32_t device_id, StratumResult* out) {
    if (!offsets || !sample_rates || !out || (!d_samples && n_tracks && offsets[n_tracks] > 0)) {
        set_error("null argument");
        return STRATUM_INVALID_INPUT;
    }
    StratumConfig def;
    config_default(&def);
    const StratumConfig& c = cfg ? *cfg : def;
    int st = config_validate(c);
    if (st != STRATUM_OK) return st;
    if (n_tracks == 0) return STRATUM_OK;
    DeviceCtx* ctx = get_ctx(device_id, &st);
    if (!ctx) return st;
    return analyze_device(ctx, d_samples, offsets, sample_rates, n_tracks, c, out);
}

// Host-buffer batches (f32 samples, or interleaved PCM16 converted on the device): contiguous shards, one host
// thread per device (examples/analyze_batch.rs:239-326: the only parallelism of the reference is across tracks; the
// gather is the result array itself).  Each shard is streamed through two device staging buffers: chunk k+1 is
// uploaded by the device's uploader thread while chunk k is analysed (pinned host memory makes the upload asynchronous;
// pageable memory still works, without the overlap), and the analysis itself runs one wave ahead of the gather (Session).
static uint32_t pcm_bytes_per_sample(uint32_t fmt) {
    switch (fmt) {
        case STRATUM_PCM_U8: return 1;
        case STRATUM_PCM_S16: return 2;
        case STRATUM_PCM_S24: return 3;
        case STRATUM_PCM_S32: return 4;
        case STRATUM_PCM_F32: return 4;
        case STRATUM_PCM_F64: return 8;
        default: return 0;
    }
}

// Bytes per frame of every PCM track into bpf; rejects the whole call on an unknown format, a channel count outside 1..64 or a
// partial frame.
static int pcm_frame_bytes(const uint64_t* boff, const uint32_t* channels, const uint32_t* formats, uint32_t n_tracks, std::vector<uint32_t>& bpf) {
    for (uint32_t i = 0; i < n_tracks; ++i) {
        const uint32_t bps = pcm_bytes_per_sample(formats[i]);
        if (bps == 0) {
            set_error("unknown PCM sample format (STRATUM_PCM_*)");
            return STRATUM_INVALID_INPUT;
        }
        if (channels[i] == 0 || channels[i] > 64 || (boff[i + 1] - boff[i]) % ((uint64_t)bps * channels[i]) != 0) {
            set_error("PCM track length is not a whole number of frames (or channels outside 1..64)");
            return STRATUM_INVALID_INPUT;
        }
        bpf[i] = bps * channels[i];
    }
    return STRATUM_OK;
}

// Chunk of a shard: tracks [i, j), `elems` bytes of host data, `frames` sample frames.
struct HostChunk {
    uint32_t i, j;
    uint64_t elems, frames;
};

// The device work of one shard of a host batch, fed chunk by chunk by stream_host_batch.  Every method returns a StratumStatus and
// leaves its message in g_last_error.
struct ChunkSink {
    virtual ~ChunkSink() = default;
    virtual int open(const std::vector<HostChunk>& chunks) = 0;  // before the first upload; chunks are those of the shard
    // Chunk k is staged at d_buf (byte 0 = the first byte of track ch.i).  after_prev must be called once, as soon as the device no
    // longer reads the previous chunk's staging buffer: it starts the upload of chunk k + 1 into that buffer.
    virtual int chunk(size_t k, const HostChunk& ch, const char* d_buf, const std::function<void()>& after_prev) = 0;
    virtual int close() = 0;  // after the last chunk, and after a failure
};

// boff: byte offsets of the tracks inside src (n_tracks + 1); bpf: bytes per sample frame of every track.  The tracks are cut into
// contiguous shards, one per device context (an id named twice, or -1 next to the current device's id, is one shard, not two), each
// streamed by its own host thread through the context's staging buffers into the sink make_sink(ctx) returns.
static int32_t stream_host_batch(const void* src, const uint64_t* boff, const std::vector<uint32_t>& bpf, uint32_t n_tracks, const int32_t* device_ids,
                                 uint32_t n_devices, const std::function<std::unique_ptr<ChunkSink>(DeviceCtx*)>& make_sink) {
    int st = STRATUM_OK;
    const uint64_t* offsets = boff;
    const size_t elt = 1;  // offsets are in bytes
    std::vector<DeviceCtx*> ctxs;
    {
        std::vector<int32_t> devs;
        if (device_ids && n_devices) devs.assign(device_ids, device_ids + n_devices);
        else devs.push_back(-1);
        for (int32_t d : devs) {
            DeviceCtx* ctx = get_ctx(d, &st);
            if (!ctx) return st;
            if (std::find(ctxs.begin(), ctxs.end(), ctx) == ctxs.end()) ctxs.push_back(ctx);
        }
    }
    const uint32_t nd = (uint32_t)ctxs.size();
    std::vector<int> status(nd, STRATUM_OK);
    std::vector<std::string> errs(nd);
    auto work = [&](uint32_t d) {
        const uint32_t a = (uint32_t)((uint64_t)n_tracks * d / nd), b = (uint32_t)((uint64_t)n_tracks * (d + 1) / nd);
        if (a == b) return;
        DeviceCtx* ctx = ctxs[d];
        auto fail = [&](int code, const std::string& msg) {
            if (status[d] == STRATUM_OK) {
                status[d] = code;
                errs[d] = msg;
            }
        };
        // One call at a time per device: the staging buffers, the conversion buffer, the arenas and the streams belong to the
        // context, so the whole shard (upload, conversion, analysis) runs under its lock; concurrent callers queue up here.
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (cudaSetDevice(ctx->device) != cudaSuccess) return fail(STRATUM_PROCESSING_ERROR, "cudaSetDevice failed");
        // Chunk sizes ramp up: a small first chunk keeps the un-overlapped first upload short, later chunks grow to
        // STRATUM_B200_STAGE_MB of mono f32 (default 3876 MB = 128 three-minute tracks: its 74 ms upload at 55 GB/s still hides behind the
        // ~85 ms the chunk's wave takes, and larger chunks lengthen the ramp; device-resident batches use waves of up to 208); at least
        // one track per chunk
        uint64_t chunk_frames = (uint64_t)128 * 7938000;  // = the wave cap of a session: one full-size chunk is one wave
        if (const char* e = getenv("STRATUM_B200_STAGE_MB")) chunk_frames = std::max<uint64_t>((uint64_t)(atof(e) * 1024 * 1024 / 4), 1u << 16);
        static const bool no_ramp = getenv("STRATUM_B200_STAGE_NO_RAMP") != nullptr;
        auto frames_of_track = [&](uint32_t q) { return (offsets[q + 1] - offsets[q]) / bpf[q]; };
        std::vector<HostChunk> chunks;
        uint64_t max_el = 0;
        // ramp: "a,b" = first chunk a/8 of a full chunk, growth by b/8 of a full chunk per step (default 2,2: 1/4, 1/2, 3/4, 1 ...)
        static const char* ramp_env = getenv("STRATUM_B200_STAGE_RAMP");
        int ramp_first = 2, ramp_step = 2;
        if (ramp_env) sscanf(ramp_env, "%d,%d", &ramp_first, &ramp_step);
        ramp_first = std::min(std::max(ramp_first, 1), 8);
        ramp_step = std::min(std::max(ramp_step, 1), 8);
        uint64_t cur_frames = no_ramp ? chunk_frames : std::max<uint64_t>(chunk_frames * ramp_first / 8, 1u << 16);
        for (uint32_t i = a; i < b;) {
            uint32_t j = i;
            uint64_t fr = 0;
            while (j < b && j - i < WAVE_MAX_TRACKS && (j == i || fr + frames_of_track(j) <= cur_frames)) {
                fr += frames_of_track(j);
                ++j;
            }
            const uint64_t el = offsets[j] - offsets[i];
            chunks.push_back(HostChunk{i, j, el, fr});
            max_el = std::max(max_el, el);
            i = j;
            cur_frames = std::min<uint64_t>(chunk_frames, cur_frames + chunk_frames * ramp_step / 8);
        }
        const size_t buf_bytes = (size_t)align_up(max_el * elt + 64, 256);
        {
            if (!ctx->copy_stream && cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess)
                return fail(STRATUM_PROCESSING_ERROR, "copy stream creation failed");
            if (!grow_device(ctx->d_stage, ctx->stage_cap, 2 * buf_bytes)) return fail(STRATUM_PROCESSING_ERROR, "staging buffer allocation failed");
        }
        char* bufs[2] = {reinterpret_cast<char*>(ctx->d_stage), reinterpret_cast<char*>(ctx->d_stage) + buf_bytes};
        if (!ctx->uploader) ctx->uploader.reset(new Worker());
        // Uploads run on the device's uploader thread, in pieces of 128 MB with a stream synchronisation after each piece: the
        // analysis of chunk k issues small host<->device copies of its own (track records, counts, results) that would otherwise
        // queue behind a multi-gigabyte transfer on the copy engine and stall the wave until the next chunk has landed (measured:
        // no overlap at all with 2 GB transfers enqueued in one piece).
        auto upload = [&, ctx](size_t k) -> bool {
            const HostChunk& ch = chunks[k];
            if (cudaSetDevice(ctx->device) != cudaSuccess) return false;
            g_h2d_bytes.fetch_add(ch.elems * elt);
            const char* hsrc = static_cast<const char*>(src) + offsets[ch.i] * elt;
            const size_t total = ch.elems * elt, piece = (size_t)128 << 20;
            for (size_t o = 0; o < total; o += piece) {
                if (cudaMemcpyAsync(bufs[k & 1] + o, hsrc + o, std::min(piece, total - o), cudaMemcpyHostToDevice, ctx->copy_stream) != cudaSuccess) return false;
                if (cudaStreamSynchronize(ctx->copy_stream) != cudaSuccess) return false;
            }
            return true;
        };
        std::unique_ptr<ChunkSink> sink = make_sink(ctx);
        int s2 = sink->open(chunks);
        if (s2 != STRATUM_OK) return fail(s2, g_last_error);
        std::future<bool> up = ctx->uploader->post([&] { return upload(0); });
        bool ok = true;
        for (size_t k = 0; ok && k < chunks.size(); ++k) {
            {
                HostSpan span_up(k == 0 ? "host_first_upload" : "host_chunk_wait_upload");  // > 0 later on only when an upload outlasts the analysis beside it
                ok = up.get();
            }
            if (!ok) {
                fail(STRATUM_PROCESSING_ERROR, "host to device copy failed");
                break;
            }
            bool posted = false;
            auto after_prev = [&] {  // the previous chunk's work is done: its staging buffer takes chunk k+1
                if (k + 1 < chunks.size()) {
                    up = ctx->uploader->post([&, k] { return upload(k + 1); });
                    posted = true;
                }
            };
            {
                HostSpan span_an("host_chunk_submit");  // wall time of queueing the chunk (includes gathering the previous one)
                s2 = sink->chunk(k, chunks[k], bufs[k & 1], after_prev);
            }
            if (s2 != STRATUM_OK) {
                fail(s2, g_last_error);
                ok = false;
                if (posted) up.get();  // the upload lambda refers to this frame
                break;
            }
        }
        s2 = sink->close();
        if (s2 != STRATUM_OK) fail(s2, g_last_error);
        cudaStreamSynchronize(ctx->copy_stream);
    };
    if (nd == 1) {
        work(0);
    } else {
        std::vector<std::thread> th;
        for (uint32_t d = 0; d < nd; ++d) th.emplace_back(work, d);
        for (auto& t : th) t.join();
    }
    for (uint32_t d = 0; d < nd; ++d)
        if (status[d] != STRATUM_OK) {
            set_error(errs[d]);
            return status[d];
        }
    return STRATUM_OK;
}

// The analysis of the staged chunks: mono f32 samples straight from the staging buffer, or interleaved PCM (formats != nullptr)
// converted and mixed down on the device into the conversion buffer first.  The waves run one ahead of the gather (Session).
struct AnalysisSink final : ChunkSink {
    DeviceCtx* ctx;
    Session S;
    const uint64_t* offsets;
    const std::vector<uint32_t>& bpf;
    const uint32_t *sample_rates, *channels, *formats;
    StratumResult* out;
    size_t meta_each = 0;
    AnalysisSink(DeviceCtx* c, const StratumConfig& cfg, const uint64_t* offs, const std::vector<uint32_t>& bpf_, const uint32_t* srs, const uint32_t* chans,
                 const uint32_t* fmts, StratumResult* o)
        : ctx(c), S(*c, cfg), offsets(offs), bpf(bpf_), sample_rates(srs), channels(chans), formats(fmts), out(o) {}
    uint64_t frames_of_track(uint32_t q) const { return (offsets[q + 1] - offsets[q]) / bpf[q]; }

    int open(const std::vector<HostChunk>& chunks) override {
        if (formats) {
            uint64_t max_fr = 0;
            uint32_t max_cn = 0;
            for (const HostChunk& ch : chunks) {
                max_fr = std::max(max_fr, ch.frames);
                max_cn = std::max(max_cn, ch.j - ch.i);
            }
            // per-chunk offset / channel tables of the PCM path, two sets (the conversion of chunk k+1 is queued while chunk k runs)
            meta_each = (size_t)align_up((size_t)(max_cn + 1) * 16 + (size_t)max_cn * 8 + 64, 256);
            if (!grow_device(ctx->d_conv, ctx->conv_cap, (max_fr + 16) * sizeof(float)) || !grow_device(ctx->d_meta, ctx->meta_cap, 2 * meta_each)) {
                set_error("staging buffer allocation failed");
                return STRATUM_PROCESSING_ERROR;
            }
        }
        return S.open();
    }

    int chunk(size_t k, const HostChunk& ch, const char* d_buf, const std::function<void()>& after_prev) override {
        const uint32_t cn = ch.j - ch.i;
        std::vector<uint64_t> rel(cn + 1, 0), lens(cn);  // per-track offsets in mono frames inside the chunk
        for (uint32_t q = 0; q < cn; ++q) {
            lens[q] = frames_of_track(ch.i + q);
            rel[q + 1] = rel[q] + lens[q];
        }
        const float* d_mono = reinterpret_cast<const float*>(d_buf);
        if (formats) {
            // decoder arithmetic on the device: interleaved PCM -> mono f32 (examples/analyze_batch.rs:70-165).  Queued on
            // the analysis stream, so it runs after the previous chunk's waves have finished with the conversion buffer.
            char* hm = static_cast<char*>(ctx->h_meta[k & 1].need(meta_each));
            if (!hm) {
                set_error("pinned host allocation failed");
                return STRATUM_PROCESSING_ERROR;
            }
            uint64_t* h_poff = reinterpret_cast<uint64_t*>(hm);
            uint64_t* h_ooff = h_poff + (cn + 1);
            uint32_t* h_ch = reinterpret_cast<uint32_t*>(h_ooff + (cn + 1));
            uint32_t* h_fmt = h_ch + cn;
            uint64_t max_frames = 0;
            for (uint32_t q = 0; q <= cn; ++q) {
                h_poff[q] = offsets[ch.i + q] - offsets[ch.i];
                h_ooff[q] = rel[q];
            }
            for (uint32_t q = 0; q < cn; ++q) {
                h_ch[q] = channels[ch.i + q];
                h_fmt[q] = formats[ch.i + q];
                max_frames = std::max(max_frames, lens[q]);
            }
            char* dm = ctx->d_meta + (k & 1) * meta_each;
            uint64_t* d_poff = reinterpret_cast<uint64_t*>(dm);
            uint64_t* d_ooff = d_poff + (cn + 1);
            uint32_t* d_ch = reinterpret_cast<uint32_t*>(d_ooff + (cn + 1));
            uint32_t* d_fmt = d_ch + cn;
            cudaMemcpyAsync(dm, hm, (size_t)(cn + 1) * 16 + (size_t)cn * 8, cudaMemcpyHostToDevice, ctx->stream);
            launch_pcm_to_mono(ctx->stream, d_buf, ctx->d_conv, d_poff, d_ooff, d_ch, d_fmt, cn, max_frames);
            d_mono = ctx->d_conv;
        }
        return S.submit(d_mono, rel.data(), lens.data(), sample_rates + ch.i, cn, out + ch.i, after_prev);
    }

    int close() override {
        const int st = S.drain();
        S.close();
        return st;
    }
};

// boff: byte offsets of the tracks inside src (n_tracks + 1).  formats == nullptr: mono f32 samples analysed straight from the staging
// buffer; otherwise interleaved PCM in the given per-track format and channel count, converted and mixed down on the device.
static int32_t analyze_host_batch(const void* src, const uint64_t* boff, const uint32_t* sample_rates, const uint32_t* channels, const uint32_t* formats,
                                  uint32_t n_tracks, const StratumConfig* cfg, const int32_t* device_ids, uint32_t n_devices, StratumResult* out) {
    const bool pcm = formats != nullptr;
    if (!boff || !sample_rates || !out || (!src && n_tracks && boff[n_tracks] > 0) || (pcm && !channels)) {
        set_error("null argument");
        return STRATUM_INVALID_INPUT;
    }
    StratumConfig def;
    config_default(&def);
    const StratumConfig& c = cfg ? *cfg : def;
    int st = config_validate(c);
    if (st != STRATUM_OK) return st;
    if (n_tracks == 0) return STRATUM_OK;
    std::vector<uint32_t> bpf(n_tracks, 4);  // bytes per mono frame
    if (pcm && (st = pcm_frame_bytes(boff, channels, formats, n_tracks, bpf)) != STRATUM_OK) return st;
    return stream_host_batch(src, boff, bpf, n_tracks, device_ids, n_devices, [&](DeviceCtx* ctx) -> std::unique_ptr<ChunkSink> {
        return std::unique_ptr<ChunkSink>(new AnalysisSink(ctx, c, boff, bpf, sample_rates, channels, formats, out));
    });
}

// ---- loudness (BS.1770-4 / EBU R128; include/stratum_b200.h: StratumLoudness) --------------------------------------------------------
// K-weighting coefficients at sample rate sr from the analog prototype (libebur128's derivation), in double:
// k = stage 1 b0 b1 b2 a1 a2, stage 2 b0 b1 b2 a1 a2.
static void kweight_coeffs(uint32_t sr, double* k) {
    const double fs = (double)sr;
    {
        const double f0 = 1681.974450955533, G = 3.999843853973347, Q = 0.7071752369554196;
        const double K = tan(M_PI * f0 / fs), Vh = pow(10.0, G / 20.0), Vb = pow(Vh, 0.4996667741545416);
        const double a0 = 1.0 + K / Q + K * K;
        k[0] = (Vh + Vb * K / Q + K * K) / a0;
        k[1] = 2.0 * (K * K - Vh) / a0;
        k[2] = (Vh - Vb * K / Q + K * K) / a0;
        k[3] = 2.0 * (K * K - 1.0) / a0;
        k[4] = (1.0 - K / Q + K * K) / a0;
    }
    {
        const double f0 = 38.13547087602444, Q = 0.5003270373238773;
        const double K = tan(M_PI * f0 / fs), d = 1.0 + K / Q + K * K;
        k[5] = 1.0;
        k[6] = -2.0;
        k[7] = 1.0;
        k[8] = 2.0 * (K * K - 1.0) / d;
        k[9] = (1.0 - K / Q + K * K) / d;
    }
}

static uint32_t true_peak_factor(uint32_t sr) { return sr < 96000 ? 4 : (sr < 192000 ? 2 : 1); }

// c[j] = sinc((j - 24) / L) * Hann(j / 48); the phase-0 taps are exactly 1 (j = 24) and 0, so the filter interpolates.
static void true_peak_taps(uint32_t L, float* c) {
    for (int j = 0; j <= 48; ++j) {
        const int d = j - 24;
        double v;
        if (d % (int)L == 0) v = d == 0 ? 1.0 : 0.0;
        else {
            const double t = M_PI * (double)d / (double)L;
            v = sin(t) / t * 0.5 * (1.0 - cos(2.0 * M_PI * (double)j / 48.0));
        }
        c[j] = (float)v;
    }
}

// M = A^S: A is the zero-input map of one sample on the state (z1, z2 of stage 1, z1, z2 of stage 2) of k_loudness.cu's cascade.
static void kweight_power(const double* k, uint32_t S, double* M) {
    double A[16], R[16], T[16];
    for (int j = 0; j < 4; ++j) {
        double s[4] = {0.0, 0.0, 0.0, 0.0};
        s[j] = 1.0;
        const double y1 = s[0];
        const double z1a = -k[3] * y1 + s[1], z2a = -k[4] * y1;
        const double y2 = k[5] * y1 + s[2];
        const double z1b = k[6] * y1 - k[8] * y2 + s[3], z2b = k[7] * y1 - k[9] * y2;
        const double col[4] = {z1a, z2a, z1b, z2b};
        for (int i = 0; i < 4; ++i) A[4 * i + j] = col[i];
    }
    auto mul = [&](const double* X, const double* Y, double* out) {
        for (int i = 0; i < 4; ++i)
            for (int j = 0; j < 4; ++j) {
                double acc = 0.0;
                for (int q = 0; q < 4; ++q) acc += X[4 * i + q] * Y[4 * q + j];
                T[4 * i + j] = acc;
            }
        memcpy(out, T, sizeof T);
    };
    for (int i = 0; i < 16; ++i) R[i] = (i % 5 == 0) ? 1.0 : 0.0;
    for (uint32_t e = S; e; e >>= 1) {
        if (e & 1) mul(A, R, R);
        mul(A, A, A);
    }
    memcpy(M, R, sizeof R);
}

// Per-track failure of the loudness measurement (0 = measured).
static int loud_track_status(uint32_t sr, uint64_t frames, char* msg, size_t cap) {
    if (frames == 0 || sr == 0) {
        snprintf(msg, cap, "%s", frames == 0 ? "empty track: no sample frames" : "sample rate 0");
        return STRATUM_INVALID_INPUT;
    }
    if (sr < 8000 || sr > 384000) {
        snprintf(msg, cap, "sample rate %u Hz is outside the 8000..384000 Hz range of the loudness measurement", sr);
        return STRATUM_NOT_IMPLEMENTED;
    }
    return STRATUM_OK;
}

// Sub-block frames S, segments covering the track, whole sub-blocks, momentary blocks J and short-term windows K of one track
// (all counts 0 for a track that fails).
struct LoudGeom {
    bool ok;
    uint32_t S, nseg, nfull, J, K;
};
static LoudGeom loud_geom(uint32_t sr, uint64_t frames) {
    char msg[128];
    LoudGeom g;
    g.ok = loud_track_status(sr, frames, msg, sizeof msg) == STRATUM_OK;
    g.S = g.ok ? (sr + 5) / 10 : 1;
    g.nseg = g.ok ? (uint32_t)((frames + g.S - 1) / g.S) : 0;
    g.nfull = g.ok ? (uint32_t)(frames / g.S) : 0;
    g.J = g.nfull > 3 ? g.nfull - 3 : 0;
    g.K = g.nfull > 29 ? g.nfull - 29 : 0;
    return g;
}

// The host pools of the albums of one call: one buffer holding the album records, then every album's momentary powers, then every
// album's short-term powers; albums one after the other, members in ascending track index.  Member q's powers go to
// buf[m_at[q] ..) and buf[q_at[q] ..); the shards of a host batch fill disjoint ranges.
struct AlbumPools {
    const uint32_t* album_of = nullptr;
    uint32_t n_albums = 0;
    std::vector<uint64_t> m_at, q_at;
    uint64_t mom0 = 0, sht0 = 0, n_mom = 0, n_sht = 0;  // buf offsets of the two pools and their lengths, in doubles
    std::vector<double> buf;
    LoudAlbum* albums() { return reinterpret_cast<LoudAlbum*>(buf.data()); }
    bool member(uint32_t q) const { return album_of && album_of[q] < n_albums; }
};

static void album_layout(const uint32_t* album_of, uint32_t n_albums, const uint64_t* offsets, const std::vector<uint32_t>& bpf,
                         const uint32_t* sample_rates, uint32_t n_tracks, AlbumPools& P) {
    P.album_of = album_of;
    P.n_albums = n_albums;
    if (n_albums == 0) return;
    std::vector<LoudAlbum> al(n_albums, LoudAlbum{0, 0, 0, 0});
    std::vector<LoudGeom> g(n_tracks);
    for (uint32_t q = 0; q < n_tracks; ++q) {
        if (!P.member(q)) continue;
        g[q] = loud_geom(sample_rates[q], (offsets[q + 1] - offsets[q]) / bpf[q]);
        al[album_of[q]].J += g[q].J;
        al[album_of[q]].K += g[q].K;
    }
    for (LoudAlbum& a : al) {
        a.m0 = P.n_mom;
        a.q0 = P.n_sht;
        P.n_mom += a.J;
        P.n_sht += a.K;
    }
    P.mom0 = (n_albums * sizeof(LoudAlbum) + sizeof(double) - 1) / sizeof(double);
    P.sht0 = P.mom0 + P.n_mom;
    P.buf.assign(P.sht0 + P.n_sht, 0.0);
    memcpy(P.buf.data(), al.data(), n_albums * sizeof(LoudAlbum));
    P.m_at.assign(n_tracks, 0);
    P.q_at.assign(n_tracks, 0);
    std::vector<uint64_t> mf(n_albums), qf(n_albums);
    for (uint32_t a = 0; a < n_albums; ++a) {
        mf[a] = P.mom0 + al[a].m0;
        qf[a] = P.sht0 + al[a].q0;
    }
    for (uint32_t q = 0; q < n_tracks; ++q) {
        if (!P.member(q)) continue;
        P.m_at[q] = mf[album_of[q]];
        P.q_at[q] = qf[album_of[q]];
        mf[album_of[q]] += g[q].J;
        qf[album_of[q]] += g[q].K;
    }
}

// The channel side of a loudness call: the caller's channel map (null: the default map of every track) and the per-channel results
// (null: none).  Track q's entries of both start at at[q], the channels of the tracks before it.
struct LoudChannels {
    const uint8_t* map = nullptr;
    StratumLoudness* out = nullptr;
    std::vector<uint64_t> at;
};

// The series side of a loudness call (include/stratum_b200.h: stratum_b200_loudness_series_pcm): the caller's arrays in the order of
// LoudSeries (null: that series is neither produced nor read back), and per series where track q's entries start, at[s][q]: the
// lengths of the tracks before it.
struct LoudSeriesOut {
    double* dst[4] = {nullptr, nullptr, nullptr, nullptr};  // momentary, short-term, sample-peak, true-peak
    std::vector<uint64_t> at[4];
    uint32_t count() const { return (dst[0] != nullptr) + (dst[1] != nullptr) + (dst[2] != nullptr) + (dst[3] != nullptr); }
    bool peaks() const { return dst[2] || dst[3]; }
    static uint32_t length(const LoudGeom& g, int k) { return k == 0 ? g.J : (k == 1 ? g.K : g.nseg); }
};

static void series_layout(double* mom, double* sht, double* spk, double* tpk, const uint64_t* offsets, const std::vector<uint32_t>& bpf,
                          const uint32_t* sample_rates, uint32_t n_tracks, LoudSeriesOut& so) {
    double* d[4] = {mom, sht, spk, tpk};
    for (int k = 0; k < 4; ++k) {
        so.dst[k] = d[k];
        so.at[k].assign(d[k] ? n_tracks : 0, 0);
    }
    if (!so.count()) return;
    uint64_t next[4] = {0, 0, 0, 0};
    for (uint32_t q = 0; q < n_tracks; ++q) {
        const LoudGeom g = loud_geom(sample_rates[q], (offsets[q + 1] - offsets[q]) / bpf[q]);
        for (int k = 0; k < 4; ++k)
            if (d[k]) {
                so.at[k][q] = next[k];
                next[k] += LoudSeriesOut::length(g, k);
            }
    }
}

// Weight of a channel class (include/stratum_b200.h: StratumChannelClass); codes are checked by channels_validate.
static double loud_class_weight(uint8_t code) {
    switch (code) {
        case STRATUM_CH_FRONT: return 1.0;
        case STRATUM_CH_SURROUND: return 1.41;
        case STRATUM_CH_DUAL_MONO: return 2.0;
        default: return 0.0;
    }
}

// The loudness of the staged chunks: one launch of each kernel per chunk over all its tracks, straight from the staged PCM.  Chunk
// k's results are read back while chunk k+1 runs.
struct LoudnessSink final : ChunkSink {
    DeviceCtx* ctx;
    const uint64_t* offsets;
    const std::vector<uint32_t>& bpf;
    const uint32_t *sample_rates, *channels, *formats;
    StratumLoudness* out;
    AlbumPools* pools;  // null without albums
    const LoudChannels& chans_;  // channel map, per-channel results
    const LoudSeriesOut& ser_;  // requested series
    cudaStream_t stream;  // every launch and copy of the sink; ctx->stream unless set before open()
    struct Slot {
        uint32_t i = 0, j = 0;
        bool queued = false, blocks = false;  // blocks: the chunk's momentary / short-term powers were read back
        uint64_t n_seg = 0;
        std::vector<PendingStage> stages;
    } slot[2];
    LoudnessSink(DeviceCtx* c, const uint64_t* offs, const std::vector<uint32_t>& bpf_, const uint32_t* srs, const uint32_t* chans, const uint32_t* fmts,
                 StratumLoudness* o, AlbumPools* p, const LoudChannels& lc, const LoudSeriesOut& so)
        : ctx(c), offsets(offs), bpf(bpf_), sample_rates(srs), channels(chans), formats(fmts), out(o), pools(p), chans_(lc), ser_(so), stream(c->stream) {}
    bool has_member(uint32_t i, uint32_t j) const {
        for (uint32_t q = i; pools && q < j; ++q)
            if (pools->member(q)) return true;
        return false;
    }

    // Records of tracks [i, j) (byte offsets relative to track i) into rec and their channel weights into wt (both may be null);
    // returns the work items, segments and channels.
    void plan(uint32_t i, uint32_t j, LoudTrack* rec, double* wt, uint64_t* n_work, uint64_t* n_seg, uint64_t* n_ch, uint32_t* max_c) const {
        uint64_t w = 0, sg = 0, nc = 0;
        uint32_t mc = 1;
        for (uint32_t q = i; q < j; ++q) {
            const uint32_t sr = sample_rates[q], C = channels[q];
            const uint64_t frames = (offsets[q + 1] - offsets[q]) / bpf[q];
            const LoudGeom g = loud_geom(sr, frames);
            const bool ok = g.ok;
            const uint32_t S = g.S, nseg = g.nseg, nfull = g.nfull;
            if (rec) {
                LoudTrack& T = rec[q - i];
                memset(&T, 0, sizeof T);
                T.byte_off = offsets[q] - offsets[i];
                T.frames = frames;
                T.work = w;
                T.seg0 = sg;
                T.ch0 = nc;
                T.C = C;
                T.fmt = formats[q];
                T.S = S;
                T.nseg = nseg;
                T.nfull = nfull;
                T.J = g.J;
                T.K = g.K;
                if (ok) {
                    T.L = true_peak_factor(sr);
                    kweight_coeffs(sr, T.kw);
                    kweight_power(T.kw, S, T.M);
                    true_peak_taps(T.L, T.taps);
                }
            }
            if (wt)
                for (uint32_t c = 0; c < C; ++c) wt[nc + c] = chans_.map ? loud_class_weight(chans_.map[chans_.at[q] + c]) : loud_channel_weight(C, c);
            w += (uint64_t)nseg * C;
            sg += nseg;
            nc += C;
            if (ok) mc = std::max(mc, C);
        }
        *n_work = w;
        *n_seg = sg;
        *n_ch = nc;
        *max_c = mc;
    }

    // Device work area of a chunk: records and weight table (uploaded together), track then per-channel results (zeroed and read
    // back together), cascade states and energies, per-segment areas, with per-channel results their areas, with peak series the
    // work items' peaks, and one region of n_seg doubles per requested series.
    static size_t rec_bytes(uint64_t n_tracks, uint64_t n_ch) { return align_up(n_tracks * sizeof(LoudTrack), 256) + n_ch * sizeof(double); }
    size_t ws_bytes(uint64_t n_tracks, uint64_t n_work, uint64_t n_seg, uint64_t n_ch) const {
        return align_up(rec_bytes(n_tracks, n_ch), 256) + align_up((n_tracks + n_ch) * sizeof(LoudOut), 256) + align_up(5 * n_work * sizeof(double), 256) +
               align_up(4 * n_seg * sizeof(double), 256) + (chans_.out ? align_up(4 * n_work * sizeof(double), 256) : 0) +
               (ser_.peaks() ? align_up(2 * n_work * sizeof(float), 256) : 0) + ser_.count() * align_up(n_seg * sizeof(double), 256);
    }

    int open(const std::vector<HostChunk>& chunks) override {
        size_t need = 0, rec_max = 0, out_max = 0, blk_bytes = 0, ser_bytes = 0;
        for (const HostChunk& ch : chunks) {
            uint64_t w, sg, nc;
            uint32_t mc;
            plan(ch.i, ch.j, nullptr, nullptr, &w, &sg, &nc, &mc);
            need = std::max(need, ws_bytes(ch.j - ch.i, w, sg, nc));
            rec_max = std::max(rec_max, rec_bytes(ch.j - ch.i, nc));
            out_max = std::max<size_t>(out_max, (ch.j - ch.i + nc) * sizeof(LoudOut));
            if (has_member(ch.i, ch.j)) blk_bytes = std::max<size_t>(blk_bytes, 2 * sg * sizeof(double));
            ser_bytes = std::max<size_t>(ser_bytes, ser_.count() * sg * sizeof(double));
        }
        for (int b = 0; b < 2 && (blk_bytes || ser_bytes); ++b)
            if ((blk_bytes && !ctx->loud_blk[b].need(blk_bytes)) || (ser_bytes && !ctx->loud_ser[b].need(ser_bytes))) {
                set_error("pinned host allocation failed");
                return STRATUM_PROCESSING_ERROR;
            }
        for (int b = 0; b < 2; ++b)
            if (!ctx->loud_rec[b].need(rec_max) || !ctx->loud_out[b].need(out_max)) {
                set_error("pinned host allocation failed");
                return STRATUM_PROCESSING_ERROR;
            }
        if (!grow_device(ctx->d_loud, ctx->loud_cap, need)) {
            set_error("loudness work area allocation failed");
            return STRATUM_PROCESSING_ERROR;
        }
        for (cudaEvent_t& e : ctx->loud_ev)
            if (!e && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) {
                set_error("event creation failed");
                return STRATUM_PROCESSING_ERROR;
            }
        return STRATUM_OK;
    }

    int chunk(size_t k, const HostChunk& ch, const char* d_buf, const std::function<void()>& after_prev) override {
        const uint32_t n = ch.j - ch.i;
        char* h_rec = static_cast<char*>(ctx->loud_rec[k & 1].p);
        LoudTrack* h_tr = reinterpret_cast<LoudTrack*>(h_rec);
        LoudOut* h_out = static_cast<LoudOut*>(ctx->loud_out[k & 1].p);
        const uint64_t wt_off = align_up((uint64_t)n * sizeof(LoudTrack), 256);
        uint64_t n_work, n_seg, n_ch;
        uint32_t max_c;
        plan(ch.i, ch.j, h_tr, reinterpret_cast<double*>(h_rec + wt_off), &n_work, &n_seg, &n_ch, &max_c);
        char* d = ctx->d_loud;
        LoudTrack* d_tr = reinterpret_cast<LoudTrack*>(d);
        const double* d_wt = reinterpret_cast<const double*>(d + wt_off);
        d += align_up(rec_bytes(n, n_ch), 256);
        LoudOut* d_out = reinterpret_cast<LoudOut*>(d);
        LoudOut* d_chout = d_out + n;
        d += align_up((n + n_ch) * sizeof(LoudOut), 256);
        double* d_st = reinterpret_cast<double*>(d);
        double* d_en = d_st + 4 * n_work;
        d += align_up(5 * n_work * sizeof(double), 256);
        double* d_ws = reinterpret_cast<double*>(d);
        d += align_up(4 * n_seg * sizeof(double), 256);
        double* d_cws = chans_.out ? reinterpret_cast<double*>(d) : nullptr;
        if (chans_.out) d += align_up(4 * n_work * sizeof(double), 256);
        float* d_pk = ser_.peaks() ? reinterpret_cast<float*>(d) : nullptr;
        if (d_pk) d += align_up(2 * n_work * sizeof(float), 256);
        double* d_ser[4];
        for (int q = 0; q < 4; ++q) {
            d_ser[q] = ser_.dst[q] ? reinterpret_cast<double*>(d) : nullptr;
            if (d_ser[q]) d += align_up(n_seg * sizeof(double), 256);
        }
        cudaStream_t s = stream;
        CUDA_OK(cudaMemcpyAsync(d_tr, h_rec, rec_bytes(n, n_ch), cudaMemcpyHostToDevice, s));
        CUDA_OK(cudaMemsetAsync(d_out, 0, (size_t)(n + n_ch) * sizeof(LoudOut), s));
        g_h2d_bytes.fetch_add(rec_bytes(n, n_ch));
        {
            StageTimer tm(s, "loudness_pass1");
            launch_loud_pass1(s, d_buf, d_tr, n, n_work, d_st);
        }
        {
            StageTimer tm(s, "loudness_scan");
            launch_loud_scan(s, d_tr, n, max_c, d_st);
        }
        {
            StageTimer tm(s, "loudness_pass2");
            launch_loud_pass2(s, d_buf, d_tr, n, n_work, d_st, d_en, d_chout, d_pk);
        }
        {
            StageTimer tm(s, "loudness_gate");
            launch_loud_gate(s, d_tr, n, d_wt, d_en, d_ws, n_seg, d_out, d_cws, n_work, d_chout, chans_.out ? max_c : 0, d_pk,
                             LoudSeries{d_ser[0], d_ser[1], d_ser[2], d_ser[3]});
        }
        CUDA_OK(cudaGetLastError());
        const uint64_t n_read = chans_.out ? n + n_ch : n;  // the per-channel results follow the track results
        CUDA_OK(cudaMemcpyAsync(h_out, d_out, (size_t)n_read * sizeof(LoudOut), cudaMemcpyDeviceToHost, s));
        g_d2h_bytes.fetch_add(n_read * sizeof(LoudOut));
        const bool blocks = has_member(ch.i, ch.j);
        if (blocks) {  // the momentary and short-term regions of the work area are adjacent: one copy for both
            CUDA_OK(cudaMemcpyAsync(ctx->loud_blk[k & 1].p, d_ws + n_seg, 2 * n_seg * sizeof(double), cudaMemcpyDeviceToHost, s));
            g_d2h_bytes.fetch_add(2 * n_seg * sizeof(double));
        }
        double* h_ser = static_cast<double*>(ctx->loud_ser[k & 1].p);
        for (int q = 0; q < 4 && n_seg; ++q)  // the requested series one after the other, n_seg doubles each
            if (d_ser[q]) {
                CUDA_OK(cudaMemcpyAsync(h_ser, d_ser[q], n_seg * sizeof(double), cudaMemcpyDeviceToHost, s));
                g_d2h_bytes.fetch_add(n_seg * sizeof(double));
                h_ser += n_seg;
            }
        CUDA_OK(cudaEventRecord(ctx->loud_ev[k & 1], s));
        Slot& cur = slot[k & 1];
        cur.i = ch.i;
        cur.j = ch.j;
        cur.queued = true;
        cur.blocks = blocks;
        cur.n_seg = n_seg;
        cur.stages.swap(g_pending);
        g_pending.clear();
        const int st = gather((k + 1) & 1);  // the previous chunk: its staging buffer is free once it has finished
        after_prev();
        return st;
    }

    int gather(int b) {
        Slot& sl = slot[b];
        if (!sl.queued) return STRATUM_OK;
        sl.queued = false;
        CUDA_OK(cudaEventSynchronize(ctx->loud_ev[b]));
        resolve_stage_times(sl.stages);
        const LoudTrack* h_tr = static_cast<const LoudTrack*>(ctx->loud_rec[b].p);
        const LoudOut* h_out = static_cast<const LoudOut*>(ctx->loud_out[b].p);
        const uint32_t n = sl.j - sl.i;
        for (uint32_t q = sl.i; q < sl.j; ++q) {
            const LoudTrack& T = h_tr[q - sl.i];
            loud_result(T, h_out[q - sl.i], sample_rates[q], channels[q], out[q]);
            if (chans_.out)
                for (uint32_t c = 0; c < T.C; ++c) loud_result(T, h_out[n + T.ch0 + c], sample_rates[q], 1, chans_.out[chans_.at[q] + c]);
            if (out[q].status != STRATUM_OK) continue;
            if (sl.blocks && pools->member(q)) {
                const double* blk = static_cast<const double*>(ctx->loud_blk[b].p);
                memcpy(pools->buf.data() + pools->m_at[q], blk + T.seg0, (size_t)T.J * sizeof(double));
                memcpy(pools->buf.data() + pools->q_at[q], blk + sl.n_seg + T.seg0, (size_t)T.K * sizeof(double));
            }
            const double* h_ser = static_cast<const double*>(ctx->loud_ser[b].p);
            const uint32_t len[4] = {T.J, T.K, T.nseg, T.nseg};
            for (int s = 0; s < 4; ++s)
                if (ser_.dst[s]) {
                    memcpy(ser_.dst[s] + ser_.at[s][q], h_ser + T.seg0, (size_t)len[s] * sizeof(double));
                    h_ser += sl.n_seg;
                }
        }
        return STRATUM_OK;
    }

    static void loud_result(const LoudTrack& T, const LoudOut& o, uint32_t sr, uint32_t C, StratumLoudness& r) {
        memset(&r, 0, sizeof r);
        r.sample_rate = sr;
        r.channels = C;
        r.frames = T.frames;
        r.status = loud_track_status(r.sample_rate, r.frames, r.error, sizeof r.error);
        if (r.status != STRATUM_OK) return;
        r.integrated_lufs = o.integrated;
        r.momentary_max_lufs = o.momentary_max;
        r.short_term_max_lufs = o.short_term_max;
        r.loudness_range_lu = o.loudness_range;
        float f;
        memcpy(&f, &o.sample_peak_bits, sizeof f);
        r.sample_peak = f;
        memcpy(&f, &o.true_peak_bits, sizeof f);
        r.true_peak = f;
        r.n_momentary = T.J;
        r.n_short_term = T.K;
    }

    int close() override {
        const int s1 = gather(0), s2 = gather(1);
        return s1 != STRATUM_OK ? s1 : s2;
    }
};

static int32_t loudness_validate(const uint64_t* boff, const uint32_t* sample_rates, const uint32_t* channels, const uint32_t* formats, uint32_t n_tracks,
                                 StratumLoudness* out, bool have_pcm, std::vector<uint32_t>& bpf) {
    if (!boff || !sample_rates || !channels || !formats || !out || (!have_pcm && n_tracks && boff[n_tracks] > boff[0])) {
        set_error("null argument");
        return STRATUM_INVALID_INPUT;
    }
    bpf.assign(n_tracks, 1);
    return pcm_frame_bytes(boff, channels, formats, n_tracks, bpf);
}

// Channel classes: every code of the map a StratumChannelClass.  Runs after every other check of the call.
static int32_t channels_validate(const uint8_t* map, StratumLoudness* channel_out, const uint32_t* channels, uint32_t n_tracks, LoudChannels& lc) {
    lc.map = map;
    lc.out = channel_out;
    lc.at.assign(n_tracks + 1, 0);
    for (uint32_t q = 0; q < n_tracks; ++q) lc.at[q + 1] = lc.at[q] + channels[q];
    for (uint32_t q = 0; map && q < n_tracks; ++q)
        for (uint32_t c = 0; c < channels[q]; ++c)
            if (map[lc.at[q] + c] > STRATUM_CH_DUAL_MONO) {
                set_error("track " + std::to_string(q) + " channel " + std::to_string(c) + ": channel class " + std::to_string(map[lc.at[q] + c]) +
                          " is not one of STRATUM_CH_UNUSED (0) .. STRATUM_CH_DUAL_MONO (3)");
                return STRATUM_INVALID_INPUT;
            }
    return STRATUM_OK;
}

int32_t stratum_b200_loudness_channel_map(uint32_t wave_mask, uint32_t channels, int32_t dual_mono, uint8_t* map) {
    if (!map || channels < 1 || channels > 64) {
        set_error(!map ? "null argument" : "channels outside 1..64");
        return STRATUM_INVALID_INPUT;
    }
    const uint32_t side = 0x200u | 0x400u;  // SPEAKER_SIDE_LEFT, SPEAKER_SIDE_RIGHT
    uint32_t bits = wave_mask;
    for (uint32_t c = 0; c < channels; ++c) {
        uint8_t code;
        if (wave_mask == 0) {  // the default map of the channel count
            const double w = loud_channel_weight(channels, c);
            code = w == 0.0 ? STRATUM_CH_UNUSED : (w == 1.0 ? STRATUM_CH_FRONT : STRATUM_CH_SURROUND);
        } else if (bits == 0) {
            code = STRATUM_CH_UNUSED;  // beyond the set bits
        } else {
            const uint32_t bit = bits & (~bits + 1u);  // the lowest set bit left
            bits &= bits - 1u;
            if (bit == 0x8u || bit > 0x20000u) code = STRATUM_CH_UNUSED;  // SPEAKER_LOW_FREQUENCY; reserved bits and SPEAKER_ALL
            else if (bit & side) code = STRATUM_CH_SURROUND;
            else if (bit == 0x10u || bit == 0x20u) code = (wave_mask & side) ? STRATUM_CH_FRONT : STRATUM_CH_SURROUND;  // BACK_LEFT / RIGHT
            else code = STRATUM_CH_FRONT;
        }
        map[c] = code;
    }
    if (dual_mono && channels == 1 && map[0] != STRATUM_CH_UNUSED) map[0] = STRATUM_CH_DUAL_MONO;
    return STRATUM_OK;
}

// Album ids: each below n_albums or STRATUM_NO_ALBUM.
static int32_t albums_validate(const uint32_t* album_of, uint32_t n_tracks, uint32_t n_albums, const StratumLoudness* album_out) {
    if (n_albums == 0 && !album_of) return STRATUM_OK;
    if (n_albums > 0 && (!album_of || !album_out)) {
        set_error("null argument");
        return STRATUM_INVALID_INPUT;
    }
    for (uint32_t q = 0; q < n_tracks; ++q)
        if (album_of[q] >= n_albums && album_of[q] != STRATUM_NO_ALBUM) {
            set_error("track " + std::to_string(q) + ": album id " + std::to_string(album_of[q]) + " is not below n_albums = " + std::to_string(n_albums) +
                      " (STRATUM_NO_ALBUM for a track of no album)");
            return STRATUM_INVALID_INPUT;
        }
    return STRATUM_OK;
}

// The album results once every member is measured: status, frames and peaks from the member results on the host; the gates, maxima
// and range of the albums with all members measured from one launch of loud_album_gate_kernel over the pools, on device `device`.
static int32_t album_phase(int32_t device, AlbumPools& P, uint32_t n_tracks, const StratumLoudness* out, StratumLoudness* album_out) {
    const uint32_t na = P.n_albums;
    std::vector<uint32_t> members(na, 0);
    for (uint32_t a = 0; a < na; ++a) memset(&album_out[a], 0, sizeof album_out[a]);
    for (uint32_t q = 0; q < n_tracks; ++q) {
        if (!P.member(q)) continue;
        StratumLoudness& r = album_out[P.album_of[q]];
        ++members[P.album_of[q]];
        if (r.status != STRATUM_OK) continue;
        if (out[q].status != STRATUM_OK) {  // no values over a partial album
            r.status = out[q].status;
            snprintf(r.error, sizeof r.error, "track %u: %.100s", q, out[q].error);
            r.frames = 0;
            r.sample_peak = r.true_peak = 0.0;
            continue;
        }
        r.frames += out[q].frames;
        r.sample_peak = std::max(r.sample_peak, out[q].sample_peak);
        r.true_peak = std::max(r.true_peak, out[q].true_peak);
    }
    uint32_t n_ok = 0;
    for (uint32_t a = 0; a < na; ++a) {
        StratumLoudness& r = album_out[a];
        if (members[a] == 0) {
            r.status = STRATUM_INVALID_INPUT;
            snprintf(r.error, sizeof r.error, "album has no tracks");
        }
        if (r.status == STRATUM_OK) ++n_ok;
    }
    if (n_ok == 0) return STRATUM_OK;
    int st = STRATUM_OK;
    DeviceCtx* ctx = get_ctx(device, &st);
    if (!ctx) return st;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) {
        set_error("cudaSetDevice failed");
        return STRATUM_PROCESSING_ERROR;
    }
    // device: the host buffer as is (records, momentary pool, short-term pool), the selection scratch, the results
    const size_t buf_bytes = P.buf.size() * sizeof(double), keep_bytes = P.n_sht * sizeof(double);
    if (!grow_device(ctx->d_album, ctx->album_cap, buf_bytes + keep_bytes + na * sizeof(LoudOut))) {
        set_error("album work area allocation failed");
        return STRATUM_PROCESSING_ERROR;
    }
    double* d = reinterpret_cast<double*>(ctx->d_album);
    LoudOut* d_out = reinterpret_cast<LoudOut*>(d + P.buf.size() + P.n_sht);
    std::vector<LoudOut> h_out(na);
    cudaStream_t s = ctx->stream;
    CUDA_OK(cudaMemcpyAsync(d, P.buf.data(), buf_bytes, cudaMemcpyHostToDevice, s));
    g_h2d_bytes.fetch_add(buf_bytes);
    {
        StageTimer tm(s, "loudness_album_gate");
        launch_loud_album_gate(s, reinterpret_cast<const LoudAlbum*>(d), na, d + P.mom0, d + P.sht0, d + P.buf.size(), d_out);
    }
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(h_out.data(), d_out, na * sizeof(LoudOut), cudaMemcpyDeviceToHost, s));
    g_d2h_bytes.fetch_add(na * sizeof(LoudOut));
    std::vector<PendingStage> stages;
    stages.swap(g_pending);
    CUDA_OK(cudaStreamSynchronize(s));
    resolve_stage_times(stages);
    for (uint32_t a = 0; a < na; ++a) {
        StratumLoudness& r = album_out[a];
        if (r.status != STRATUM_OK) continue;
        r.integrated_lufs = h_out[a].integrated;
        r.momentary_max_lufs = h_out[a].momentary_max;
        r.short_term_max_lufs = h_out[a].short_term_max;
        r.loudness_range_lu = h_out[a].loudness_range;
        r.n_momentary = P.albums()[a].J;
        r.n_short_term = P.albums()[a].K;
    }
    return STRATUM_OK;
}

int32_t stratum_b200_loudness_series_lengths(uint32_t sample_rate, uint64_t frames, uint32_t* n_momentary, uint32_t* n_short_term, uint32_t* n_peaks) {
    char msg[128];
    const int st = loud_track_status(sample_rate, frames, msg, sizeof msg);
    const LoudGeom g = loud_geom(sample_rate, frames);
    if (n_momentary) *n_momentary = LoudSeriesOut::length(g, 0);
    if (n_short_term) *n_short_term = LoudSeriesOut::length(g, 1);
    if (n_peaks) *n_peaks = LoudSeriesOut::length(g, 2);
    return st;
}

int32_t stratum_b200_loudness_series_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                         const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                         const uint8_t* channel_map, const int32_t* device_ids, uint32_t n_devices, StratumLoudness* out,
                                         StratumLoudness* album_out, StratumLoudness* channel_out, double* momentary_lufs, double* short_term_lufs,
                                         double* sample_peaks, double* true_peaks) {
    std::vector<uint32_t> bpf;
    LoudChannels lc;
    LoudSeriesOut so;
    int st = loudness_validate(byte_offsets, sample_rates, channels, formats, n_tracks, out, pcm != nullptr, bpf);
    if (st == STRATUM_OK) st = albums_validate(album_of_track, n_tracks, n_albums, album_out);
    if (st == STRATUM_OK) st = channels_validate(channel_map, channel_out, channels, n_tracks, lc);
    if (st != STRATUM_OK) return st;
    AlbumPools pools;
    album_layout(album_of_track, n_albums, byte_offsets, bpf, sample_rates, n_tracks, pools);
    series_layout(momentary_lufs, short_term_lufs, sample_peaks, true_peaks, byte_offsets, bpf, sample_rates, n_tracks, so);
    AlbumPools* pp = n_albums ? &pools : nullptr;
    if (n_tracks)
        st = stream_host_batch(pcm, byte_offsets, bpf, n_tracks, device_ids, n_devices, [&](DeviceCtx* ctx) -> std::unique_ptr<ChunkSink> {
            return std::unique_ptr<ChunkSink>(new LoudnessSink(ctx, byte_offsets, bpf, sample_rates, channels, formats, out, pp, lc, so));
        });
    if (st != STRATUM_OK || n_albums == 0) return st;
    return album_phase(device_ids && n_devices ? device_ids[0] : -1, pools, n_tracks, out, album_out);
}

int32_t stratum_b200_loudness_series_pcm_device(const void* d_pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                                const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                                const uint8_t* channel_map, int32_t device_id, StratumLoudness* out, StratumLoudness* album_out,
                                                StratumLoudness* channel_out, double* momentary_lufs, double* short_term_lufs, double* sample_peaks,
                                                double* true_peaks) {
    std::vector<uint32_t> bpf;
    LoudChannels lc;
    LoudSeriesOut so;
    int st = loudness_validate(byte_offsets, sample_rates, channels, formats, n_tracks, out, d_pcm != nullptr, bpf);
    if (st == STRATUM_OK) st = albums_validate(album_of_track, n_tracks, n_albums, album_out);
    if (st == STRATUM_OK) st = channels_validate(channel_map, channel_out, channels, n_tracks, lc);
    if (st != STRATUM_OK) return st;
    AlbumPools pools;
    album_layout(album_of_track, n_albums, byte_offsets, bpf, sample_rates, n_tracks, pools);
    series_layout(momentary_lufs, short_term_lufs, sample_peaks, true_peaks, byte_offsets, bpf, sample_rates, n_tracks, so);
    if (n_tracks) {
        DeviceCtx* ctx = get_ctx(device_id, &st);
        if (!ctx) return st;
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (cudaSetDevice(ctx->device) != cudaSuccess) {
            set_error("cudaSetDevice failed");
            return STRATUM_PROCESSING_ERROR;
        }
        // the whole batch is one chunk: one launch of each kernel
        const std::vector<HostChunk> one{HostChunk{0, n_tracks, byte_offsets[n_tracks] - byte_offsets[0], 0}};
        LoudnessSink sink(ctx, byte_offsets, bpf, sample_rates, channels, formats, out, n_albums ? &pools : nullptr, lc, so);
        st = sink.open(one);
        if (st != STRATUM_OK) return st;
        const int s1 = sink.chunk(0, one[0], static_cast<const char*>(d_pcm) + byte_offsets[0], [] {});
        const int s2 = sink.close();
        st = s1 != STRATUM_OK ? s1 : s2;
    }
    if (st != STRATUM_OK || n_albums == 0) return st;
    return album_phase(device_id, pools, n_tracks, out, album_out);
}

int32_t stratum_b200_loudness_mapped_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                         const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                         const uint8_t* channel_map, const int32_t* device_ids, uint32_t n_devices, StratumLoudness* out,
                                         StratumLoudness* album_out, StratumLoudness* channel_out) {
    return stratum_b200_loudness_series_pcm(pcm, byte_offsets, sample_rates, channels, formats, n_tracks, album_of_track, n_albums, channel_map, device_ids,
                                            n_devices, out, album_out, channel_out, nullptr, nullptr, nullptr, nullptr);
}

int32_t stratum_b200_loudness_mapped_pcm_device(const void* d_pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                                const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                                const uint8_t* channel_map, int32_t device_id, StratumLoudness* out, StratumLoudness* album_out,
                                                StratumLoudness* channel_out) {
    return stratum_b200_loudness_series_pcm_device(d_pcm, byte_offsets, sample_rates, channels, formats, n_tracks, album_of_track, n_albums, channel_map,
                                                   device_id, out, album_out, channel_out, nullptr, nullptr, nullptr, nullptr);
}

int32_t stratum_b200_loudness_albums_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                         const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                         const int32_t* device_ids, uint32_t n_devices, StratumLoudness* out, StratumLoudness* album_out) {
    return stratum_b200_loudness_mapped_pcm(pcm, byte_offsets, sample_rates, channels, formats, n_tracks, album_of_track, n_albums, nullptr, device_ids,
                                            n_devices, out, album_out, nullptr);
}

int32_t stratum_b200_loudness_albums_pcm_device(const void* d_pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                                const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                                int32_t device_id, StratumLoudness* out, StratumLoudness* album_out) {
    return stratum_b200_loudness_mapped_pcm_device(d_pcm, byte_offsets, sample_rates, channels, formats, n_tracks, album_of_track, n_albums, nullptr,
                                                   device_id, out, album_out, nullptr);
}

int32_t stratum_b200_loudness_batch_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                        const uint32_t* formats, uint32_t n_tracks, const int32_t* device_ids, uint32_t n_devices, StratumLoudness* out) {
    return stratum_b200_loudness_mapped_pcm(pcm, byte_offsets, sample_rates, channels, formats, n_tracks, nullptr, 0, nullptr, device_ids, n_devices, out,
                                            nullptr, nullptr);
}

int32_t stratum_b200_loudness_batch_pcm_device(const void* d_pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                               const uint32_t* formats, uint32_t n_tracks, int32_t device_id, StratumLoudness* out) {
    return stratum_b200_loudness_mapped_pcm_device(d_pcm, byte_offsets, sample_rates, channels, formats, n_tracks, nullptr, 0, nullptr, device_id, out,
                                                   nullptr, nullptr);
}

// Analysis and loudness of the same staged chunks: one upload feeds both.  The loudness passes of a chunk are queued first, on a
// stream of their own, so they need not wait behind the analysis waves (where the waves keep the device busy they still add their
// own kernel time: DESIGN §2).  The staged chunk is complete when chunk() is called (the uploads synchronise per piece), so that
// stream needs no event to read it.  The previous chunk's staging buffer is released once both halves are done with it: the
// loudness half after its gather, the analysis half once its mono conversion has run.
struct AnalysisLoudnessSink final : ChunkSink {
    AnalysisSink ana;
    LoudnessSink loud;
    AnalysisLoudnessSink(DeviceCtx* c, const StratumConfig& cfg, const uint64_t* offs, const std::vector<uint32_t>& bpf, const uint32_t* srs,
                         const uint32_t* chans, const uint32_t* fmts, StratumResult* o, StratumLoudness* lo, AlbumPools* p, const LoudChannels& lc,
                         const LoudSeriesOut& so)
        : ana(c, cfg, offs, bpf, srs, chans, fmts, o), loud(c, offs, bpf, srs, chans, fmts, lo, p, lc, so) {}

    int open(const std::vector<HostChunk>& chunks) override {
        DeviceCtx* ctx = ana.ctx;
        if (!ctx->loud_stream && cudaStreamCreateWithFlags(&ctx->loud_stream, cudaStreamNonBlocking) != cudaSuccess) {
            set_error("loudness stream creation failed");
            return STRATUM_PROCESSING_ERROR;
        }
        loud.stream = ctx->loud_stream;
        // the loudness buffers first: Session::open sizes the analysis arena from the device memory still free
        const int st = loud.open(chunks);
        return st != STRATUM_OK ? st : ana.open(chunks);
    }

    int chunk(size_t k, const HostChunk& ch, const char* d_buf, const std::function<void()>& after_prev) override {
        int done = 0;
        const std::function<void()> half_done = [&] {
            if (++done == 2) after_prev();
        };
        const int st = loud.chunk(k, ch, d_buf, half_done);
        return st != STRATUM_OK ? st : ana.chunk(k, ch, d_buf, half_done);
    }

    int close() override {
        const int s1 = ana.close(), s2 = loud.close();
        cudaStreamSynchronize(loud.stream);  // after a failure inside loud.chunk, launches without a recorded event may still read the staging buffer
        return s1 != STRATUM_OK ? s1 : s2;
    }
};

int32_t stratum_b200_analyze_loudness_series_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                                 const uint32_t* formats, uint32_t n_tracks, const StratumConfig* cfg, const uint32_t* album_of_track,
                                                 uint32_t n_albums, const uint8_t* channel_map, const int32_t* device_ids, uint32_t n_devices,
                                                 StratumResult* out, StratumLoudness* loudness_out, StratumLoudness* album_out,
                                                 StratumLoudness* channel_out, double* momentary_lufs, double* short_term_lufs, double* sample_peaks,
                                                 double* true_peaks) {
    // the order of stratum_b200_analyze_batch_pcm: NULL pointers, the configuration, the PCM layout; then the album ids, the channel map
    if (!byte_offsets || !sample_rates || !channels || !formats || !out || !loudness_out || (!pcm && n_tracks && byte_offsets[n_tracks] > 0)) {
        set_error("null argument");
        return STRATUM_INVALID_INPUT;
    }
    StratumConfig def;
    config_default(&def);
    const StratumConfig& c = cfg ? *cfg : def;
    std::vector<uint32_t> bpf;
    LoudChannels lc;
    LoudSeriesOut so;
    int st = config_validate(c);
    if (st == STRATUM_OK) st = loudness_validate(byte_offsets, sample_rates, channels, formats, n_tracks, loudness_out, pcm != nullptr, bpf);
    if (st == STRATUM_OK) st = albums_validate(album_of_track, n_tracks, n_albums, album_out);
    if (st == STRATUM_OK) st = channels_validate(channel_map, channel_out, channels, n_tracks, lc);
    if (st != STRATUM_OK) return st;
    AlbumPools pools;
    album_layout(album_of_track, n_albums, byte_offsets, bpf, sample_rates, n_tracks, pools);
    series_layout(momentary_lufs, short_term_lufs, sample_peaks, true_peaks, byte_offsets, bpf, sample_rates, n_tracks, so);
    AlbumPools* pp = n_albums ? &pools : nullptr;
    if (n_tracks)
        st = stream_host_batch(pcm, byte_offsets, bpf, n_tracks, device_ids, n_devices, [&](DeviceCtx* ctx) -> std::unique_ptr<ChunkSink> {
            return std::unique_ptr<ChunkSink>(
                new AnalysisLoudnessSink(ctx, c, byte_offsets, bpf, sample_rates, channels, formats, out, loudness_out, pp, lc, so));
        });
    if (st != STRATUM_OK || n_albums == 0) return st;
    return album_phase(device_ids && n_devices ? device_ids[0] : -1, pools, n_tracks, loudness_out, album_out);
}

int32_t stratum_b200_analyze_loudness_mapped_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                                 const uint32_t* formats, uint32_t n_tracks, const StratumConfig* cfg, const uint32_t* album_of_track,
                                                 uint32_t n_albums, const uint8_t* channel_map, const int32_t* device_ids, uint32_t n_devices,
                                                 StratumResult* out, StratumLoudness* loudness_out, StratumLoudness* album_out,
                                                 StratumLoudness* channel_out) {
    return stratum_b200_analyze_loudness_series_pcm(pcm, byte_offsets, sample_rates, channels, formats, n_tracks, cfg, album_of_track, n_albums, channel_map,
                                                    device_ids, n_devices, out, loudness_out, album_out, channel_out, nullptr, nullptr, nullptr, nullptr);
}

int32_t stratum_b200_analyze_loudness_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                          const uint32_t* formats, uint32_t n_tracks, const StratumConfig* cfg, const uint32_t* album_of_track,
                                          uint32_t n_albums, const int32_t* device_ids, uint32_t n_devices, StratumResult* out,
                                          StratumLoudness* loudness_out, StratumLoudness* album_out) {
    return stratum_b200_analyze_loudness_mapped_pcm(pcm, byte_offsets, sample_rates, channels, formats, n_tracks, cfg, album_of_track, n_albums, nullptr,
                                                    device_ids, n_devices, out, loudness_out, album_out, nullptr);
}

int32_t stratum_b200_debug_loudness_filters(uint32_t sample_rate, double* kweight10, float* taps49) {
    char msg[128];
    if (loud_track_status(sample_rate, 1, msg, sizeof msg) != STRATUM_OK) return -1;
    const uint32_t L = true_peak_factor(sample_rate);
    if (kweight10) kweight_coeffs(sample_rate, kweight10);
    if (taps49) true_peak_taps(L, taps49);
    return (int32_t)L;
}

void stratum_b200_debug_mel_schedule(const int32_t* mel_off, uint32_t n_mels, int32_t* schedule256) {
    if (!mel_off || !schedule256 || n_mels > 40) return;
    mel_fold_schedule(mel_off, n_mels, schedule256);
}

int32_t stratum_b200_debug_bpm_grid(float min_bpm, float max_bpm, float bpm_resolution, float* out, int32_t cap) {
    if (!(min_bpm > 0.0f) || !(max_bpm > min_bpm) || !(bpm_resolution > 0.0f)) return -1;
    return bpm_grid(min_bpm, max_bpm, bpm_resolution, out, out ? cap : 0);
}

uint32_t stratum_b200_debug_plan_waves(const uint64_t* offsets, const uint32_t* sample_rates, uint32_t n_tracks, const StratumConfig* cfg, double budget_gb,
                                       uint32_t* wave_of_track) {
    StratumConfig def;
    config_default(&def);
    const StratumConfig& c = cfg ? *cfg : def;
    std::vector<uint64_t> lens(n_tracks);
    for (uint32_t q = 0; q < n_tracks; ++q) lens[q] = offsets[q + 1] - offsets[q];
    WaveLimits lim{(uint64_t)(budget_gb * 1e9 / 4), WAVE_MAX_TRACKS, WAVE_CAP_SAMPLES};
    const DevCfg kd = make_devcfg(c);
    uint32_t i = 0, nw = 0;
    while (i < n_tracks) {
        WavePlan wp;
        pack_wave(i, n_tracks, lens.data(), sample_rates, c, kd, lim, wp);
        for (uint32_t q : wp.idx) wave_of_track[q] = nw;
        ++nw;
    }
    return nw;
}

static std::vector<uint64_t> scaled_offsets(const uint64_t* offsets, uint32_t n, uint64_t elt) {
    std::vector<uint64_t> b((size_t)n + 1, 0);
    if (offsets)
        for (uint32_t i = 0; i <= n; ++i) b[i] = offsets[i] * elt;
    return b;
}

int32_t stratum_b200_analyze_batch(const float* samples, const uint64_t* offsets, const uint32_t* sample_rates, uint32_t n_tracks, const StratumConfig* cfg,
                                   const int32_t* device_ids, uint32_t n_devices, StratumResult* out) {
    const std::vector<uint64_t> b = scaled_offsets(offsets, n_tracks, sizeof(float));
    return analyze_host_batch(samples, offsets ? b.data() : nullptr, sample_rates, nullptr, nullptr, n_tracks, cfg, device_ids, n_devices, out);
}

int32_t stratum_b200_analyze_batch_pcm16(const int16_t* pcm, const uint64_t* offsets, const uint32_t* sample_rates, const uint32_t* channels, uint32_t n_tracks,
                                         const StratumConfig* cfg, const int32_t* device_ids, uint32_t n_devices, StratumResult* out) {
    const std::vector<uint64_t> b = scaled_offsets(offsets, n_tracks, sizeof(int16_t));
    const std::vector<uint32_t> fmt(n_tracks, (uint32_t)STRATUM_PCM_S16);
    if (!channels) {
        set_error("null argument");
        return STRATUM_INVALID_INPUT;
    }
    return analyze_host_batch(pcm, offsets ? b.data() : nullptr, sample_rates, channels, fmt.data(), n_tracks, cfg, device_ids, n_devices, out);
}

int32_t stratum_b200_analyze_batch_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels, const uint32_t* formats,
                                       uint32_t n_tracks, const StratumConfig* cfg, const int32_t* device_ids, uint32_t n_devices, StratumResult* out) {
    if (!formats || !channels) {
        set_error("null argument");
        return STRATUM_INVALID_INPUT;
    }
    return analyze_host_batch(pcm, byte_offsets, sample_rates, channels, formats, n_tracks, cfg, device_ids, n_devices, out);
}

int32_t stratum_b200_analyze_audio(const float* samples, uint64_t n_samples, uint32_t sample_rate, const StratumConfig* cfg, StratumResult* out) {
    if (!out) {
        set_error("null argument");
        return STRATUM_INVALID_INPUT;
    }
    const uint64_t offsets[2] = {0, n_samples};
    const int st = stratum_b200_analyze_batch(samples, offsets, &sample_rate, 1, cfg, nullptr, 0, out);
    if (st != STRATUM_OK) {
        memset(out, 0, sizeof *out);
        out->status = st;
        snprintf(out->error, sizeof out->error, "%s", g_last_error.c_str());
        return st;
    }
    return out->status;
}

int32_t stratum_b200_warning_strings(const StratumResult* r, char* buf, size_t cap) {  // lib.rs:1567-1589, exact strings
    std::string all;
    char tmp[256];
    if (r->warnings & STRATUM_WARN_BPM_FAILED) all += "BPM detection failed: insufficient onsets or estimation error\n";
    if (r->warnings & STRATUM_WARN_LOW_GRID_STABILITY) {
        snprintf(tmp, sizeof tmp, "Low beat grid stability: %.2f (may indicate tempo variation)\n", r->grid_stability);
        all += tmp;
    }
    if (r->warnings & STRATUM_WARN_LOW_KEY_CONFIDENCE) {
        snprintf(tmp, sizeof tmp, "Low key detection confidence: %.2f (may indicate ambiguous or atonal music)\n", r->key_confidence);
        all += tmp;
    }
    if (r->warnings & STRATUM_WARN_LOW_KEY_CLARITY) {
        snprintf(tmp, sizeof tmp, "Low key clarity: %.2f (track may be atonal or have weak tonality)\n", r->key_clarity);
        all += tmp;
    }
    if (buf && cap > 0) {
        strncpy(buf, all.c_str(), cap - 1);
        buf[cap - 1] = 0;
    }
    return (int32_t)all.size();
}

void stratum_b200_compute_confidence(const StratumResult* r, StratumConfidence* out) {  // analysis/confidence.rs:121-297
    char wb[1024];
    stratum_b200_warning_strings(r, wb, sizeof wb);
    const std::string warns = wb;
    auto contains = [&](const char* needle) { return warns.find(needle) != std::string::npos; };
    auto clamp01 = [](float x) { return x < 0.0f ? 0.0f : (x > 1.0f ? 1.0f : x); };
    float bc = 0.0f;
    if (r->bpm > 0.0f) {
        bc = clamp01(r->bpm_confidence);
        if (contains("BPM")) bc = bc * 0.7f;
    }
    float kc = 0.0f;
    if (r->key_confidence > 0.0f) {
        const float base = clamp01(r->key_confidence);
        const float ca = r->key_clarity < 0.2f ? 0.6f : (r->key_clarity < 0.5f ? 0.85f : 1.0f);
        const float wa = (contains("key") || contains("Key") || contains("tonality")) ? 0.7f : 1.0f;
        kc = base * ca * wa;
    }
    const float gs = clamp01(r->grid_stability);
    float overall;
    if (bc > 0.0f && kc > 0.0f) overall = clamp01(bc * 0.4f + kc * 0.3f + gs * 0.3f);
    else if (bc > 0.0f) overall = bc * 0.6f;
    else if (kc > 0.0f) overall = kc * 0.6f;
    else overall = 0.0f;
    uint32_t flags = r->flags;
    if (bc < 0.3f) flags |= STRATUM_FLAG_MULTIMODAL_BPM;
    if (kc < 0.2f) flags |= STRATUM_FLAG_WEAK_TONALITY;
    if (gs < 0.3f) flags |= STRATUM_FLAG_TEMPO_VARIATION;
    out->bpm_confidence = bc;
    out->key_confidence = kc;
    out->grid_stability = gs;
    out->overall_confidence = overall;
    out->flags = flags;
}

int32_t stratum_b200_key_name(int32_t key_is_minor, uint32_t key_index, int32_t numerical, char* buf, size_t cap) {  // analysis/result.rs:31-87
    static const char* NOTE[12] = {"C", "C#", "D", "D#", "E", "F", "F#", "G", "G#", "A", "A#", "B"};
    std::string s;
    if (!numerical) {
        s = NOTE[key_index % 12];
        if (key_is_minor) s += "m";
    } else {
        const int cof_major[12] = {0, 7, 2, 9, 4, 11, 6, 1, 8, 3, 10, 5};
        const int cof_minor[12] = {9, 4, 11, 6, 1, 8, 3, 10, 5, 0, 7, 2};
        const int* t = key_is_minor ? cof_minor : cof_major;
        int pos = 0;
        for (int i = 0; i < 12; ++i)
            if (t[i] == (int)(key_index % 12)) {
                pos = i;
                break;
            }
        s = std::to_string(pos + 1) + (key_is_minor ? "B" : "A");
    }
    if (buf && cap > 0) {
        strncpy(buf, s.c_str(), cap - 1);
        buf[cap - 1] = 0;
    }
    return (int32_t)s.size();
}

void stratum_b200_result_free(StratumResult* results, uint32_t n) {
    if (!results) return;
    for (uint32_t i = 0; i < n; ++i) {
        free(results[i].beats);
        free(results[i].downbeats);
        free(results[i].bars);
        free(results[i].onsets);
        free(results[i].hmm_beat_frames);
        free(results[i].tempogram_candidates);
        results[i].tempogram_candidates = nullptr;
        results[i].n_tempogram_candidates = -1;
        results[i].beats = results[i].downbeats = results[i].bars = nullptr;
        results[i].onsets = nullptr;
        results[i].hmm_beat_frames = nullptr;
        results[i].n_beats = results[i].n_downbeats = results[i].n_bars = results[i].n_onsets = results[i].n_hmm_beat_frames = 0;
    }
}

int32_t stratum_b200_last_error(char* buf, size_t cap) {
    if (buf && cap > 0) {
        strncpy(buf, g_last_error.c_str(), cap - 1);
        buf[cap - 1] = 0;
    }
    return (int32_t)g_last_error.size();
}

uint64_t stratum_b200_launch_count(void) { return g_launches.load(); }

int32_t stratum_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

void stratum_b200_shutdown(void) {
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    for (auto& kv : g_ctx) {
        DeviceCtx* c = kv.second;
        if (!c) continue;
        if (c->ready) {
            cudaSetDevice(c->device);
            cudaStreamSynchronize(c->stream);
            if (c->loud_stream) cudaStreamSynchronize(c->loud_stream);
            for (void* p : c->owned) cudaFree(p);
            cudaFree(c->fa);
            cudaFree(c->oa);
            cudaFree(c->ia);
            cudaFree(c->d_tracks);
            cudaFree(c->d_sr_index);
            cudaFree(c->d_list);
            cudaFree(c->d_gain);
            cudaFree(c->d_srtab);
            cudaFree(c->d_stage);
            cudaFree(c->d_conv);
            cudaFree(c->d_meta);
            cudaFree(c->d_loud);
            cudaFree(c->d_album);
            cudaFree(c->d_count);
            c->uploader.reset();
            for (WaveJob& j : c->jobs) {
                j.h_tracks.release();
                j.h_oa.release();
                j.h_ia.release();
                j.h_small.release();
                if (j.ev0) cudaEventDestroy(j.ev0);
                if (j.ev1) cudaEventDestroy(j.ev1);
            }
            c->h_meta[0].release();
            c->h_meta[1].release();
            for (int b = 0; b < 2; ++b) {
                c->loud_rec[b].release();
                c->loud_out[b].release();
                c->loud_blk[b].release();
                c->loud_ser[b].release();
                if (c->loud_ev[b]) cudaEventDestroy(c->loud_ev[b]);
            }
            c->h_count.release();
            if (c->ev_legacy) cudaEventDestroy(c->ev_legacy);
            if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
            if (c->loud_stream) cudaStreamDestroy(c->loud_stream);
            cudaStreamDestroy(c->stream);
            if (c->key_stream) cudaStreamDestroy(c->key_stream);
        }
        delete c;
    }
    g_ctx.clear();
}

size_t stratum_b200_sizeof(int32_t which) {
    switch (which) {
        case 0: return sizeof(StratumConfig);
        case 1: return sizeof(StratumResult);
        case 2: return sizeof(StratumConfidence);
        case 3: return sizeof(StratumLoudness);
        default: return 0;
    }
}

int64_t stratum_b200_stft(const float* samples, uint64_t n, uint32_t frame_size, uint32_t hop, float gain, float* out, uint64_t out_cap) {
    if (frame_size < 64 || frame_size > 16384 || (frame_size & (frame_size - 1)) != 0) {
        set_error("frame_size must be a power of two between 64 and 16384");
        return -STRATUM_NOT_IMPLEMENTED;
    }
    if (hop == 0 || !samples || !out) {
        set_error("invalid argument");
        return -STRATUM_INVALID_INPUT;
    }
    if (n < frame_size) return 0;
    int st;
    DeviceCtx* ctx = get_ctx(-1, &st);
    if (!ctx) return -st;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    cudaSetDevice(ctx->device);
    const uint32_t frames = (uint32_t)((n - frame_size) / hop + 1);
    const uint64_t need = (uint64_t)frames * (frame_size / 2 + 1);
    if (need > out_cap) {
        set_error("output buffer too small");
        return -STRATUM_INVALID_INPUT;
    }
    float *d_in = nullptr, *d_out = nullptr;
    if (cudaMalloc(&d_in, n * sizeof(float)) != cudaSuccess || cudaMalloc(&d_out, need * sizeof(float)) != cudaSuccess) {
        cudaFree(d_in);
        set_error("allocation failed");
        return -STRATUM_PROCESSING_ERROR;
    }
    cudaMemcpyAsync(d_in, samples, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
    GenStft gen{};
    if (frame_size != 2048 && frame_size != 8192) {
        gen = get_gen_stft(*ctx, frame_size);
        if (gen.n == 0) {
            cudaFree(d_in);
            cudaFree(d_out);
            set_error("table allocation failed");
            return -STRATUM_PROCESSING_ERROR;
        }
    }
    launch_stft_raw(ctx->stream, d_in, n, frame_size, hop, gain, ctx->tab, d_out, frames, &gen);
    cudaMemcpyAsync(out, d_out, need * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_in);
    cudaFree(d_out);
    if (e != cudaSuccess) {
        set_error(std::string("CUDA error: ") + cudaGetErrorString(e));
        return -STRATUM_PROCESSING_ERROR;
    }
    return frames;
}

double stratum_b200_fp32_peak_tflops(int32_t device_id) {
    int st;
    DeviceCtx* ctx = get_ctx(device_id, &st);
    if (!ctx) return 0.0;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return 0.0;
    float* d = nullptr;
    if (cudaMalloc(&d, 256) != cudaSuccess) return 0.0;
    const double tf = measure_fp32_peak_tflops(ctx->stream, d);
    cudaFree(d);
    return tf;
}

int32_t stratum_b200_debug_check_divisions(uint64_t n, uint32_t seed, uint64_t* mismatches3) {
    int st;
    DeviceCtx* ctx = get_ctx(-1, &st);
    if (!ctx) return st;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    CUDA_OK(cudaSetDevice(ctx->device));
    unsigned long long* d = nullptr;
    CUDA_OK(cudaMalloc(&d, 3 * sizeof(unsigned long long)));
    const int rc = check_divisions(ctx->stream, n, seed, d);
    unsigned long long h[3] = {~0ull, ~0ull, ~0ull};
    const cudaError_t e = cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost);
    cudaFree(d);
    CUDA_OK(e);
    for (int i = 0; i < 3; ++i) mismatches3[i] = h[i];
    return rc == 0 ? STRATUM_OK : STRATUM_PROCESSING_ERROR;
}

int32_t stratum_b200_synth_batch(float* d_out, uint32_t n_tracks, uint64_t n_samples, uint32_t sample_rate, const float* params5, int32_t device_id) {
    int st;
    DeviceCtx* ctx = get_ctx(device_id, &st);
    if (!ctx) return st;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    CUDA_OK(cudaSetDevice(ctx->device));
    float* d_p = nullptr;
    CUDA_OK(cudaMalloc(&d_p, sizeof(float) * 5 * n_tracks));
    CUDA_OK(cudaMemcpyAsync(d_p, params5, sizeof(float) * 5 * n_tracks, cudaMemcpyHostToDevice, ctx->stream));
    launch_synth(ctx->stream, d_out, n_tracks, n_samples, sample_rate, d_p);
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_p);
    CUDA_OK(e);
    return STRATUM_OK;
}

int64_t stratum_b200_debug_array(const char* name, float* out, int64_t cap) {
    std::lock_guard<std::mutex> lk(g_debug_mu);
    auto it = g_debug_arrays.find(name);
    if (it == g_debug_arrays.end()) return -1;
    const int64_t n = (int64_t)it->second.size();
    if (out && cap > 0) memcpy(out, it->second.data(), sizeof(float) * (size_t)std::min<int64_t>(n, cap));
    return n;
}

void stratum_b200_debug_enable(int32_t on) {
    g_debug.store(on);
    if (!on) {
        std::lock_guard<std::mutex> lk(g_debug_mu);
        g_debug_arrays.clear();
    }
}

int32_t stratum_b200_stage_times(char* names, size_t cap, double* ms, int32_t max_stages) {
    std::lock_guard<std::mutex> lk(g_stage_mu);
    std::string all;
    int32_t n = 0;
    for (const std::string& s : g_stage_order) {
        if (n >= max_stages) break;
        all += s + "\n";
        if (ms) ms[n] = g_stage_ms[s];
        ++n;
    }
    if (names && cap > 0) {
        strncpy(names, all.c_str(), cap - 1);
        names[cap - 1] = 0;
    }
    return n;
}

void stratum_b200_stage_times_reset(void) {
    std::lock_guard<std::mutex> lk(g_stage_mu);
    g_stage_ms.clear();
    g_stage_order.clear();
}

void stratum_b200_stage_timing_enable(int32_t on) { g_timing.store(on); }

double stratum_b200_last_call_device_ms(void) { return (double)g_last_call_us.load() / 1000.0; }

uint32_t stratum_b200_last_call_waves(void) { return g_last_call_waves.load(); }

void stratum_b200_transfer_bytes(uint64_t* h2d, uint64_t* d2h) {
    if (h2d) *h2d = g_h2d_bytes.load();
    if (d2h) *d2h = g_d2h_bytes.load();
}

}  // extern "C"
