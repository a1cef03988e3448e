// engine.cu -- host-side engine: database packing, geometry choice, precision ladder, launches.
//
// Plays the role of the reference's escalation drivers searchDatabaseSW / searchDatabase<MODE>
// (reference src/opal.cpp:496-535, 983-1021) and of lane refill (loadNextSequence, :472-490), but
// scheduled for a GPU: the database is sorted by length once (longest first), adjacent targets
// are paired into the two 16-bit lanes of a group, warps pull groups of similar length from a
// global counter, and the 16 -> 32 bit escalation re-runs exactly the flagged targets.
#include "engine.h"

#include <emmintrin.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <climits>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <thread>
#include <unordered_map>

#include "r_list.h"
#include "pairs_kernel.cuh"
#include "search_kernel.cuh"

namespace opalb200 {

// ------------------------------------------------------------------ errors
static thread_local std::string g_lastError;
void set_error(const std::string& msg) { g_lastError = msg; }
const char* last_error() { return g_lastError.c_str(); }

#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                   \
            return false;                                                                    \
        }                                                                                    \
    } while (0)

// ------------------------------------------------------------------ phase tracing (OPAL_B200_TRACE=1)
struct PhaseTrace {
    bool on;
    const char* what;
    std::chrono::steady_clock::time_point last;
    std::string line;
    explicit PhaseTrace(const char* w) : on(getenv("OPAL_B200_TRACE") != nullptr), what(w) { if (on) last = std::chrono::steady_clock::now(); }
    void mark(const char* phase) {
        if (!on) return;
        const auto now = std::chrono::steady_clock::now();
        char buf[96];
        snprintf(buf, sizeof(buf), " %s %.0f us,", phase, std::chrono::duration<double, std::micro>(now - last).count());
        line += buf;
        last = now;
    }
    ~PhaseTrace() { if (on && !line.empty()) fprintf(stderr, "[opal-b200] %s:%s\n", what, line.c_str()); }
};

// ------------------------------------------------------------------ kernel registry
#define OPAL_DECLARE_TABLE(R) const void* const* kernel_table_R##R(); const void* const* kernel_chain_table_R##R();
OPAL_R_LIST(OPAL_DECLARE_TABLE)
#undef OPAL_DECLARE_TABLE

const std::vector<KernelTable>& kernel_tables() {
    static const std::vector<KernelTable> tables = {
#define OPAL_TABLE_ENTRY(R) {R, kernel_table_R##R(), kernel_chain_table_R##R()},
        OPAL_R_LIST(OPAL_TABLE_ENTRY)
#undef OPAL_TABLE_ENTRY
    };
    return tables;
}

// ------------------------------------------------------------------ per-device resource cache
// opalSearchDatabase packs and uploads its database on every call (the reference's signature takes
// host pointers each time), so the CUDA allocations behind a call are recycled instead of being
// returned to the driver: cudaMalloc / cudaMallocHost / stream and event creation cost far more
// than the search itself on a 12k-sequence database.  Blocks are matched by size (first cached block
// within 2x of the request); the cache is bounded and thread-safe.
namespace {
struct DeviceInfo { bool known = false; int numSMs = 0, smemLimit = 0, major = 0; };
struct CachedBlock { void* p; size_t bytes; };
struct ResourceCache {
    std::mutex mu;
    std::vector<CachedBlock> freeDevice[kMaxDevices], freePinned;
    std::unordered_map<void*, size_t> liveBytes;
    std::vector<cudaStream_t> streams[kMaxDevices];
    std::vector<cudaEvent_t> events[kMaxDevices];
    DeviceInfo info[kMaxDevices];
    size_t cachedDevice[kMaxDevices] = {0}, cachedPinned = 0;
};
ResourceCache& cache() { static ResourceCache* c = new ResourceCache(); return *c; }  // leaked on purpose: no teardown order issues
constexpr size_t kMaxCachedDevice = 8ull << 30, kMaxCachedPinned = 2ull << 30;

bool take_block(std::vector<CachedBlock>& list, size_t bytes, void** out, size_t* got) {
    size_t best = list.size();
    for (size_t i = 0; i < list.size(); i++)
        if (list[i].bytes >= bytes && list[i].bytes <= 2 * bytes + (1 << 16) && (best == list.size() || list[i].bytes < list[best].bytes)) best = i;
    if (best == list.size()) return false;
    *out = list[best].p; *got = list[best].bytes;
    list[best] = list.back(); list.pop_back();
    return true;
}
}  // namespace

bool device_alloc(int device, void** p, size_t bytes) {
    bytes = std::max<size_t>(bytes, 256);
    ResourceCache& c = cache();
    {
        std::lock_guard<std::mutex> lk(c.mu);
        size_t got = 0;
        if (take_block(c.freeDevice[device], bytes, p, &got)) { c.cachedDevice[device] -= got; c.liveBytes[*p] = got; return true; }
    }
    CUDA_TRY(cudaMalloc(p, bytes));
    std::lock_guard<std::mutex> lk(c.mu);
    c.liveBytes[*p] = bytes;
    return true;
}
void device_release(int device, void* p) {
    if (!p) return;
    ResourceCache& c = cache();
    std::lock_guard<std::mutex> lk(c.mu);
    const size_t bytes = c.liveBytes[p];
    c.liveBytes.erase(p);
    if (c.cachedDevice[device] + bytes > kMaxCachedDevice) { cudaFree(p); return; }
    c.freeDevice[device].push_back({p, bytes});
    c.cachedDevice[device] += bytes;
}
static bool pinned_alloc(void** p, size_t bytes) {
    bytes = std::max<size_t>(bytes, 256);
    ResourceCache& c = cache();
    {
        std::lock_guard<std::mutex> lk(c.mu);
        size_t got = 0;
        if (take_block(c.freePinned, bytes, p, &got)) { c.cachedPinned -= got; c.liveBytes[*p] = got; return true; }
    }
    CUDA_TRY(cudaMallocHost(p, bytes));
    std::lock_guard<std::mutex> lk(c.mu);
    c.liveBytes[*p] = bytes;
    return true;
}
static void pinned_release(void* p) {
    if (!p) return;
    ResourceCache& c = cache();
    std::lock_guard<std::mutex> lk(c.mu);
    const size_t bytes = c.liveBytes[p];
    c.liveBytes.erase(p);
    if (c.cachedPinned + bytes > kMaxCachedPinned) { cudaFreeHost(p); return; }
    c.freePinned.push_back({p, bytes});
    c.cachedPinned += bytes;
}
// Returns every cached (not live) device and pinned block to the driver.
void trim_cache() {
    ResourceCache& c = cache();
    std::vector<std::pair<int, void*>> dev;
    std::vector<void*> pinned;
    {
        std::lock_guard<std::mutex> lk(c.mu);
        for (int d = 0; d < kMaxDevices; d++) {
            for (const CachedBlock& b : c.freeDevice[d]) dev.push_back({d, b.p});
            c.freeDevice[d].clear();
            c.cachedDevice[d] = 0;
        }
        for (const CachedBlock& b : c.freePinned) pinned.push_back(b.p);
        c.freePinned.clear();
        c.cachedPinned = 0;
    }
    int saved = -1;
    if (cudaGetDevice(&saved) != cudaSuccess) saved = -1;
    for (const auto& b : dev) { cudaSetDevice(b.first); cudaFree(b.second); }
    for (void* p : pinned) cudaFreeHost(p);
    if (saved >= 0) cudaSetDevice(saved);
}

static bool stream_acquire(int device, cudaStream_t* s) {
    ResourceCache& c = cache();
    {
        std::lock_guard<std::mutex> lk(c.mu);
        auto& v = c.streams[device];
        if (!v.empty()) { *s = v.back(); v.pop_back(); return true; }
    }
    CUDA_TRY(cudaStreamCreateWithFlags(s, cudaStreamNonBlocking));
    return true;
}
static void stream_release(int device, cudaStream_t s) {
    if (!s) return;
    ResourceCache& c = cache();
    std::lock_guard<std::mutex> lk(c.mu);
    c.streams[device].push_back(s);
}
static bool event_acquire(int device, cudaEvent_t* e) {
    ResourceCache& c = cache();
    {
        std::lock_guard<std::mutex> lk(c.mu);
        auto& v = c.events[device];
        if (!v.empty()) { *e = v.back(); v.pop_back(); return true; }
    }
    CUDA_TRY(cudaEventCreate(e));
    return true;
}
static void event_release(int device, cudaEvent_t e) {
    if (!e) return;
    ResourceCache& c = cache();
    std::lock_guard<std::mutex> lk(c.mu);
    c.events[device].push_back(e);
}
static bool device_info(int device, DeviceInfo* out) {
    ResourceCache& c = cache();
    {
        std::lock_guard<std::mutex> lk(c.mu);
        if (c.info[device].known) { *out = c.info[device]; return true; }
    }
    DeviceInfo di;
    CUDA_TRY(cudaDeviceGetAttribute(&di.numSMs, cudaDevAttrMultiProcessorCount, device));
    CUDA_TRY(cudaDeviceGetAttribute(&di.smemLimit, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    CUDA_TRY(cudaDeviceGetAttribute(&di.major, cudaDevAttrComputeCapabilityMajor, device));
    di.known = true;
    std::lock_guard<std::mutex> lk(c.mu);
    c.info[device] = di;
    *out = di;
    return true;
}

// Copy with non-temporal stores: the staged bytes go to memory instead of staying dirty in the writing core's
// cache, where the copy engine would have to fetch them line by line through the coherence fabric.
static void stream_copy(uint8_t* dst, const uint8_t* src, size_t n) {
    if (n < 256) { memcpy(dst, src, n); return; }
    const size_t head = (16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15;
    memcpy(dst, src, head);
    dst += head; src += head; n -= head;
    size_t i = 0;
    for (; i + 64 <= n; i += 64) {
        const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i));
        const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 16));
        const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 32));
        const __m128i d = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 48));
        _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i), a);
        _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 16), b);
        _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 32), c);
        _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 48), d);
    }
    memcpy(dst + i, src + i, n - i);
}

// ------------------------------------------------------------------ host worker pool
// Packing a database is a host-side gather of every sequence into pinned memory; on the drop-in path it is paid
// per call and is memory-bound on one core, so it is spread over a few persistent threads (the reference arm of
// the benchmark uses every host thread as well).  The caller takes part in the work; pool threads never touch CUDA.
namespace {
class HostPool {
public:
    static HostPool& get() { static HostPool* p = new HostPool(); return *p; }  // leaked on purpose, like the cache
    int width() const { return (int)workers_.size() + 1; }
    // Runs fn(part) for part in [0, parts); done(part) is called on the calling thread, in part order, as soon as
    // parts 0..part have all finished.  Several callers may have jobs in the pool at once (the slices and devices of
    // one drop-in call stage, publish and write records concurrently): workers take parts from whichever job has some
    // left, and every caller works on its own job until it is through.
    void run(int parts, const std::function<void(int)>& fn, const std::function<void(int)>& done) {
        if (workers_.empty() || parts <= 1) {
            for (int k = 0; k < parts; k++) { fn(k); done(k); }
            return;
        }
        Job job;
        job.fn = &fn; job.parts = parts;
        std::vector<std::atomic<char>> finished((size_t)parts);
        for (auto& f : finished) f.store(0, std::memory_order_relaxed);
        job.finished = finished.data();
        {
            std::lock_guard<std::mutex> lk(mu_);
            jobs_.push_back(&job);
        }
        cv_.notify_all();
        int reported = 0;
        auto report = [&]() {
            while (reported < parts && finished[reported].load(std::memory_order_acquire)) done(reported++);
        };
        for (;;) {
            const int k = job.next.fetch_add(1);
            if (k >= parts) break;
            fn(k);
            finished[k].store(1, std::memory_order_release);
            report();
        }
        while (reported < parts) { report(); std::this_thread::yield(); }
        // the job leaves the list; workers that still hold it (between taking a part number and finding none left) let go first
        std::unique_lock<std::mutex> lk(mu_);
        jobs_.erase(std::find(jobs_.begin(), jobs_.end(), &job));
        idle_.wait(lk, [&] { return job.holders == 0; });
    }

private:
    struct Job {
        const std::function<void(int)>* fn = nullptr;
        std::atomic<char>* finished = nullptr;
        int parts = 0, holders = 0;  // holders: workers inside this job (guarded by mu_)
        std::atomic<int> next{0};
    };
    HostPool() {
        int width = std::min((int)std::thread::hardware_concurrency(), 16);
        if (const char* e = getenv("OPAL_B200_HOST_THREADS")) width = std::max(1, std::min(atoi(e), 64));
        const int n = std::max(0, width - 1);
        for (int i = 0; i < n; i++) workers_.emplace_back([this] { loop(); });
        for (auto& t : workers_) t.detach();
    }
    void loop() {
        size_t turn = 0;
        for (;;) {
            Job* job = nullptr;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] {
                    for (size_t i = 0; i < jobs_.size(); i++) {  // round-robin over the jobs that still have parts to hand out
                        Job* j = jobs_[(turn + i) % jobs_.size()];
                        if (j->next.load(std::memory_order_relaxed) < j->parts) { job = j; turn += i + 1; return true; }
                    }
                    return false;
                });
                job->holders++;
            }
            for (;;) {
                const int k = job->next.fetch_add(1);
                if (k >= job->parts) break;
                (*job->fn)(k);
                job->finished[k].store(1, std::memory_order_release);
            }
            {
                std::lock_guard<std::mutex> lk(mu_);
                job->holders--;
            }
            idle_.notify_all();
        }
    }
    std::vector<std::thread> workers_;
    std::mutex mu_;
    std::condition_variable cv_, idle_;
    std::vector<Job*> jobs_;
};
}  // namespace

void parallel_for(long long n, long long grain, const std::function<void(long long, long long)>& body) {
    HostPool& pool = HostPool::get();
    const int parts = (int)std::max<long long>(1, std::min<long long>(n / std::max<long long>(grain, 1), pool.width()));
    if (parts <= 1) { body(0, n); return; }
    pool.run(parts, [&](int k) { body(n * k / parts, n * (k + 1) / parts); }, [](int) {});
}

// ------------------------------------------------------------------ layouts
// Everything about a database that depends only on its sequence LENGTHS -- the length sort, the index maps, the offsets
// of the plain / paired / folded streams, the planner's prefix sums -- is computed once and remembered, keyed by the
// length array itself (compared in full: a few MB, ~0.1 ms): the drop-in opalSearchDatabase packs its database on
// every call, and callers run query after query against the same sequences (reference test/perf:15-24).  The residues
// are NOT cached: they are staged and uploaded on every call, as the signature demands.
void TaskLens::build() {
    for (int sh = 0; sh < 6; sh++) {
        const size_t g = (size_t)1 << sh, cnt = (len.size() + g - 1) / g;
        prefix[sh].assign(cnt + 1, 0.0);
        for (size_t k = 0; k < cnt; k++) prefix[sh][k + 1] = prefix[sh][k] + len[k * g];
    }
}

const TaskLens& Layout::pair_lens() const {
    std::call_once(pairOnce_, [this] {
        const int m = (nonEmpty + 1) / 2;
        pairLens_.len.resize((size_t)m);
        for (int k = 0; k < m; k++) pairLens_.len[k] = sortedLen[2 * (size_t)k];
        pairLens_.build();
    });
    return pairLens_;
}
const TaskLens& Layout::target_lens() const {
    std::call_once(targetOnce_, [this] {
        targetLens_.len.assign(sortedLen.begin(), sortedLen.begin() + nonEmpty);
        targetLens_.build();
    });
    return targetLens_;
}

// Parts of a database for several devices and / or pipelined slices.  Devices: the sorted order is dealt round-robin
// (equal residue count, equal length mix -- every device's longest target is about as long as the others').  Slices
// of one device: slice 0 holds ITS longest sequences, a tenth of its residues -- the targets whose single-warp sweeps
// last longest are uploaded and started first, and a small first slice means the kernels start early; the other
// slices are runs of the remaining sequences in CALLER order with equal residue counts, so that staging them reads
// the caller's memory sequentially (a slice cut from the sorted order is a gather of every k-th sequence: measured
// 26 GB/s on 16 threads against 65 GB/s for runs) and none of them has a long tail of its own.
std::shared_ptr<const std::vector<std::vector<int>>> Layout::parts(int devices, int perDevice) const {
    std::lock_guard<std::mutex> lk(partsMu_);
    for (const auto& e : parts_)
        if (e.first.first == devices && e.first.second == perDevice) return e.second;
    auto out = std::make_shared<std::vector<std::vector<int>>>((size_t)devices * perDevice);
    const int n = (int)order.size();
    for (int d = 0; d < devices; d++) {
        std::vector<int>* mine = &(*out)[(size_t)d * perDevice];
        long long total = 0;
        for (int p = d; p < n; p += devices) total += sortedLen[p];
        if (perDevice == 1) {
            for (int p = d; p < n; p += devices) mine[0].push_back(order[p]);
            std::sort(mine[0].begin(), mine[0].end());  // ascending caller index: sequential reads of the caller's memory
            continue;
        }
        std::vector<int> rest;
        long long head = 0;
        for (int p = d; p < n; p += devices) {
            if (head * 10 < total) { mine[0].push_back(order[p]); head += sortedLen[p]; }
            else rest.push_back(order[p]);
        }
        std::sort(mine[0].begin(), mine[0].end());
        std::sort(rest.begin(), rest.end());
        const long long tail = total - head;
        long long seen = 0;
        for (int i : rest) {
            const int k = 1 + (int)std::min<long long>(perDevice - 2, tail > 0 ? seen * (perDevice - 1) / tail : 0);
            mine[k].push_back(i);
            seen += lens[i];
        }
    }
    parts_.push_back({{devices, perDevice}, out});
    return out;
}

namespace {
std::mutex g_layoutMu;
std::vector<std::shared_ptr<Layout>> g_layouts;  // most recently used last
constexpr size_t kMaxLayouts = 12, kMaxLayoutBytes = 384u << 20;

std::shared_ptr<Layout> find_layout(const int* lens, int n) {
    std::lock_guard<std::mutex> lk(g_layoutMu);
    for (size_t k = g_layouts.size(); k-- > 0;) {
        const std::shared_ptr<Layout>& l = g_layouts[k];
        if ((int)l->lens.size() == n && (n == 0 || memcmp(l->lens.data(), lens, sizeof(int) * (size_t)n) == 0)) {
            std::shared_ptr<Layout> hit = l;
            g_layouts.erase(g_layouts.begin() + (long)k);
            g_layouts.push_back(hit);
            return hit;
        }
    }
    return nullptr;
}
void remember_layout(const std::shared_ptr<Layout>& l) {
    std::lock_guard<std::mutex> lk(g_layoutMu);
    g_layouts.push_back(l);
    size_t bytes = 0;
    for (const auto& e : g_layouts) bytes += 44 * e->lens.size();
    while (g_layouts.size() > kMaxLayouts || (bytes > kMaxLayoutBytes && g_layouts.size() > 1)) {
        bytes -= 44 * g_layouts.front()->lens.size();
        g_layouts.erase(g_layouts.begin());
    }
}
}  // namespace
void trim_layouts() {
    std::lock_guard<std::mutex> lk(g_layoutMu);
    g_layouts.clear();
}

// Thread stride in the profile: a multiple of 4 words (16-byte aligned LDS.128) with an odd number of
// 16-byte units, so the 8 lanes of a quarter-warp hit 8 different bank groups whatever their residues are.
static int rpad_of(int R) { const int r4 = (R + 3) / 4; return 4 * ((r4 % 2 == 0) ? r4 + 1 : r4); }

// Picks (G, R, passes, warps per scheduler partition) for a query of Q rows over `taskLens` (one entry
// per task, longest first) on `numSMs` SMs, and returns the estimated cycles in *estCycles.
//
// Timing model (cycles): the time of one wavefront step of a warp that shares its scheduler partition with k - 1
// others, measured on B200 with tools/steptime_probe.py (kStepCycles below; the integer pipe retires one packed
// DPX instruction per 2 cycles per partition and a cell pair costs ~5.5 of them, 11 cycles per row ideal -- one
// warp alone is latency-bound far above that, three warps together come within 40 %).  Two bounds:
//   throughput:  sum over warp-tasks of steps * stepTime / (partitions * k)
//   tail:        the longest target's steps * stepTime  (it cannot be split across warps)
// Small databases with a long tail (BASELINE configs[1]) are tail-bound and want G = 32 and k = 1;
// large ones are throughput-bound and want k = 3.
// kStepCycles[flavor class][k - 1][i] = cycles per step at R = kStepR[i]; class 0 = SW score + end, 1 = SW score,
// 2 = NW / HW / OV.  Linear in between.
static const int kStepR[7] = {4, 8, 9, 12, 17, 24, 33};
static const double kStepCycles[3][3][7] = {
    {{193, 260, 276, 287, 366, 479, 608}, {243, 349, 382, 418, 570, 745, 925}, {301, 468, 520, 574, 782, 1042, 1320}},
    {{183, 203, 236, 270, 313, 418, 565}, {224, 281, 314, 399, 473, 620, 846}, {262, 382, 408, 539, 672, 896, 1193}},
    {{289, 342, 347, 382, 425, 491, 598}, {333, 407, 423, 492, 605, 713, 918}, {390, 470, 514, 608, 762, 921, 1240}},
};
static double step_cycles_lockstep(int flavorClass, int k, int R) {
    const double* t = kStepCycles[flavorClass][std::min(std::max(k, 1), 3) - 1];
    if (R <= kStepR[0]) return t[0] * (0.5 + 0.5 * R / kStepR[0]);
    for (int i = 1; i < 7; i++)
        if (R <= kStepR[i]) return t[i - 1] + (t[i] - t[i - 1]) * (R - kStepR[i - 1]) / (double)(kStepR[i] - kStepR[i - 1]);
    return t[6] * R / kStepR[6];
}
// The table was taken with all warps of a partition in lockstep (equal tasks started together), the worst case for
// pipe contention; with tasks of mixed lengths the same probe measures less, by a ratio that depends on the strip
// height (SW score + end at R = 9 / 17 / 33: k = 1: 0.92 / 0.90 / 0.91, k = 2: 0.97 / 0.92 / 0.97, k = 3: 0.98 throughout).
static double step_cycles(int flavorClass, int k, int R) {
    static const double ratio[3][3] = {{0.917, 0.904, 0.908}, {0.966, 0.923, 0.965}, {0.975, 0.980, 0.983}};
    const double* r = ratio[std::min(std::max(k, 1), 3) - 1];
    const double f = R <= 9 ? r[0] : R <= 17 ? r[0] + (r[1] - r[0]) * (R - 9) / 8.0 : R <= 33 ? r[1] + (r[2] - r[1]) * (R - 17) / 16.0 : r[2];
    return f * step_cycles_lockstep(flavorClass, k, R);
}
// Resident warps per scheduler partition the kernels are compiled for (launch_bound_for in search_kernel.cuh).
// (The 32-bit NW/HW/OV kernels at the tallest strips exist only uncapped, for two.)
static int max_warps_per_partition(int mode, int R, int lanes) {
    return (lanes == 1 && mode != kModeSW) ? launch_bound_for(kFlavorGlobal, R) / 128 : 3;
}

static thread_local int t_forceK = 0, t_forceG = 0, t_forceR = 0;  // development override (OPAL_B200_SPLIT): geometry of the bulk group
// Several searches in flight (search_batch): the tail of one search overlaps the bulk of the next, so a plan is priced
// mostly by the SM time it takes, not by when its last task ends.  Measured on BASELINE configs[1], 32 queries with
// three in flight: plans with three warps per partition give 3975 - 4010 GCUPS, the single-search optimum 3770.
static thread_local bool t_overlapped = false;
void set_thread_overlapped(bool on) { t_overlapped = on; }

static bool pick_geometry(int Q, int A, int lanes, const TaskLens& tl, size_t lo, size_t hi, int smemLimit, int numSMs, int mode,
                          bool latencyClass, int flavorClass, Geometry* out, double* estCycles, bool folded = false) {
    const int planes = lanes == 2 ? 2 : 1;
    const auto& tables = kernel_tables();
    double bestCost = 1e300;
    bool found = false;
    const double tasks = (double)(hi - lo);
    const double maxLen = hi > lo ? tl.len[lo] : 0;
    // The (strip height, group size) pairs worth pricing depend only on the query and the alphabet, not on the task
    // range: they are filtered once and remembered (a plan prices some ninety task ranges, on the path of every
    // drop-in call).
    struct Viable { int Q = -1, A = 0, lanes = 0, smemLimit = 0, minPasses = 0; std::vector<std::pair<int, int>> list; };
    static thread_local Viable memo[3];
    Viable& viable = memo[latencyClass ? (folded ? 2 : 1) : 0];
    int minPasses = 1 << 20;  // fewest passes any geometry that fits shared memory needs
    if (viable.Q == Q && viable.A == A && viable.lanes == lanes && viable.smemLimit == smemLimit) {
        minPasses = viable.minPasses;
    } else {
        for (size_t ti = 0; ti < tables.size(); ti++)
            for (int G = latencyClass ? 32 : 1; G <= 32; G *= 2) {
                const int rows = (folded ? 2 : 1) * G * tables[ti].R;
                const size_t smem = (size_t)planes * (A + 1) * ((G * rpad_of(tables[ti].R) + 31) / 32 * 32) * 4;
                if (smem <= (size_t)smemLimit) minPasses = std::min(minPasses, (Q + rows - 1) / rows);
            }
        viable.Q = -1;  // list rebuilt below
    }
    auto worth_pricing = [&](size_t ti, int G) -> bool {
        const int R = tables[ti].R;
        const size_t smem = (size_t)planes * (A + 1) * ((G * rpad_of(R) + 31) / 32 * 32) * 4;
        if (smem > (size_t)smemLimit) return false;
        const int rows = (folded ? 2 : 1) * G * R;
        const int passes = (Q + rows - 1) / rows;
        if (folded && passes > 1) return false;
        // more than a third of the swept rows padding: never the best choice unless nothing smaller exists
        if ((long long)passes * rows * 3 > (long long)Q * 4 + 96 && !(G == (latencyClass ? 32 : 1) && ti == 0)) return false;
        // more passes than the tallest geometry needs (one more for queries that take several anyway): the same
        // cells plus boundary rows through HBM and further launches
        if (passes > minPasses + (minPasses > 1 ? 1 + minPasses / 2 : 0)) return false;
        return true;
    };
    if (viable.Q != Q) {
        viable.list.clear();
        for (size_t ti = 0; ti < tables.size(); ti++)
            for (int G = latencyClass ? 32 : 1; G <= 32; G *= 2)
                if (worth_pricing(ti, G)) viable.list.push_back({(int)ti, G});
        viable.Q = Q; viable.A = A; viable.lanes = lanes; viable.smemLimit = smemLimit; viable.minPasses = minPasses;
    }
    auto consider = [&](size_t ti, int G, int k, bool forced) {
        const int R = tables[ti].R;
        if (!latencyClass && ((t_forceK > 0 && k != t_forceK) || (t_forceG > 0 && G != t_forceG) || (t_forceR > 0 && R != t_forceR))) return;
        const int Rpad = rpad_of(R);
        const int rowStride = (G * Rpad + 31) / 32 * 32;
        const size_t smem = (size_t)planes * (A + 1) * rowStride * 4;
        if (smem > (size_t)smemLimit) return;
        const int rows = (folded ? 2 : 1) * G * R;  // a folded task has its second 32 R rows in the high half-words
        const int passes = (Q + rows - 1) / rows;
        if (folded && passes > 1) return;
        if (folded && mode != kModeSW && !single_event_compare(R)) return;  // tall NW / HW / OV strips are compiled without folding
        (void)forced;
        const int groupsPerWarp = 32 / G;
        if (lo % groupsPerWarp) return;  // a warp takes groupsPerWarp consecutive tasks (and TaskLens::strided wants it so)
        // a warp-task lasts as long as its longest group: every groupsPerWarp-th task of the sorted list
        int sh = 0;
        while ((1 << sh) < groupsPerWarp) sh++;
        double warpTasks = 1;
        double warpSteps = tl.strided(sh, lo, hi, &warpTasks);
        warpSteps += warpTasks * (G - 1 + (folded ? kFoldLag : 0));
        warpTasks = std::max(1.0, warpTasks);
        // with fewer warp-tasks than resident warps the partitions are not shared k ways
        const int kEff = (int)std::max(1.0, std::min((double)k, std::ceil(warpTasks / (numSMs * 4.0))));
        const double stepTime = step_cycles(flavorClass, kEff, R);
        const double warpsBusy = std::min((double)numSMs * 4 * k, warpTasks);
        double throughput = warpSteps * stepTime / warpsBusy;
        // Two warps share a partition only while both have work: with few tasks per warp a large part of the run is
        // spent with single warps finishing alone at the (slower) one-warp rate.  Measured on 10k-sequence databases:
        // +40 % at 2.2 tasks per warp, nothing from about 3.5 tasks per warp on.
        if (k >= 2) {
            const double tasksPerWarp = warpTasks / ((double)numSMs * 4 * k);
            if (tasksPerWarp < 3.5) throughput *= 1.0 + 0.3 * (3.5 - std::max(tasksPerWarp, 1.0));
        }
        // (Measured on BASELINE configs[1]: with three warps on its partition the longest task advances at ~630 cycles
        // per step of R = 17, with two at ~540 -- no faster than the table says, although it sits on the oldest warp.)
        // A launch takes the longer of the two plus a little of the other (fitted on forced splits of BASELINE
        // configs[1], tools/split_sweep.sh: within 6 % of the measured time for latency classes of 8 - 128 targets).
        const double tail = (t_overlapped ? 0.6 : 0.95) * (maxLen + G - 1 + (folded ? kFoldLag : 0)) * stepTime;
        // every further pass is a kernel of its own (drain, launch, boundary rows through HBM): measured ~4 % each
        double cost = passes * (std::max(throughput, tail) + 0.05 * std::min(throughput, tail) + 30000.0) *
                      (1.0 + 0.04 * (passes - 1));
        // With searches overlapping, three warps per partition gain more than their steady-state step time says (the
        // SMs a search leaves early are taken by the next one): measured +7 - 9 % over two, against +3 % priced above.
        if (t_overlapped && k >= 3) cost *= 0.94;
        if (forced || cost < bestCost) {
            bestCost = cost;
            found = true;
            out->G = G; out->R = R; out->tableIndex = (int)ti; out->passes = passes; out->Rpad = Rpad;
            out->rowStride = rowStride; out->smemBytes = smem; out->warpsPerPartition = k;
            out->padTop = (mode == kModeNW) ? 0 : passes * rows - Q;
            out->folded = folded;
        }
    };
    for (const auto& tg : viable.list)
        for (int k = 1; k <= (latencyClass ? 1 : max_warps_per_partition(mode, tables[tg.first].R, lanes)); k++)
            consider((size_t)tg.first, tg.second, k, false);
    // Development override: OPAL_B200_GEOMETRY="G,R,k" forces a geometry (ignored when it does not fit).
    if (const char* env = getenv("OPAL_B200_GEOMETRY")) {
        int G = 0, R = 0, k = 0;
        if (!latencyClass && sscanf(env, "%d,%d,%d", &G, &R, &k) == 3 && G >= 1 && G <= 32 && (G & (G - 1)) == 0 && k >= 1 &&
            k <= max_warps_per_partition(mode, R, lanes))
            for (size_t ti = 0; ti < tables.size(); ti++)
                if (tables[ti].R == R) consider(ti, G, k, true);
    }
    if (!found) set_error("alphabet too large for the shared-memory query profile");
    if (estCycles) *estCycles = bestCost;
    return found;
}

// Work is dealt by entries of the paired stream (pads included), so that a 35 000-residue target costs what 35 000
// residues cost and not one warp's walk along it.  A block covers kPackEntriesPerBlock consecutive entries: its first
// thread finds the pair of the first entry by bisection -- a chain of dependent loads that costs more than everything
// else a block of 256 entries would do, hence the larger blocks (61 -> 20 us for the 4.4 M entries of BASELINE
// configs[1]) -- and every thread walks forward from there, entry by entry in steps of the block size.
constexpr int kPackEntriesPerBlock = 4096;
static __global__ void pack_pairs_kernel(const uint8_t* residues, const long long* offsets, const int* lengths, int numTargets,
                                  const long long* pairOffsets, int numPairs, long long entries, uint16_t* pairStream, int* maxCode) {
    __shared__ int basePair, blockMax;
    const long long e0 = (long long)blockIdx.x * kPackEntriesPerBlock;
    if (threadIdx.x == 0) {
        blockMax = 0;
        int lo = 0, hi = numPairs;  // last pair whose first column is at or before e0 (entries before pair 0 are padding)
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (pairOffsets[mid] <= e0) lo = mid; else hi = mid;
        }
        basePair = lo;
    }
    __syncthreads();
    int p = basePair;
    uint32_t mx = 0;
    for (int it = 0; it < kPackEntriesPerBlock / 256; it++) {
        const long long e = e0 + it * 256 + threadIdx.x;
        if (e >= entries) break;
        uint32_t word = 0;
        if (numPairs > 0) {
            while (p + 1 < numPairs && pairOffsets[p + 1] <= e) p++;
            const long long c = e - pairOffsets[p];
            const int a = 2 * p, b = 2 * p + 1;
            if (c >= 0 && c < lengths[a]) {
                const uint32_t r0 = (uint32_t)residues[offsets[a] + c] + 1u;
                word = r0 & 0xffu;
                mx = max(mx, r0);  // from the raw residue: code 255 (+ 1) does not fit the byte and is searched at 32 bits
                if (b < numTargets && c < lengths[b]) {
                    const uint32_t r1 = (uint32_t)residues[offsets[b] + c] + 1u;
                    word |= (r1 & 0xffu) << 8;
                    mx = max(mx, r1);
                }
            }
        }
        pairStream[e] = (uint16_t)word;
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    if ((threadIdx.x & 31) == 0 && mx > 0) atomicMax(&blockMax, (int)mx);
    __syncthreads();
    // largest residue code seen: one global atomic per block, and only while it still raises the value
    if (threadIdx.x == 0 && blockMax > 0 && blockMax - 1 > *(volatile int*)maxCode) atomicMax(maxCode, blockMax - 1);
}

// Folded stream of the longest targets (see SearchParams::folded): entry c of target p, c in [0, T + 32), is
// (res[c] + 1) | (res[c - 32] + 1) << 8 with 0 where the index falls outside the target; 32 zero entries before
// the first target and after every target.  One thread per entry; its target (one of at most kFoldTargets) by bisection.
static __global__ void pack_folded_kernel(const uint8_t* residues, const long long* offsets, const int* lengths, const long long* foldOffsets,
                                          int numFold, long long entries, uint16_t* foldStream) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= entries) return;
    int p = 0, hi = numFold;  // last target whose first column is at or before e
    while (hi - p > 1) {
        const int mid = (p + hi) >> 1;
        if (foldOffsets[mid] <= e) p = mid; else hi = mid;
    }
    const long long c = e - foldOffsets[p];
    const int T = lengths[p];
    uint32_t word = 0;
    if (c >= 0 && c < T + kFoldLag) {
        if (c < T) word = (uint32_t)residues[offsets[p] + c] + 1u;
        if (c >= kFoldLag) word |= ((uint32_t)residues[offsets[p] + c - kFoldLag] + 1u) << 8;
    }
    foldStream[e] = (uint16_t)word;
}

// The layout of a database: found in the cache or built (and, for scattered databases, remembered).  `order` is the
// caller's permutation of a packed database (NULL: identity); NULL + error text on invalid lengths.
std::shared_ptr<const Layout> layout_for(const int* lens, const int* order, int n, bool packed, bool* cachedOut) {
    std::shared_ptr<Layout> lay = packed ? nullptr : find_layout(lens, n);
    if (cachedOut) *cachedOut = lay != nullptr;
    if (lay) return lay;
    lay = std::make_shared<Layout>();
    Layout& L = *lay;
    int maxLen = 0;
    for (int i = 0; i < n; i++) {
        if (lens[i] < 0) { set_error("negative sequence length"); return nullptr; }
        maxLen = std::max(maxLen, lens[i]);
    }
    L.lens.assign(lens, lens + n);
    L.order.resize(n);
    L.pos.resize(n);
    if (packed) {
        for (int p = 0; p < n; p++) L.order[p] = order ? order[p] : p;
    } else if (maxLen <= (1 << 22) && n >= (1 << 17) && (long long)HostPool::get().width() * (maxLen + 2) <= (16LL << 20)) {
        // large database: counting sort with one histogram per host thread (contiguous index ranges, so the
        // result is still stable in caller order) -- the scatter is a cache miss per sequence
        const int W = HostPool::get().width(), B = maxLen + 1;
        std::vector<int> hist((size_t)W * B, 0);
        HostPool::get().run(W, [&](int k) {
            int* h = hist.data() + (size_t)k * B;
            for (long long i = (long long)n * k / W, e = (long long)n * (k + 1) / W; i < e; i++) h[maxLen - lens[i]]++;
        }, [](int) {});
        int at = 0;
        for (int b = 0; b < B; b++)
            for (int k = 0; k < W; k++) { const int c = hist[(size_t)k * B + b]; hist[(size_t)k * B + b] = at; at += c; }
        HostPool::get().run(W, [&](int k) {
            int* h = hist.data() + (size_t)k * B;
            for (long long i = (long long)n * k / W, e = (long long)n * (k + 1) / W; i < e; i++) L.order[h[maxLen - lens[i]]++] = (int)i;
        }, [](int) {});
    } else if (maxLen <= (1 << 22)) {
        std::vector<int> start(maxLen + 2, 0);
        for (int i = 0; i < n; i++) start[maxLen - lens[i] + 1]++;
        for (int k = 1; k <= maxLen + 1; k++) start[k] += start[k - 1];
        for (int i = 0; i < n; i++) L.order[start[maxLen - lens[i]]++] = i;
    } else {
        for (int i = 0; i < n; i++) L.order[i] = i;
        std::stable_sort(L.order.begin(), L.order.end(), [&](int a, int b) { return lens[a] > lens[b]; });
    }
    // Residues are stored in the order they are copied in -- caller order for scattered sequences (sequential
    // reads of the caller's memory, runs of adjacent sequences merge into one memcpy), sorted order for a
    // packed database -- and offsets[p] says where sorted position p lives.  Nothing needs the sorted
    // sequences to be adjacent: the 16-bit kernels stream the paired layout built on the device below.
    L.copyOff.resize((size_t)n + 1);
    long long sum = 0;
    for (int i = 0; i < n; i++) { L.copyOff[i] = sum; sum += lens[i]; }
    L.copyOff[n] = sum;
    L.total = sum;
    L.sortedLen.resize(n);
    L.offsets.resize((size_t)n + 1);
    parallel_for(n, 65536, [&](long long lo, long long hi) {
        for (long long p = lo; p < hi; p++) {
            const int i = L.order[p];
            L.pos[i] = (int)p;
            L.sortedLen[p] = packed ? lens[p] : lens[i];
            L.offsets[p] = packed ? L.copyOff[p] : L.copyOff[i];
        }
    });
    L.offsets[n] = sum;
    L.nonEmpty = n;
    while (L.nonEmpty > 0 && L.sortedLen[L.nonEmpty - 1] == 0) L.nonEmpty--;
    // paired stream: [32 zeros][pair 0 columns][32 zeros][pair 1 ...]; the longest targets also get a folded
    // stream (an even number of them: the bulk keeps whole pairs)
    L.numPairs = (n + 1) / 2;
    L.numFold = getenv("OPAL_B200_NO_FOLD") ? 0 : std::min(n & ~1, kFoldTargets);
    while (L.numFold > 0 && L.sortedLen[L.numFold - 1] < kFoldMinLength) L.numFold -= 2;
    L.numFold = std::max(L.numFold, 0);
    L.pairOff.resize((size_t)std::max(L.numPairs, 1));
    L.foldOff.resize((size_t)std::max(L.numFold, 1));
    L.entries = 32;
    L.pairOff[0] = 32;
    for (int p = 0; p < L.numPairs; p++) { L.pairOff[p] = L.entries; L.entries += L.sortedLen[2 * (size_t)p] + 32; }
    L.entries += 64;
    L.foldEntries = 32;
    L.foldOff[0] = 32;
    for (int p = 0; p < L.numFold; p++) { L.foldOff[p] = L.foldEntries; L.foldEntries += L.sortedLen[p] + kFoldLag + 32; }
    L.foldEntries += 64;
    if (!packed) remember_layout(lay);
    return lay;
}

// ------------------------------------------------------------------ device-side selection (search_topk)
// Sorted positions in [0, to) whose 16-bit result is "re-run me" (or missing): the ladder's hand-over list, gathered on
// the device so that only the list travels to the host, not every score.
static __global__ void collect_flagged_kernel(const int* score, int to, int* outList, int* outCount) {
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < to; p += gridDim.x * blockDim.x) {
        const int sc = score[p];
        if (sc == kScoreOverflow || sc == kScoreNone) outList[atomicAdd(outCount, 1)] = p;
    }
}

// Boundary rows of a chained launch start out "not written yet" (search_kernel.cuh: kChainEmpty).
static __global__ void fill_words_kernel(uint32_t* p, size_t n, uint32_t v) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

// Zero-length targets (the tail of the length-sorted order) get their defined result without a sweep.
static __global__ void fill_empty_kernel(int* score, int* endQ, int* endT, int from, int to, int sc, int eq, int et) {
    for (int p = from + blockIdx.x * blockDim.x + threadIdx.x; p < to; p += gridDim.x * blockDim.x) { score[p] = sc; endQ[p] = eq; endT[p] = et; }
}

// The k best of n results under the key (score descending, caller index ascending): radix select over the 64-bit key
// (score biased to unsigned | ~caller index) -- eight passes of one 1024-thread block, a 256-bin shared-memory
// histogram each, narrow the k-th largest key down byte by byte (keys are unique, so exactly k results lie at or above
// it); a ninth pass writes those k records {caller index, score, endQ, endT}, unordered.  All of it reads the score
// array where the search kernels left it: 8 n bytes per pass out of L2.
__device__ __forceinline__ unsigned long long topk_key(int score, int callerIndex) {
    return ((unsigned long long)((unsigned)score ^ 0x80000000u) << 32) | (unsigned long long)(0xffffffffu - (unsigned)callerIndex);
}
static __global__ void __launch_bounds__(1024) topk_select_kernel(const int* score, const int* endQ, const int* endT, const int* order,
                                                                  int n, int k, int wantEnd, int4* records) {
    __shared__ unsigned hist[256];
    __shared__ unsigned long long prefix;  // the bytes of the k-th largest key decided so far (high bytes)
    __shared__ unsigned remaining, written;
    if (threadIdx.x == 0) { prefix = 0; remaining = (unsigned)k; written = 0; }
    for (int byte = 7; byte >= 0; byte--) {
        if (threadIdx.x < 256) hist[threadIdx.x] = 0;
        __syncthreads();
        const unsigned long long pre = prefix;
        const int shift = 8 * byte;
        for (int p = threadIdx.x; p < n; p += blockDim.x) {
            const unsigned long long key = topk_key(score[p], order[p]);
            if (byte == 7 || (key >> (shift + 8)) == pre) atomicAdd(&hist[(unsigned)(key >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned need = remaining, b = 255;
            for (;; b--) {  // buckets from the top: the one that holds the k-th largest key
                if (hist[b] >= need || b == 0) break;
                need -= hist[b];
            }
            remaining = need;
            prefix = (pre << 8) | b;
        }
        __syncthreads();
    }
    const unsigned long long threshold = prefix;
    for (int p = threadIdx.x; p < n; p += blockDim.x) {
        if (topk_key(score[p], order[p]) >= threshold) {
            const unsigned slot = atomicAdd(&written, 1u);
            if (slot < (unsigned)k) records[slot] = make_int4(order[p], score[p], wantEnd ? endQ[p] : 0x7fffffff, wantEnd ? endT[p] : 0x7fffffff);
        }
    }
}

// ------------------------------------------------------------------ DeviceDb
DeviceDb* DeviceDb::create(unsigned char* const* db, int n, const int* lens, int device) {
    return build(db, nullptr, lens, nullptr, n, device);
}

DeviceDb* DeviceDb::create_sorted(const unsigned char* residues, const int* sortedLens, const int* order, int n, int device) {
    for (int p = 1; p < n; p++)
        if (sortedLens[p] > sortedLens[p - 1]) { set_error("packed database is not sorted longest first"); return nullptr; }
    if (order) {  // must be a permutation of 0..n-1
        std::vector<char> seen((size_t)std::max(n, 1), 0);
        for (int p = 0; p < n; p++) {
            if (order[p] < 0 || order[p] >= n || seen[order[p]]) { set_error("packed database: order[] is not a permutation"); return nullptr; }
            seen[order[p]] = 1;
        }
    }
    return build(nullptr, residues, sortedLens, order, n, device);
}

bool SearchContext::alloc_search_buffers() {
    if (!stream_acquire(db_.device, &stream_) || !event_acquire(db_.device, &evStart_) || !event_acquire(db_.device, &evStop_) ||
        !event_acquire(db_.device, &evFork_)) return false;
    // One device block [score | endQ | endT | task list (2n)] and one pinned block [score | endQ | endT]: every
    // stream operation has a fixed cost that exceeds the transfer itself at these sizes, so results come back in
    // a single copy.
    const size_t nWords = (size_t)std::max(db_.n, 1);
    if (!device_alloc(db_.device, (void**)&dResults_, sizeof(int) * 5 * nWords)) return false;
    // (the copy back covers entries no kernel writes -- skipped and zero-length targets, never read by the host)
    CUDA_TRY(cudaMemsetAsync(dResults_, 0xff, sizeof(int) * 3 * nWords, stream_));
    if (!pinned_alloc((void**)&hResults_, sizeof(int) * 3 * nWords)) return false;
    dScore_ = dResults_; dEndQ_ = dResults_ + nWords; dEndT_ = dResults_ + 2 * nWords; dTaskList_ = dResults_ + 3 * nWords;
    hScore_ = hResults_; hEndQ_ = hResults_ + nWords; hEndT_ = hResults_ + 2 * nWords;
    return true;
}

// Either `db` (n scattered sequences in caller order, lens[i]) or `packed` (contiguous, already sorted, lens[p],
// order[p]) is given.  Returns with the upload in flight on the database's stream (see ensure_uploaded()).
DeviceDb* DeviceDb::build(unsigned char* const* db, const unsigned char* packed, const int* lens, const int* order, int n, int device) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count || device >= kMaxDevices) {
        set_error("no usable CUDA device");
        return nullptr;
    }
    std::unique_ptr<DeviceDb> d(new DeviceDb());
    DbArrays& a = d->db_;
    a.device = device;
    a.n = n;
    auto ok = [&]() -> bool {
        CUDA_TRY(cudaSetDevice(device));
        DeviceInfo di;
        if (!device_info(device, &di)) return false;
        if (di.major < 10) { set_error("device is not sm_100 or newer"); return false; }
        a.numSMs = di.numSMs;
        a.smemLimit = di.smemLimit;
        PhaseTrace trace("build");
        trace.mark("setup");

        // ---- the layout: length sort (longest first, stable in caller order), index maps, stream offsets.  A pure
        // function of the length array: remembered between calls for scattered databases (see "layouts" above).
        bool cached = false;
        std::shared_ptr<const Layout> lay = layout_for(lens, order, n, packed != nullptr, &cached);
        if (!lay) return false;
        a.lay = lay;
        const long long total = lay->total;
        const std::vector<long long>& copyOff = lay->copyOff;
        a.totalResidues = total;
        trace.mark(cached ? "layout (cached)" : "layout");
        d->contexts_.push_back(std::make_unique<SearchContext>(a));
        SearchContext& ctx = *d->contexts_[0];
        if (!ctx.alloc_search_buffers()) return false;
        trace.mark("buffers");

        // ---- one pinned block [offsets | pair offsets | lengths | max code | residues], one upload.  (Every stream
        // operation costs tens of microseconds on its own here, far more than its share of a few MB, so the
        // database goes up in a single copy once the gather is complete.)  The residues part stays as the host
        // copy the alignment stage replays against.  Paired stream: [32 zeros][pair 0 columns][32 zeros][pair 1 ...].
        a.numPairs = lay->numPairs;
        a.numFold = lay->numFold;
        const size_t nOff = (size_t)n + 1, nPair = (size_t)std::max(a.numPairs, 1), nLen = (size_t)std::max(n, 1);
        const size_t nFold = (size_t)std::max(a.numFold, 1);
        const size_t indexBytes = (sizeof(long long) * (nOff + nPair + nFold) + sizeof(int) * (nLen + 1) + 255) / 256 * 256;
        const size_t bytes = indexBytes + (size_t)total + 64;
        if (!pinned_alloc((void**)&a.hBlock, bytes)) return false;
        if (!device_alloc(device, (void**)&a.dBlock, bytes)) return false;
        long long* hOff = reinterpret_cast<long long*>(a.hBlock);
        long long* hPair = hOff + nOff;
        long long* hFold = hPair + nPair;
        int* hLen = reinterpret_cast<int*>(hFold + nFold);
        a.hResidues = a.hBlock + indexBytes;
        a.dOffsets = reinterpret_cast<long long*>(a.dBlock);
        a.dPairOffsets = a.dOffsets + nOff;
        a.dFoldOffsets = a.dPairOffsets + nPair;
        a.dLengths = reinterpret_cast<int*>(a.dFoldOffsets + nFold);
        a.dMaxCode = a.dLengths + nLen;
        a.dResidues = a.dBlock + indexBytes;
        memcpy(hOff, lay->offsets.data(), sizeof(long long) * nOff);
        memcpy(hPair, lay->pairOff.data(), sizeof(long long) * nPair);
        memcpy(hFold, lay->foldOff.data(), sizeof(long long) * nFold);
        hLen[0] = 0;
        if (n > 0) memcpy(hLen, lay->sortedLen.data(), sizeof(int) * (size_t)n);
        hLen[nLen] = 0;  // max code, raised by the pairing kernel
        const long long entries = lay->entries, foldEntries = lay->foldEntries;
        uint8_t* staging = a.hResidues;
        memset(staging + total, 0, 64);
        // Parts of about equal residue count, cut at sequence boundaries; each is uploaded as soon as it and all
        // parts before it are staged, so the copy engine runs behind the host copy.  The copy engine reads lines
        // that sit dirty in ONE core's cache at full speed and several times slower when they are spread over the
        // caches of many cores (measured: 4.5 MB in 96 us after a 1-thread memcpy, 680 us after a 16-thread one).
        // So: long runs are copied with non-temporal stores (nothing stays in a cache) and may be split over a
        // few threads; scattered short sequences are copied by the calling thread alone unless the database is
        // far larger than the caches.
        HostPool& pool = HostPool::get();
        const bool oneRun = packed || (n > 0 && db[n - 1] + lens[n - 1] == db[0] + total);  // the usual arena-loaded database
        int stageThreads = total >= (16LL << 20) ? pool.width() : (oneRun && total >= (2 << 20) ? std::min(pool.width(), 8) : 1);
        if (const char* e = getenv("OPAL_B200_STAGE_THREADS")) stageThreads = std::max(1, std::min(atoi(e), pool.width()));
        const bool threaded = stageThreads > 1;
        const long long partBytes = total >= (64LL << 20) ? (8 << 20) : std::max<long long>(256 << 10, total / (2 * stageThreads));
        const int parts = (int)std::max<long long>(1, std::min<long long>(total / partBytes, 4096));
        std::vector<int> cut((size_t)parts + 1, n);
        cut[0] = 0;
        for (int k = 1; k < parts; k++) {
            const long long target = total * k / parts;
            cut[k] = std::max(cut[k - 1], (int)(std::lower_bound(copyOff.begin(), copyOff.begin() + n, target) - copyOff.begin()));
        }
        auto stage = [&](int k) {
            const int lo = cut[k], hi = cut[k + 1];
            if (lo >= hi) return;
            if (packed) { stream_copy(staging + copyOff[lo], packed + copyOff[lo], (size_t)(copyOff[hi] - copyOff[lo])); _mm_sfence(); return; }
            int j = lo;
            while (j < hi) {  // one copy per run of sequences that are adjacent in the caller's memory
                int e = j + 1;
                while (e < hi && db[e] == db[e - 1] + lens[e - 1]) e++;
                const long long len = copyOff[e] - copyOff[j];
                if (len >= 4096) stream_copy(staging + copyOff[j], db[j], (size_t)len);
                else if (len > 0) memcpy(staging + copyOff[j], db[j], (size_t)len);
                j = e;
            }
            _mm_sfence();
        };
        cudaError_t copyError = cudaSuccess;
        size_t uploaded = 0;  // bytes of the block already handed to the copy engine
        auto upload = [&](int k) {
            const size_t end = k == parts - 1 ? bytes : indexBytes + (size_t)copyOff[cut[k + 1]];
            for (size_t at = uploaded; at < end; at += (size_t)1 << 30) {
                const cudaError_t ce = cudaMemcpyAsync(a.dBlock + at, a.hBlock + at, std::min(end - at, (size_t)1 << 30), cudaMemcpyHostToDevice, ctx.stream_);
                if (ce != cudaSuccess) copyError = ce;
            }
            uploaded = std::max(uploaded, end);
        };
        trace.mark("index");
        ctx.uploadPending_ = true;
        if (trace.on) CUDA_TRY(cudaEventRecord(ctx.evStart_, ctx.stream_));
        if (threaded) pool.run(parts, stage, upload);
        else for (int k = 0; k < parts; k++) { stage(k); upload(k); }
        CUDA_TRY(copyError);
        trace.mark("stage+issue");
        if (trace.on) CUDA_TRY(cudaEventRecord(ctx.evFork_, ctx.stream_));
        if (!device_alloc(device, (void**)&a.dPairStream, sizeof(uint16_t) * (size_t)entries)) return false;
        if (!pinned_alloc((void**)&a.hMaxCode, sizeof(int))) return false;
        {
            const long long blocks = (entries + kPackEntriesPerBlock - 1) / kPackEntriesPerBlock;
            pack_pairs_kernel<<<(unsigned)blocks, 256, 0, ctx.stream_>>>(a.dResidues, a.dOffsets, a.dLengths, n, a.dPairOffsets,
                                                                         a.numPairs, entries, a.dPairStream, a.dMaxCode);
            CUDA_TRY(cudaGetLastError());
        }
        if (a.numFold > 0) {
            if (!device_alloc(device, (void**)&a.dFoldStream, sizeof(uint16_t) * (size_t)foldEntries)) return false;
            pack_folded_kernel<<<(unsigned)((foldEntries + 255) / 256), 256, 0, ctx.stream_>>>(a.dResidues, a.dOffsets, a.dLengths,
                                                                                            a.dFoldOffsets, a.numFold, foldEntries, a.dFoldStream);
            CUDA_TRY(cudaGetLastError());
        }
        CUDA_TRY(cudaMemcpyAsync(a.hMaxCode, a.dMaxCode, sizeof(int), cudaMemcpyDeviceToHost, ctx.stream_));
        if (trace.on) CUDA_TRY(cudaEventRecord(ctx.evStop_, ctx.stream_));
        trace.mark("issue");
        return true;  // upload still in flight: see ensure_uploaded()
    }();
    return ok ? d.release() : nullptr;
}

// Only the first context ever waits here: build() issues the upload on its stream, and in_flight() waits for the
// upload before it makes the others.
bool SearchContext::ensure_uploaded() {
    if (!uploadPending_) return true;
    CUDA_TRY(cudaSetDevice(db_.device));
    CUDA_TRY(cudaStreamSynchronize(stream_));
    if (getenv("OPAL_B200_TRACE")) {
        float copies = 0.f, pack = 0.f;
        if (cudaEventElapsedTime(&copies, evStart_, evFork_) == cudaSuccess && cudaEventElapsedTime(&pack, evFork_, evStop_) == cudaSuccess)
            fprintf(stderr, "[opal-b200] upload on the device: copies %.0f us, pairing %.0f us\n", copies * 1e3, pack * 1e3);
    }
    uploadPending_ = false;
    return true;
}

SearchContext::~SearchContext() {
    cudaSetDevice(db_.device);
    if (stream_) cudaStreamSynchronize(stream_);
    void* own[] = {dResults_, dArgs_, dBndH_, dBndF_};
    for (void* p : own) device_release(db_.device, p);
    for (void* b : chainScratch_) device_release(db_.device, b);
    pinned_release(hResults_); pinned_release(hArgs_);
    event_release(db_.device, evStart_); event_release(db_.device, evStop_); event_release(db_.device, evFork_);
    for (cudaStream_t st : auxStreams_) { cudaStreamSynchronize(st); stream_release(db_.device, st); }
    for (cudaEvent_t e : auxEvents_) event_release(db_.device, e);
    stream_release(db_.device, stream_);
}

DbArrays::~DbArrays() {
    cudaSetDevice(device);
    void* arrays[] = {dBlock, dPairStream, dFoldStream, dOrder};
    for (void* p : arrays) device_release(device, p);
    pinned_release(hBlock); pinned_release(hMaxCode);
}

bool SearchContext::ensure_boundary() {
    if (dBndH_) return true;
    const size_t bytes = 2 * sizeof(uint32_t) * (size_t)(db_.totalResidues + 64);  // two halves: ping-pong between passes
    if (!device_alloc(db_.device, (void**)&dBndH_, bytes) || !device_alloc(db_.device, (void**)&dBndF_, bytes)) return false;
    return true;
}

// ------------------------------------------------------------------ searches
ScoreBounds Scoring::bounds() const {
    ScoreBounds b;
    const long long n = num_entries();
    if (n > 0) { b.maxEntry = INT_MIN; b.minEntry = INT_MAX; }
    for (long long i = 0; i < n; i++) { b.maxEntry = std::max(b.maxEntry, entries[i]); b.minEntry = std::min(b.minEntry, entries[i]); }
    b.absEntry = std::max<long long>(std::llabs((long long)b.maxEntry), std::llabs((long long)b.minEntry));
    b.gapMax = std::max<long long>(std::llabs((long long)Go), std::llabs((long long)Ge));
    b.args16 = b.absEntry <= 2048 && b.gapMax <= 2048;
    b.args32 = b.absEntry < (1 << 28) && b.gapMax < (1 << 28);
    return b;
}

int Scoring::validate(ScoreBounds* b) const {
    if (!valid_mode(mode)) return OPAL_B200_ERR_MODE;
    // Any unsigned char alphabet (reference src/opal.h:96-98).
    if (A <= 0 || A > 256) { set_error("alphabetLength must be in [1, 256]"); return OPAL_B200_ERR_ARGUMENT; }
    // Argument range of the widest pass (reference src/opal.cpp:183-198, 615-630), over every entry that can score a cell.
    if (Go <= INT_MIN / 2 || INT_MAX / 2 <= Go || Ge <= INT_MIN / 2 || INT_MAX / 2 <= Ge) return OPAL_B200_ERR_OVERFLOW;
    *b = bounds();
    if (b->minEntry <= INT_MIN / 2 || INT_MAX / 2 <= b->maxEntry) return OPAL_B200_ERR_OVERFLOW;
    if (Go < 0 || Ge < 0) { set_error("gap penalties must be non-negative"); return OPAL_B200_ERR_ARGUMENT; }
    if (!b->args32) return OPAL_B200_ERR_OVERFLOW;  // beyond the widths this engine carries (documented deviation)
    for (int r = 0; r < Q && !byPssm; r++)
        if (query[r] >= A) { set_error("query holds residue codes >= alphabetLength"); return OPAL_B200_ERR_ARGUMENT; }
    return 0;
}

void SearchOut::put(int i, int score, int endQuery, int endTarget) const {
    if (records) {
        OpalSearchResult* r = records[i];
        r->scoreSet = 1; r->score = score;                                  // reference src/opal.cpp:1561-1564
        r->endLocationQuery = endQuery; r->endLocationTarget = endTarget;  // :420-426, 869-905
        if (noAlignmentFill) { r->alignment = NULL; r->alignmentLength = -1; r->startLocationQuery = r->startLocationTarget = -1; }
    } else {
        scores[i] = score;
        if (endQ) endQ[i] = endQuery;
        if (endT) endT[i] = endTarget;
    }
}

// The search in progress as its planning and launches see it: built once its arguments have passed.
struct SearchContext::Run {
    const Scoring& s;
    int wantEnd;
    ScoreBounds b;  // (args16 cleared when the database holds a code the 16-bit streams cannot carry, see search())
    // NW / HW / OV at 16 bits are guarded by the kernel's range tracking (search_kernel.cuh): samples of H that stay
    // (R + 3) step inside [rangeLo, 32767] prove that no cell left it, where step = Go + Ge + |largest entry| bounds the
    // difference of neighbouring cells; a target whose samples come nearer is flagged and re-run at 32 bits.
    // rangeLo is -28000 for NW (the -infinity of E and F sits at -30000).  HW / OV track the last query row in EVERY
    // column a pair sweeps, the pad columns of its shorter member included, and a pad cell is diag + padLetterScore
    // (-16384) -- diag must stay above -16383 or the cell wraps into a large positive "score" (ADVICE r1): -16383.
    // Tracking needs the margin of the tallest strip (R = 33, rounded up to 40 steps) to stay small.
    long long step = (long long)s.Go + s.Ge + b.absEntry, rangeLo = s.mode == kModeNW ? -28000 : -16383;
    bool rangeTracking = s.mode != kModeSW && b.args16 && 40 * step <= 6000;
    const unsigned char* dQuery = nullptr;  // the arguments on the device (upload_args); no query with a PSSM
    const int* dEntries = nullptr;          // the matrix or the PSSM
    int* dCounters = nullptr;               // one launch counter per launch slot
    mutable int slot = 0;                   // the next launch slot
};

// The targets of a search by precision class (sorted positions, ascending).
struct SearchContext::Routes {
    std::vector<int> list16, list32;
    int emptyFrom = 0;  // results on the device: first sorted position of the zero-length targets (n: none)
};

// One kernel-launch group: tasks that share a precision class and a geometry.
struct SearchContext::Group {
    int type = 0;            // 0 = Packed16 (tasks are pair indices), 1 = Scalar32 (tasks are sorted-target indices)
    std::vector<int> tasks;  // longest first
    Geometry g;
    size_t smemBytes = 0;    // dynamic shared memory requested (>= g.smemBytes, see exclusive placement below)
    int maxBlocks = 0;
    double estCycles = 0;    // planner's estimate, used to share SMs between concurrent groups
};

// Splits one precision class into launch groups.  A database whose longest targets would keep single warps
// busy long after everything else has finished (the tail bound of pick_geometry) gets a "latency class":
// its longest tasks run with 32 threads per task and one warp per scheduler partition on SMs of their own,
// concurrently with the throughput-oriented bulk group on the remaining SMs.
bool SearchContext::plan_class(int type, const std::vector<int>& list, const Run& run, std::vector<Group>* groups, double deadline) {
    if (list.empty()) return true;
    const int Q = run.s.Q, A = run.s.A, mode = run.s.mode, wantEnd = run.wantEnd;
    const int lanes = type == 0 ? 2 : 1;
    // Packed16 works on the pairs fixed at packing time (targets 2p, 2p+1): a pair runs if either member
    // is wanted; results of unwanted members are simply not published.
    std::vector<int> tasks;
    if (lanes == 2) {
        for (int t : list) if (tasks.empty() || tasks.back() != (t >> 1)) tasks.push_back(t >> 1);
    } else {
        tasks = list;
    }
    // The usual list is "every non-empty target": its prefix sums live with the layout (they cost more than the rest
    // of the planning for half a million targets and depend on nothing else).
    TaskLens own;
    const bool everything = (int)list.size() == db_.lay->nonEmpty && list.front() == 0 && list.back() == db_.lay->nonEmpty - 1;
    if (!everything) {
        own.len.resize(tasks.size());
        for (size_t k = 0; k < tasks.size(); k++) own.len[k] = db_.lay->sortedLen[lanes == 2 ? 2 * tasks[k] : tasks[k]];
        own.build();
    }
    const TaskLens& tl = everything ? (lanes == 2 ? db_.lay->pair_lens() : db_.lay->target_lens()) : own;
    const size_t nT = tasks.size();

    Geometry gAll;
    double tAll = 0;
    const int flavorClass = mode == kModeSW ? (wantEnd ? 0 : 1) : 2;
    if (!pick_geometry(Q, A, lanes, tl, 0, nT, db_.smemLimit, db_.numSMs, mode, false, flavorClass, &gAll, &tAll)) return false;
    // A small class beside one that takes much longer (the sixteen targets of a global-mode search that need 32 bits
    // beside half a million that do not): it cannot end the search, so it holds the fewest SMs on which it still ends
    // well inside the other class's time instead of the many that end it soonest (measured on BASELINE configs[2],
    // NW, Q = 850: a chained 32-bit class on 12 SMs made the search 6 % slower than a plain one on 4).
    if (deadline > 0 && nT <= 256 && !getenv("OPAL_B200_GEOMETRY") && !getenv("OPAL_B200_SPLIT") && !getenv("OPAL_B200_CHAIN")) {
        for (int sms = 1; sms <= 8; sms *= 2) {
            Geometry g;
            double t = 0;
            if (!pick_geometry(Q, A, lanes, tl, 0, nT, db_.smemLimit, sms, mode, false, flavorClass, &g, &t) || t > 0.6 * deadline) continue;
            Group grp;
            grp.type = type; grp.estCycles = t; grp.tasks = tasks; grp.g = g; grp.maxBlocks = sms; grp.smemBytes = g.smemBytes;
            groups->push_back(std::move(grp));
            return true;
        }
    }
    // A class of a handful of tasks (the few targets that need 32 bits from the start, say) whose query takes several
    // passes: chained passes for all of them, no bulk group.
    if (nT < 8 && !getenv("OPAL_B200_NO_CHAIN") && !getenv("OPAL_B200_GEOMETRY")) {
        const auto& tables = kernel_tables();
        const int planes = lanes == 2 ? 2 : 1, quads = (int)((nT + 3) / 4);
        for (size_t ti = 0; ti < tables.size(); ti++) {
            const int R = tables[ti].R;
            if (!tables[ti].chainFn[0]) continue;
            const int rows = 32 * R, passes = (Q + rows - 1) / rows;
            if (passes < 2 || passes > 64 || (long long)passes * rows * 3 > (long long)Q * 4 + 96) continue;
            const int Rpad = rpad_of(R), rowStride = 32 * Rpad;
            const size_t smem = (size_t)planes * (A + 1) * rowStride * 4;
            if (smem > (size_t)db_.smemLimit || passes * quads > db_.numSMs / 3) continue;
            const double t = (tl.len[0] + 31 + 100.0 * (passes - 1)) * step_cycles(flavorClass, 1, R) * 1.08 + 40000.0;
            if (t < tAll * 0.90) {
                tAll = t;
                gAll = Geometry();
                gAll.G = 32; gAll.R = R; gAll.tableIndex = (int)ti; gAll.passes = passes; gAll.Rpad = Rpad; gAll.rowStride = rowStride;
                gAll.smemBytes = smem; gAll.warpsPerPartition = 1; gAll.padTop = mode == kModeNW ? 0 : passes * rows - Q; gAll.chain = true;
            }
        }
    }
    // candidate splits: the m longest tasks form the latency class on smL SMs
    double bestT = tAll;
    size_t bestM = 0;
    int bestSm = 0;
    Geometry bestL, bestB;
    // Folded variant of the latency class (16 bits, one pass): the 2 m longest TARGETS, one per warp in both half-words,
    // which halves the rows per thread and with them the time of the longest target.  Needs the folded stream
    // (built for the numFold longest targets) and every one of those targets wanted.
    TaskLens tlFold;
    size_t foldable = 0;
    if (lanes == 2 && db_.numFold > 0 && !getenv("OPAL_B200_NO_FOLD") && (mode == kModeSW || !getenv("OPAL_B200_NO_FOLD_GLOBAL"))) {
        while (foldable < (size_t)db_.numFold && foldable < list.size() && list[foldable] == (int)foldable) foldable++;
        tlFold.len.assign(db_.lay->sortedLen.begin(), db_.lay->sortedLen.begin() + foldable);
        tlFold.build();
    }
    if (!getenv("OPAL_B200_NO_SPLIT") && !getenv("OPAL_B200_GEOMETRY")) {
        // Development override: OPAL_B200_SPLIT="m,SMs,folded,k[,G,R]" forces the latency class (m pairs on so many
        // SMs, folded or not) and the bulk's warps per partition / group size / strip height (0 = free).
        int fm = -1, fsm = 0, fv = 0, fk = 0, fg = 0, fr = 0;
        if (const char* env = getenv("OPAL_B200_SPLIT"))
            if (sscanf(env, "%d,%d,%d,%d,%d,%d", &fm, &fsm, &fv, &fk, &fg, &fr) < 4) fm = -1;
        t_forceK = fm >= 0 ? fk : 0; t_forceG = fm >= 0 ? fg : 0; t_forceR = fm >= 0 ? fr : 0;
        for (size_t m = 4; m * 2 <= nT && m <= 4096; m *= 2) {  // (a bulk geometry that m does not align with is skipped)
            for (int variant = 0; variant < 2; variant++) {
                const size_t tasksL = variant ? 2 * m : m;
                if (variant && tasksL > foldable) continue;
                if (fm >= 0 && ((int)m != fm || variant != fv)) continue;
                for (int div = 1; div <= 4; div *= 2) {
                    int smL = (int)std::min<size_t>((tasksL + 4 * div - 1) / (4 * div), (size_t)db_.numSMs / 2);
                    if (fm >= 0) { if (div > 1) continue; smL = fsm; bestT = 1e300; }
                    if (smL < 1) continue;
                    Geometry gL, gB;
                    double tL = 0, tB = 0;
                    if (!pick_geometry(Q, A, lanes, variant ? tlFold : tl, 0, tasksL, db_.smemLimit, smL, mode, true, flavorClass, &gL, &tL, variant != 0)) continue;
                    if (!pick_geometry(Q, A, lanes, tl, m, nT, db_.smemLimit, db_.numSMs - smL, mode, false, flavorClass, &gB, &tB)) continue;
                    // One search alone ends when its slower group ends.  With searches overlapping (search_batch) the SMs a
                    // group leaves are taken by the next search, so a plan costs the SM time it holds: the latency class
                    // then shrinks to the fewest SMs its tasks fit on instead of the fewest that end them soonest (measured
                    // on an eighth of BASELINE configs[2]: up to eight searches in flight each held 4+ SMs at a third of
                    // their issue rate for a tail several times longer than its bulk).
                    const double t = (t_overlapped ? (smL * tL + (db_.numSMs - smL) * tB) / db_.numSMs : std::max(tL, tB)) + 3000.0;  // a second launch is not free
                    if (t < bestT * 0.97) { bestT = t; bestM = m; bestSm = smL; bestL = gL; bestB = gB; }
                }
            }
        }
        // Chained variant of the latency class for queries that take several passes: every pass of a task on a warp
        // of its own, all of them sweeping at once (SearchParams::chain) -- passes x quads SMs, but the longest target
        // costs its length in steps once, not once per pass.  Priced for a few strip heights: shorter strips mean
        // faster steps and more SMs.
        if (!getenv("OPAL_B200_NO_CHAIN") && fm < 0) {
            const auto& tables = kernel_tables();
            const int planes = lanes == 2 ? 2 : 1;
            const bool force = getenv("OPAL_B200_CHAIN") != nullptr;  // tests: chain whenever there are several passes
            for (size_t m = 4; m * 2 <= nT && m <= 32; m *= 2) {
                const int quads = (int)((m + 3) / 4);
                for (size_t ti = 0; ti < tables.size(); ti++) {
                    const int R = tables[ti].R;
                    if (!tables[ti].chainFn[0]) continue;  // chained variants exist for a few strip heights (search_kernel.cuh)
                    const int rows = 32 * R, passes = (Q + rows - 1) / rows;
                    if (passes < 2 || passes > 64) continue;
                    if ((long long)passes * rows * 3 > (long long)Q * 4 + 96) continue;  // more than a third padding
                    const int Rpad = rpad_of(R), rowStride = 32 * Rpad;
                    const size_t smem = (size_t)planes * (A + 1) * rowStride * 4;
                    const int smL = passes * quads;
                    if (smem > (size_t)db_.smemLimit || smL > db_.numSMs / 3) continue;
                    Geometry gL, gB;
                    gL.G = 32; gL.R = R; gL.tableIndex = (int)ti; gL.passes = passes; gL.Rpad = Rpad; gL.rowStride = rowStride;
                    gL.smemBytes = smem; gL.warpsPerPartition = 1; gL.padTop = mode == kModeNW ? 0 : passes * rows - Q; gL.chain = true;
                    // every pass trails the one above by about three chunks of 32 columns
                    const double tL = (tl.len[0] + 31 + 100.0 * (passes - 1)) * step_cycles(flavorClass, 1, R) * 1.08 + 40000.0;
                    double tB = 0;
                    if (!pick_geometry(Q, A, lanes, tl, m, nT, db_.smemLimit, db_.numSMs - smL, mode, false, flavorClass, &gB, &tB)) continue;
                    const double t = (t_overlapped ? (smL * tL + (db_.numSMs - smL) * tB) / db_.numSMs : std::max(tL, tB)) + 3000.0;
                    // (a tenth better at least: a folded or plain latency class of equal speed holds fewer SMs)
                    if (t < bestT * 0.90 || (force && !bestL.chain)) { bestT = t; bestM = m; bestSm = smL; bestL = gL; bestB = gB; }
                }
            }
        }
        t_forceK = t_forceG = t_forceR = 0;
    }
    auto add = [&](size_t lo, size_t hi, const Geometry& g, int maxBlocks, size_t otherSmem, double est) {
        Group grp;
        grp.type = type;
        grp.estCycles = est;
        if (g.folded) {  // tasks are the sorted targets 0 .. 2 hi - 1 themselves
            grp.tasks.resize(2 * hi);
            for (size_t k = 0; k < 2 * hi; k++) grp.tasks[k] = (int)k;
        } else {
            grp.tasks.assign(tasks.begin() + lo, tasks.begin() + hi);
        }
        grp.g = g;
        grp.maxBlocks = maxBlocks;
        grp.smemBytes = g.smemBytes;
        // exclusive placement: ask for enough shared memory that a block of the other group cannot join this SM
        if (otherSmem > 0 && g.smemBytes + otherSmem <= (size_t)db_.smemLimit)
            grp.smemBytes = std::min<size_t>((size_t)db_.smemLimit, (size_t)db_.smemLimit - otherSmem + 1024);
        groups->push_back(std::move(grp));
    };
    if (bestM == 0) add(0, tasks.size(), gAll, db_.numSMs, 0, tAll);
    else {
        add(0, bestM, bestL, bestSm, bestB.smemBytes, bestT);   // launched first: takes its SMs
        // every block's first tasks are assigned statically (longest first), so the bulk grid must be fully
        // resident from the start: one block per SM the latency class leaves free
        add(bestM, tasks.size(), bestB, db_.numSMs - bestSm, 0, bestT);
    }
    return true;
}

// The dynamic shared-memory ceiling of a kernel is per-function state shared by every host thread (search_batch runs
// up to eight of them over the same kernels): it is raised once per (device, kernel) to the device limit instead of
// being set to each launch's size, which another thread could lower between one thread's set and its launch.
static bool allow_full_smem(int device, const void* fn, int smemLimit) {
    static std::mutex mu;
    static std::vector<std::pair<int, const void*>> done;
    std::lock_guard<std::mutex> lk(mu);
    for (const auto& d : done)
        if (d.first == device && d.second == fn) return true;
    CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smemLimit));
    done.push_back({device, fn});
    return true;
}

// Launches every pass of one group on `stream`.
bool SearchContext::launch_group(const Group& grp, int* taskListDevice, cudaStream_t stream, const Run& run) {
    const Geometry& g = grp.g;
    const int type = grp.type, mode = run.s.mode, wantEnd = run.wantEnd, maxScore = run.b.maxEntry;
    if (g.passes > 1 && !g.chain && !ensure_boundary()) return false;
    if (run.slot + g.passes > 256) { set_error("too many passes"); return false; }
    // contiguous task ranges need no list in device memory
    bool contiguous = true;
    for (size_t k = 1; k < grp.tasks.size() && contiguous; k++) contiguous = grp.tasks[k] == grp.tasks[k - 1] + 1;
    if (!contiguous)
        CUDA_TRY(cudaMemcpyAsync(taskListDevice, grp.tasks.data(), sizeof(int) * grp.tasks.size(), cudaMemcpyHostToDevice, stream));
    // SW score+end at 16 bits uses the key-tracking flavor: exact below fastEndLimit, and warps that meet a
    // larger score sweep their tasks again with the exact per-cell tracking inside the same kernel.
    const int fastEndLimit = (32768 >> kRowBits) - std::max(maxScore, 0) - 1;
    const bool fastEnd = mode == kModeSW && wantEnd && type == 0 && g.R <= (1 << kRowBits) && fastEndLimit >= 64 &&
                         !getenv("OPAL_B200_EXACT_END");
    const int flavor = (mode == kModeSW) ? (wantEnd ? (fastEnd ? kFlavorSWEndFast : kFlavorSWEnd) : kFlavorSWScore) : kFlavorGlobal;
    const void* fn = kernel_tables()[g.tableIndex].fn[type * 4 + flavor];
    if (flavor == kFlavorGlobal && 128 * g.warpsPerPartition > launch_bound_for(flavor, g.R))
        fn = kernel_tables()[g.tableIndex].fn[type == 0 ? 8 : type * 4 + flavor];  // Packed16 variant compiled for 384 threads
    if (g.chain) fn = kernel_tables()[g.tableIndex].chainFn[type * 4 + flavor];
    if (!fn) { set_error("no kernel for this geometry"); return false; }
    if (!allow_full_smem(db_.device, fn, db_.smemLimit)) return false;
    // chained passes: one launch, passes x quads blocks; boundary rows and flags live in a block of their own
    int chainStride = 0;
    int *dChainOffsets = nullptr, *dChainDone = nullptr, *dChainTicket = nullptr;
    uint32_t *dChainH = nullptr, *dChainF = nullptr;
    if (g.chain) {
        std::vector<int> offsets(grp.tasks.size());
        for (size_t k = 0; k < grp.tasks.size(); k++) {
            offsets[k] = chainStride;
            chainStride += db_.lay->sortedLen[type == 0 ? 2 * (size_t)grp.tasks[k] : (size_t)grp.tasks[k]] + 32;
        }
        chainStride = (chainStride + 63) / 64 * 64;
        const size_t nT = grp.tasks.size(), flags = nT * (size_t)g.passes;
        const size_t ints = nT + flags + 64, words = 2 * (size_t)g.passes * (size_t)chainStride;
        int* block = nullptr;
        if (!device_alloc(db_.device, (void**)&block, sizeof(int) * (ints + words))) return false;
        chainScratch_.push_back(block);
        dChainOffsets = block; dChainDone = block + nT; dChainTicket = dChainDone + flags;
        dChainH = reinterpret_cast<uint32_t*>(block + ints); dChainF = dChainH + (size_t)g.passes * chainStride;
        CUDA_TRY(cudaMemsetAsync(block, 0, sizeof(int) * ints, stream));
        fill_words_kernel<<<std::min<size_t>((words + 1023) / 1024, 4 * (size_t)db_.numSMs), 256, 0, stream>>>(dChainH, words, type == 0 ? kChainEmpty : kChainEmpty32);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(dChainOffsets, offsets.data(), sizeof(int) * nT, cudaMemcpyHostToDevice, stream));  // (pageable: staged before the call returns)
        stats_.chainedTasks = (int)nT;
    }
    for (int pass = 0; pass < (g.chain ? 1 : g.passes); pass++) {
        SearchParams p;
        memset(&p, 0, sizeof(p));
        p.query = run.dQuery; p.matrix = run.dEntries; p.pssm = run.s.byPssm ? run.dEntries : nullptr;
        p.Q = run.s.Q; p.A = run.s.A; p.gapOpen = run.s.Go; p.gapExt = run.s.Ge; p.mode = mode; p.wantEnd = wantEnd;
        p.G = g.G; p.rowBase = pass * g.G * g.R; p.padTop = g.padTop; p.pass = pass; p.numPasses = g.passes;
        p.rowStride = g.rowStride; p.Rpad = g.Rpad;
        p.residues = db_.dResidues; p.offsets = db_.dOffsets; p.lengths = db_.dLengths;
        p.pairStream = db_.dPairStream; p.pairOffsets = db_.dPairOffsets; p.numTargets = db_.n;
        if (g.folded) { p.folded = 1; p.pairStream = db_.dFoldStream; p.pairOffsets = db_.dFoldOffsets; stats_.foldedTasks = (int)grp.tasks.size(); }
        p.taskList = contiguous ? nullptr : taskListDevice;
        p.taskBase = contiguous && !grp.tasks.empty() ? grp.tasks[0] : 0;
        p.numTasks = (int)grp.tasks.size();
        p.counter = run.dCounters + run.slot++;
        const size_t half = (size_t)(db_.totalResidues + 64);
        p.bndInH = dBndH_ ? dBndH_ + ((pass + 1) & 1) * half : nullptr; p.bndInF = dBndF_ ? dBndF_ + ((pass + 1) & 1) * half : nullptr;
        p.bndOutH = dBndH_ ? dBndH_ + (pass & 1) * half : nullptr; p.bndOutF = dBndF_ ? dBndF_ + (pass & 1) * half : nullptr;
        p.outScore = dScore_; p.outEndQ = dEndQ_; p.outEndT = dEndT_;
        p.overflowLimit = type == 0 ? 32767 - std::max(maxScore, 0) - 1 : (1 << 30);
        // The "no residue" letter of the 16-bit streams (pad columns of a pair's shorter member, idle columns).  SW: a
        // pad cell must not raise the running maximum; HW / OV: the last query row is tracked in pad columns too and
        // must stay below what the real columns gave -- very negative.  NW reads one cell per target and never a pad
        // column: 0 keeps pad cells inside the range of the real ones, so they cannot trip the range tracking.
        p.padLetterScore = type == 0 ? (mode == kModeNW ? 0 : -16384) : 0;
        p.one = 1; p.keyScale = 1 << kRowBits; p.fastEndLimit = fastEndLimit;
        {   // range tracking of the 16-bit NW / HW / OV sweeps (see SearchContext::Run for the limits)
            const long long margin = (long long)(g.R + 3) * run.step;
            p.rangeHi = run.rangeTracking ? (int)(32767 - margin) : INT_MAX;   // (not tracking: routed by the a-priori bound)
            p.rangeLo = run.rangeTracking ? (int)(run.rangeLo + margin) : INT_MIN;
        }
        if (g.chain) {
            p.chain = 1; p.chainStride = chainStride; p.chainOffsets = dChainOffsets;
            p.chainDone = dChainDone; p.chainTicket = dChainTicket;
            p.bndInH = p.bndInF = nullptr; p.bndOutH = dChainH; p.bndOutF = dChainF;
        }
        void* args[] = {&p};
        const int warpsPerBlock = 4 * g.warpsPerPartition;  // one block per SM, k warps per scheduler partition
        const long long warpsNeeded = ((long long)grp.tasks.size() * g.G + 31) / 32;
        int blocks = (int)std::max<long long>(1, std::min<long long>(grp.maxBlocks, (warpsNeeded + warpsPerBlock - 1) / warpsPerBlock));
        if (g.chain) blocks = g.passes * (int)((grp.tasks.size() + warpsPerBlock - 1) / warpsPerBlock);  // every pass of every quad
        CUDA_TRY(cudaLaunchKernel(fn, dim3(blocks), dim3(32 * warpsPerBlock), args, grp.smemBytes, stream));
        stats_.kernelLaunches++;
    }
    stats_.G = g.G; stats_.R = g.R; stats_.passes = g.passes; stats_.warpsPerPartition = g.warpsPerPartition;
    return true;
}

// Runs the given classes concurrently: every launch group gets a stream of its own (the first one the
// database's main stream), all of them ordered after `ready` and joined back into the main stream.
int SearchContext::run_classes(const std::vector<std::pair<int, const std::vector<int>*>>& classes, const Run& run) {
    std::vector<Group> groups;
    PhaseTrace trace("run_classes");
    // the class with the most targets first: what it is estimated to take is the time the small ones may hide in
    std::vector<size_t> orderOfClasses(classes.size());
    for (size_t i = 0; i < classes.size(); i++) orderOfClasses[i] = i;
    std::stable_sort(orderOfClasses.begin(), orderOfClasses.end(),
                     [&](size_t a, size_t b) { return classes[a].second->size() > classes[b].second->size(); });
    double deadline = 0;
    for (size_t i : orderOfClasses) {
        const size_t before = groups.size();
        if (!plan_class(classes[i].first, *classes[i].second, run, &groups, deadline)) return OPAL_B200_ERR_CUDA;
        if (deadline == 0)
            for (size_t g = before; g < groups.size(); g++) deadline = std::max(deadline, groups[g].estCycles);
    }
    if (groups.empty()) return 0;
    trace.mark("plan");
    stats_.groups = (int)groups.size();
    // Concurrent groups own disjoint SMs (grids are persistent, one block per SM, and every block must be
    // resident from the start because first tasks are assigned statically).  Small groups -- the latency
    // class, a handful of 32-bit targets -- get the blocks they can fill and are launched first; the
    // remaining SMs are shared by the large groups in proportion to their estimated work.
    if (groups.size() > 1) {
        auto wanted = [&](const Group& g) {
            const int wpb = 4 * g.g.warpsPerPartition;
            const long long warps = ((long long)g.tasks.size() * g.g.G + 31) / 32;
            if (g.g.chain) return (int)(g.g.passes * ((warps + wpb - 1) / wpb));  // every pass of every quad has a block
            return (int)std::max<long long>(1, std::min<long long>(g.maxBlocks, (warps + wpb - 1) / wpb));
        };
        std::stable_sort(groups.begin(), groups.end(), [&](const Group& a, const Group& b) { return wanted(a) < wanted(b); });
        std::vector<int> want(groups.size());
        std::vector<char> big(groups.size(), 0);
        for (size_t i = 0; i < groups.size(); i++) want[i] = wanted(groups[i]);
        int reserved = 0;
        double bigWork = 0;
        for (size_t i = 0; i < groups.size(); i++) {
            if (want[i] * 4 <= db_.numSMs && reserved + want[i] <= db_.numSMs / 2) { groups[i].maxBlocks = want[i]; reserved += want[i]; }
            else { big[i] = 1; bigWork += std::max(1.0, groups[i].estCycles * want[i]); }
        }
        const int left = db_.numSMs - reserved;
        for (size_t i = 0; i < groups.size(); i++) {
            if (!big[i]) continue;
            const int share = std::max(1, (int)(left * std::max(1.0, groups[i].estCycles * want[i]) / bigWork));
            groups[i].maxBlocks = std::min(share, want[i]);
        }
    }
    if (getenv("OPAL_B200_TRACE"))
        for (const Group& g : groups)
            fprintf(stderr, "[opal-b200] group type=%d%s tasks=%zu longest=%d G=%d R=%d k=%d passes=%d blocks<=%d est=%.0f kcycles\n", g.type,
                    g.g.folded ? " folded" : g.g.chain ? " chained" : "", g.tasks.size(),
                    g.tasks.empty() ? 0 : db_.lay->sortedLen[g.type == 0 && !g.g.folded ? 2 * g.tasks[0] : g.tasks[0]], g.g.G, g.g.R,
                    g.g.warpsPerPartition, g.g.passes, g.maxBlocks, g.estCycles / 1e3);
    bool badArgument = false;
    auto body = [&]() -> bool {
        size_t listOffset = 0;
        // create() returns with the upload in flight; planning above ran beside it.  The residue codes are
        // validated here, before anything indexes the profile with them.
        if (!ensure_uploaded()) return false;
        trace.mark("upload-wait");
        if (*db_.hMaxCode >= run.s.A) { set_error("database holds residue codes >= alphabetLength"); badArgument = true; return false; }
        if (!startRecorded_) { CUDA_TRY(cudaEventRecord(evStart_, stream_)); startRecorded_ = true; }  // planning is host work: keep it outside the device window
        if (groups.size() > 1) CUDA_TRY(cudaEventRecord(evFork_, stream_));
        for (size_t gi = 0; gi < groups.size(); gi++) {
            cudaStream_t st = stream_;
            if (gi > 0) {
                while (auxStreams_.size() < gi) {
                    cudaStream_t s2; cudaEvent_t e2;
                    if (!stream_acquire(db_.device, &s2) || !event_acquire(db_.device, &e2)) return false;
                    auxStreams_.push_back(s2); auxEvents_.push_back(e2);
                }
                st = auxStreams_[gi - 1];
                CUDA_TRY(cudaStreamWaitEvent(st, evFork_, 0));
            }
            if (!launch_group(groups[gi], dTaskList_ + listOffset, st, run)) return false;
            listOffset += groups[gi].tasks.size();
            if (gi > 0) {
                CUDA_TRY(cudaEventRecord(auxEvents_[gi - 1], st));
                CUDA_TRY(cudaStreamWaitEvent(stream_, auxEvents_[gi - 1], 0));
            }
        }
        return true;
    };
    return body() ? 0 : (badArgument ? OPAL_B200_ERR_ARGUMENT : OPAL_B200_ERR_CUDA);
}

int SearchContext::search(const Scoring& s, int wantEnd, const unsigned char* skip, const SearchOut& out, float* deviceMs) {
    stats_ = SearchStats();
    for (void* b : chainScratch_) device_release(db_.device, b);  // (the previous search has been waited for)
    chainScratch_.clear();
    PhaseTrace trace("search");
    if (deviceMs) *deviceMs = 0.f;
    ScoreBounds b;
    if (const int rc = s.validate(&b)) return rc;
    // The 16-bit streams store residue code + 1 in a byte, so code 255 cannot ride in them: a database that really
    // holds it (alphabetLength 256) is searched by the 32-bit class, which reads the plain stream.
    if (s.A == 256) {
        if (!ensure_uploaded()) return OPAL_B200_ERR_CUDA;
        if (*db_.hMaxCode >= 255) b.args16 = false;
    }
    Run run{s, wantEnd, b};
    Routes routes;
    if (const int rc = route(run, skip, out, &routes)) return rc;
    if (routes.list16.empty() && routes.list32.empty() && !out.dSelect) return 0;
    trace.mark("route");
    if (!upload_args(&run)) return OPAL_B200_ERR_CUDA;
    int rc = 0;
    return ladder(run, routes, out, deviceMs, trace, &rc) ? rc : OPAL_B200_ERR_CUDA;
}

// Every non-skipped target to the 16-bit or the 32-bit class; a target with nothing to align gets its result here.
// 0 or OPAL_B200_ERR_OVERFLOW (a target that 32 bits cannot hold).
int SearchContext::route(const Run& run, const unsigned char* skip, const SearchOut& out, Routes* routes) {
    const int Q = run.s.Q, Go = run.s.Go, Ge = run.s.Ge, mode = run.s.mode, maxP = run.b.maxEntry;
    const bool isSW = mode == kModeSW, args16 = run.b.args16, track16 = run.rangeTracking;
    auto& [list16, list32, emptyFrom] = *routes;
    // NW/HW/OV: every H, E, F of a (Q, T) problem lies in [-(3Go + (Q+T)Ge + |minP|), min(Q,T) maxP + Go].
    auto fits = [&](int T, long long lim) -> bool {
        const long long lo = 3LL * Go + ((long long)Q + T) * Ge + run.b.absEntry;
        const long long hi = (maxP > 0 ? (long long)std::min(Q, T) * maxP : 0) + Go + run.b.absEntry;
        return lo <= lim && hi <= lim;
    };
    // NW / HW / OV at 16 bits.  An a-priori bound on every H of a (Q, T) problem -- min(Q, T) maxP upwards,
    // (Q + T) gapExt downwards -- is hopelessly pessimistic for real sequences (it sends every target beyond ~1,500
    // residues to the 32-bit class once Q >= 1,500 with BLOSUM62), so only the values that are CERTAIN to occur are
    // bounded here: the borders of the matrix (column -1: -Go - r Ge for NW and HW; row -1: -Go - c Ge for NW).
    // Everything else is watched by the kernel's range tracking (Run).
    auto fits16 = [&](int T) -> bool {
        const long long border = (long long)Go + (mode == kModeNW ? (long long)std::max(Q, T) : mode == kModeHW ? (long long)Q : 0LL) * Ge;
        return -border >= run.rangeLo + 40 * run.step;
    };
    // The routing rule; every part of it is monotone in the target length.
    auto ok16 = [&](int T) -> bool {
        if (isSW) return args16;
        return track16 ? fits16(T) : (args16 && fits(T, 16000));  // (second form: penalties too large to track)
    };
    auto ok32 = [&](int T) -> bool {
        return isSW ? (maxP > 0 ? (long long)std::min(Q, T) * maxP : 0) < (1LL << 30) : fits(T, 1LL << 30);
    };
    (args16 ? list16 : list32).reserve((size_t)db_.n);
    emptyFrom = db_.n;
    int routeFrom = 0;
    if (!skip && Q > 0) {
        // Nothing skipped: the classes are ranges of the sorted order: [0, b) needs 32 bits, [b, nonEmpty) fits 16;
        // only the empty targets are left to the loop below.
        const int m = db_.lay->nonEmpty;
        int lo = 0, hi = m;  // first position whose target fits 16 bits
        while (lo < hi) {
            const int mid = (lo + hi) / 2;
            if (ok16(db_.lay->sortedLen[mid])) hi = mid; else lo = mid + 1;
        }
        int b = lo;
        if (!isSW && (b & 1) && b < m) b++;  // a pair is never split between the classes (see below)
        if (b > 0 && !ok32(db_.lay->sortedLen[0])) return OPAL_B200_ERR_OVERFLOW;  // the longest target decides for all
        list32.resize((size_t)b);
        for (int p = 0; p < b; p++) list32[p] = p;
        list16.resize((size_t)(m - b));
        for (int p = b; p < m; p++) list16[p - b] = p;
        routeFrom = m;
    }
    for (int p = routeFrom; p < db_.n; p++) {
        const int i = db_.lay->order[p];
        if (skip && skip[i]) continue;
        const int T = db_.lay->sortedLen[p];
        if (T == 0 && out.dSelect) { emptyFrom = std::min(emptyFrom, p); continue; }  // filled on the device
        if (T == 0 || Q <= 0) {  // nothing to align: defined as in oracle/opal_oracle.c
            int sc = 0, eq = Q - 1, et = T - 1;
            if (Q > 0 && (mode == kModeNW || mode == kModeHW)) sc = -Go - (Q - 1) * Ge;  // the query against one gap
            else if (Q <= 0 && T > 0 && mode == kModeNW) sc = -Go - (T - 1) * Ge;         // ... and the target against one
            if (isSW) { eq = -1; et = -1; }
            out.put(i, sc, run.wantEnd ? eq : -1, run.wantEnd ? et : -1);
            continue;
        }
        if (ok16(T)) list16.push_back(p);
        else if (ok32(T)) list32.push_back(p);
        else return OPAL_B200_ERR_OVERFLOW;
    }
    // The 16-bit class works on whole pairs (sorted targets 2p, 2p+1) and the two classes of NW/HW/OV run
    // concurrently, so a pair is never split between them: if one member needs 32 bits, both go there.
    if (!isSW && !list32.empty() && !list16.empty()) {
        std::vector<char> wide((size_t)db_.numPairs, 0);
        for (int p : list32) wide[p >> 1] = 1;
        std::vector<int> keep16, merged32;
        for (int p : list16) (wide[p >> 1] ? merged32 : keep16).push_back(p);
        if (!merged32.empty()) {
            std::vector<int> all(list32.size() + merged32.size());
            std::merge(list32.begin(), list32.end(), merged32.begin(), merged32.end(), all.begin());
            list32.swap(all);
            list16.swap(keep16);
        }
    }
    return 0;
}

// Launch counters (zeroed), score matrix and query travel in one pinned block, one copy; with a PSSM the block is
// counters and PSSM (the query letters are not needed).
bool SearchContext::upload_args(Run* run) {
    const Scoring& s = run->s;
    CUDA_TRY(cudaSetDevice(db_.device));
    const size_t scoreBytes = sizeof(int) * (size_t)s.num_entries(), matrixBytes = (scoreBytes + 255) / 256 * 256;
    const size_t countersBytes = sizeof(int) * 256;
    const size_t argsBytes = countersBytes + matrixBytes + (s.byPssm ? 0 : (size_t)s.Q + 16);
    if (argsBytes > argsCapacity_) {
        device_release(db_.device, dArgs_); dArgs_ = nullptr;
        pinned_release(hArgs_); hArgs_ = nullptr;
        argsCapacity_ = std::max<size_t>(8192, 2 * argsBytes);
        if (!device_alloc(db_.device, (void**)&dArgs_, argsCapacity_) || !pinned_alloc((void**)&hArgs_, argsCapacity_)) { argsCapacity_ = 0; return false; }
    }
    memset(hArgs_, 0, countersBytes);
    memcpy(hArgs_ + countersBytes, s.entries, scoreBytes);
    if (!s.byPssm) memcpy(hArgs_ + countersBytes + matrixBytes, s.query, (size_t)s.Q);
    run->dCounters = reinterpret_cast<int*>(dArgs_);
    run->dEntries = reinterpret_cast<int*>(dArgs_ + countersBytes);
    if (!s.byPssm) run->dQuery = dArgs_ + countersBytes + matrixBytes;
    CUDA_TRY(cudaMemcpyAsync(dArgs_, hArgs_, argsBytes, cudaMemcpyHostToDevice, stream_));
    return true;
}

// The precision ladder: the 16-bit class (NW / HW / OV: and the 32-bit class beside it), then at 32 bits what 16 bits
// could not hold.  Results are published after every round, or stay on the device.  False: a CUDA failure; *rc: the
// search's code otherwise.
bool SearchContext::ladder(const Run& run, Routes& routes, const SearchOut& out, float* deviceMs, PhaseTrace& trace, int* rc) {
    const int Q = run.s.Q, Go = run.s.Go, Ge = run.s.Ge, mode = run.s.mode, wantEnd = run.wantEnd;
    const bool isSW = mode == kModeSW, onDevice = out.dSelect != nullptr;
    auto& [list16, list32, emptyFrom] = routes;
    startRecorded_ = false;
    // NW/HW/OV classes are independent (routed a priori) and run concurrently; SW's 32-bit class is the
    // re-run of what overflowed 16 bits and has to follow it.
    std::vector<std::pair<int, const std::vector<int>*>> first;
    if (!list16.empty()) first.push_back({0, &list16});
    if (!isSW && !list32.empty()) first.push_back({1, &list32});
    if (!first.empty()) {
        *rc = run_classes(first, run);
        if (*rc) return *rc != OPAL_B200_ERR_CUDA;  // a CUDA failure has set the error text; other codes pass through
        CUDA_TRY(cudaEventRecord(evStop_, stream_));
        // the ladder: what 16 bits could not hold (SW: the score; NW / HW / OV: the range tracking) goes to 32
        std::vector<int> again;
        if (onDevice) {
            if (!collect(out.dSelect, emptyFrom, &again)) return false;
            if (!isSW) list32.clear();
        } else {
            if (!fetch(wantEnd, trace)) return false;
            publish(list16, wantEnd, out, &again);
            if (!isSW) { if (!publish(list32, wantEnd, out, nullptr)) *rc = OPAL_B200_ERR_OVERFLOW; list32.clear(); }
        }
        if (!again.empty()) {
            stats_.rerun32 = (int)again.size();
            std::vector<int> merged(list32.size() + again.size());
            std::merge(list32.begin(), list32.end(), again.begin(), again.end(), merged.begin());
            list32.swap(merged);
        }
    }
    if (!list32.empty()) {
        *rc = run_classes({{1, &list32}}, run);
        if (*rc) return *rc != OPAL_B200_ERR_CUDA;
        CUDA_TRY(cudaEventRecord(evStop_, stream_));
        if (onDevice) {
            std::vector<int> still;
            if (!collect(out.dSelect, emptyFrom, &still)) return false;
            if (!still.empty()) *rc = OPAL_B200_ERR_OVERFLOW;
        } else {
            if (!fetch(wantEnd, trace)) return false;
            if (!publish(list32, wantEnd, out, nullptr)) *rc = OPAL_B200_ERR_OVERFLOW;
        }
    }
    if (onDevice && emptyFrom < db_.n) {  // zero-length targets: the defined result, written where a sweep would have left it
        int sc = 0, eq = Q - 1, et = -1;
        if (mode == kModeNW || mode == kModeHW) sc = -Go - (Q - 1) * Ge;
        if (isSW) { eq = 0x7fffffff; et = 0x7fffffff; }
        fill_empty_kernel<<<std::min(db_.numSMs, (db_.n - emptyFrom + 255) / 256), 256, 0, stream_>>>(dScore_, dEndQ_, dEndT_, emptyFrom, db_.n, sc, eq, et);
        CUDA_TRY(cudaGetLastError());
    }
    trace.mark("publish");
    if (deviceMs && startRecorded_) CUDA_TRY(cudaEventElapsedTime(deviceMs, evStart_, evStop_));
    return true;
}

// [score | endQ | endT] of every target back to the host: they are adjacent on both sides, one copy.
bool SearchContext::fetch(int wantEnd, PhaseTrace& trace) {
    const size_t nWords = (size_t)std::max(db_.n, 1);
    CUDA_TRY(cudaMemcpyAsync(hResults_, dResults_, sizeof(int) * (wantEnd ? 3 : 1) * nWords, cudaMemcpyDeviceToHost, stream_));
    trace.mark("launch");
    CUDA_TRY(cudaStreamSynchronize(stream_));
    trace.mark("wait");
    return true;
}

// The fetched results of `list` go back to caller order: a scatter, split over the host pool for large databases.
// Targets flagged for 32 bits go to *overflowed (sorted); without it, false when there is any.
bool SearchContext::publish(const std::vector<int>& list, int wantEnd, const SearchOut& out, std::vector<int>* overflowed) {
    std::mutex mu;
    bool placed = true;
    parallel_for((long long)list.size(), 65536, [&](long long lo, long long hi) {
        std::vector<int> flagged;
        for (long long k = lo; k < hi; k++) {
            const int p = list[(size_t)k], i = db_.lay->order[p];
            const int sc = hScore_[p];
            if (sc == kScoreOverflow || sc == kScoreNone) { flagged.push_back(p); continue; }
            out.put(i, sc, (wantEnd && hEndQ_[p] != 0x7fffffff) ? hEndQ_[p] : -1, (wantEnd && hEndT_[p] != 0x7fffffff) ? hEndT_[p] : -1);
        }
        if (!flagged.empty()) {
            std::lock_guard<std::mutex> lk(mu);
            if (overflowed) overflowed->insert(overflowed->end(), flagged.begin(), flagged.end());
            else placed = false;
        }
    });
    if (overflowed) std::sort(overflowed->begin(), overflowed->end());
    return placed;
}

// Results on the device (search_topk): the hand-over list of the ladder is gathered there (a count and the flagged
// positions come back instead of every score).
bool SearchContext::collect(int* dSelect, int emptyFrom, std::vector<int>* flagged) {
    if (emptyFrom <= 0) return true;
    CUDA_TRY(cudaMemsetAsync(dSelect, 0, sizeof(int), stream_));
    collect_flagged_kernel<<<std::min(db_.numSMs * 4, (emptyFrom + 255) / 256), 256, 0, stream_>>>(dScore_, emptyFrom, dSelect + 1, dSelect);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(hResults_, dSelect, sizeof(int), cudaMemcpyDeviceToHost, stream_));
    CUDA_TRY(cudaStreamSynchronize(stream_));
    const int count = hResults_[0];
    if (count > 0) {
        CUDA_TRY(cudaMemcpyAsync(hResults_, dSelect + 1, sizeof(int) * (size_t)count, cudaMemcpyDeviceToHost, stream_));
        CUDA_TRY(cudaStreamSynchronize(stream_));
        flagged->assign(hResults_, hResults_ + count);
        std::sort(flagged->begin(), flagged->end());
    }
    return true;
}

int SearchContext::search_topk(const Scoring& s, int wantEnd, int k, const int* map, int* outIndex, int* outScore, int* outEndQ, int* outEndT) {
    const int kk = std::min(k, db_.n);
    if (kk <= 0) return 0;
    if (s.Q <= 0) {  // degenerate: every result is written by the host anyway
        std::vector<int> sc((size_t)db_.n), eq((size_t)db_.n, -1), et((size_t)db_.n, -1);
        const int rc = search(s, wantEnd, nullptr, SearchOut::arrays(sc.data(), eq.data(), et.data()), nullptr);
        if (rc) return rc;
        std::vector<int> idx((size_t)db_.n);
        for (int i = 0; i < db_.n; i++) idx[i] = i;
        auto better = [&](int a, int b) { return sc[a] != sc[b] ? sc[a] > sc[b] : (map ? map[a] < map[b] : a < b); };
        std::partial_sort(idx.begin(), idx.begin() + kk, idx.end(), better);
        for (int j = 0; j < kk; j++) { outIndex[j] = idx[j]; outScore[j] = sc[idx[j]]; outEndQ[j] = wantEnd ? eq[idx[j]] : -1; outEndT[j] = wantEnd ? et[idx[j]] : -1; }
        return 0;
    }
    // Device path: the search leaves [score | endQ | endT] in HBM, the k best are selected there (caller indices of a
    // shard ascend with the map, so the key can use them) and 16 k bytes come back.
    if (cudaSetDevice(db_.device) != cudaSuccess) { set_error("cudaSetDevice failed"); return OPAL_B200_ERR_CUDA; }
    const size_t selectInts = (size_t)db_.n + 4 * (size_t)kk + 16;
    int* dSelect = nullptr;  // [count | flagged positions (n) | k records]
    if (!device_alloc(db_.device, (void**)&dSelect, sizeof(int) * selectInts)) return OPAL_B200_ERR_CUDA;
    const int rc = search(s, wantEnd, nullptr, SearchOut::on_device(dSelect), nullptr);
    if (rc) { device_release(db_.device, dSelect); return rc; }
    int4* dRecords = reinterpret_cast<int4*>(dSelect + (((size_t)db_.n + 4) & ~(size_t)3));
    topk_select_kernel<<<1, 1024, 0, stream_>>>(dScore_, dEndQ_, dEndT_, db_.dOrder, db_.n, kk, wantEnd, dRecords);
    std::vector<int4> rec((size_t)kk);
    if (cudaGetLastError() != cudaSuccess ||
        cudaMemcpyAsync(rec.data(), dRecords, sizeof(int4) * (size_t)kk, cudaMemcpyDeviceToHost, stream_) != cudaSuccess ||
        cudaStreamSynchronize(stream_) != cudaSuccess) {
        set_error("top-k selection failed"); device_release(db_.device, dSelect); return OPAL_B200_ERR_CUDA;
    }
    device_release(db_.device, dSelect);
    std::sort(rec.begin(), rec.end(), [&](const int4& a, const int4& b) { return a.y != b.y ? a.y > b.y : (map ? map[a.x] < map[b.x] : a.x < b.x); });
    for (int j = 0; j < kk; j++) {
        outIndex[j] = rec[j].x; outScore[j] = rec[j].y;
        outEndQ[j] = (wantEnd && rec[j].z != 0x7fffffff) ? rec[j].z : -1;
        outEndT[j] = (wantEnd && rec[j].w != 0x7fffffff) ? rec[j].w : -1;
    }
    return 0;
}

// The device copy of the index map (sorted position -> caller index) that the selection reads, made once in the
// database arrays, where every context reads it.
bool DeviceDb::ensure_order() {
    if (db_.dOrder) return true;
    if (!ensure_uploaded() || !device_alloc(db_.device, (void**)&db_.dOrder, sizeof(int) * (size_t)std::max(db_.n, 1)) ||
        cudaMemcpyAsync(db_.dOrder, db_.lay->order.data(), sizeof(int) * (size_t)db_.n, cudaMemcpyHostToDevice, stream()) != cudaSuccess ||
        cudaStreamSynchronize(stream()) != cudaSuccess) {
        set_error("upload of the index map failed");
        return false;
    }
    return true;
}

int DeviceDb::check(const Scoring& s) {
    ScoreBounds b;
    if (const int rc = s.validate(&b)) return rc;
    if (s.Q <= 0 || db_.lay->nonEmpty == 0) return 0;  // nothing is swept, so no residue code is read (see run_classes)
    if (!ensure_uploaded()) return OPAL_B200_ERR_CUDA;
    if (*db_.hMaxCode >= s.A) { set_error("database holds residue codes >= alphabetLength"); return OPAL_B200_ERR_ARGUMENT; }
    return 0;
}

// Searches claim the next index in order and stop claiming after a failure, so every search below the lowest failed
// one has run: its code is the one a loop of single searches would have returned.  The upload is waited for before
// the contexts are made, so none of them waits for it on a thread of its own.
int DeviceDb::in_flight(int num, int inFlight, const std::function<int(SearchContext&, int)>& job, float* batchMs) {
    if (batchMs) *batchMs = 0.f;
    if (num <= 0) return 0;
    const int K = std::max(1, std::min(std::min(inFlight, num), 16));
    if (cudaSetDevice(db_.device) != cudaSuccess) { set_error("cudaSetDevice failed"); return OPAL_B200_ERR_CUDA; }
    if (!ensure_uploaded()) return OPAL_B200_ERR_CUDA;
    while ((int)contexts_.size() < K) {
        auto c = std::make_unique<SearchContext>(db_);
        if (!c->alloc_search_buffers()) return OPAL_B200_ERR_CUDA;
        contexts_.push_back(std::move(c));
    }
    cudaEvent_t evBatch = nullptr;
    if (!event_acquire(db_.device, &evBatch)) return OPAL_B200_ERR_CUDA;
    if (cudaEventRecord(evBatch, stream()) != cudaSuccess) { event_release(db_.device, evBatch); set_error("cudaEventRecord failed"); return OPAL_B200_ERR_CUDA; }
    std::atomic<int> next(0);
    std::atomic<bool> stop(false);
    std::vector<int> rcs((size_t)num, 0);
    std::vector<std::string> errors((size_t)num);
    std::vector<float> lastStop((size_t)K, 0.f);
    std::vector<int> launches((size_t)K, 0), reruns((size_t)K, 0);
    auto worker = [&](int k) {
        SearchContext& ctx = *contexts_[k];
        while (!stop.load()) {
            const int q = next.fetch_add(1);
            if (q >= num) break;
            const int rc = job(ctx, q);
            if (rc) { rcs[q] = rc; errors[q] = last_error(); stop.store(true); break; }
            launches[k] += ctx.stats_.kernelLaunches; reruns[k] += ctx.stats_.rerun32;
            float ms = 0.f;
            if (ctx.startRecorded_ && cudaEventElapsedTime(&ms, evBatch, ctx.evStop_) == cudaSuccess) lastStop[k] = std::max(lastStop[k], ms);
        }
    };
    if (K == 1) worker(0);
    else {
        std::vector<std::thread> th;
        for (int k = 1; k < K; k++) th.emplace_back([&worker, k]() { t_overlapped = true; worker(k); });
        t_overlapped = true;
        worker(0);
        t_overlapped = false;
        for (auto& t : th) t.join();
    }
    event_release(db_.device, evBatch);
    for (int q = 0; q < num; q++)
        if (rcs[q]) { set_error(errors[q]); return rcs[q]; }
    if (batchMs) *batchMs = *std::max_element(lastStop.begin(), lastStop.end());
    SearchStats& stats = contexts_[0]->stats_;  // batch totals
    stats.kernelLaunches = stats.rerun32 = 0;
    for (int k = 0; k < K; k++) { stats.kernelLaunches += launches[k]; stats.rerun32 += reruns[k]; }
    return 0;
}

int DeviceDb::search_batch(const std::vector<Scoring>& searches, int wantEnd, int* scores, int* endQ, int* endT, int inFlight,
                           float* batchMs) {
    return in_flight((int)searches.size(), inFlight, [&](SearchContext& ctx, int q) {
        const size_t base = (size_t)q * (size_t)db_.n;
        const SearchOut out = SearchOut::arrays(scores + base, endQ ? endQ + base : nullptr, endT ? endT + base : nullptr);
        return ctx.search(searches[q], wantEnd, nullptr, out, nullptr);
    }, batchMs);
}

int DeviceDb::search_batch_topk(const std::vector<Scoring>& searches, int wantEnd, int k, const int* map, int* outIndex, int* outScore,
                                int* outEndQ, int* outEndT, int inFlight) {
    if (k <= 0 || searches.empty()) return 0;
    if (cudaSetDevice(db_.device) != cudaSuccess) { set_error("cudaSetDevice failed"); return OPAL_B200_ERR_CUDA; }
    if (!ensure_order()) return OPAL_B200_ERR_CUDA;
    return in_flight((int)searches.size(), inFlight, [&](SearchContext& ctx, int q) {
        const size_t base = (size_t)q * (size_t)k;
        return ctx.search_topk(searches[q], wantEnd, k, map, outIndex + base, outScore + base, outEndQ + base, outEndT + base);
    }, nullptr);
}

// ------------------------------------------------------------------ pairs path
#define CUDA_TRY_RC(expr)                                                                    \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                   \
            return OPAL_B200_ERR_CUDA;                                                       \
        }                                                                                    \
    } while (0)

// One precision class of a pairs call, grouped and planned: tasks of one query are consecutive (longest target first),
// blocks serve runs of them (PairBlock), and every query has its strip geometry (PairQuery).
struct PairsSearch::Class {
    int type = 0, rIndex = 0, maxG = 1, maxPasses = 1;
    std::vector<PairQuery> queryTab;
    std::vector<PairTask> tasks;
    std::vector<PairBlock> blocks;
    long long streamEntries = 0, bndWords = 0;
};

PairsSearch::~PairsSearch() {
    cudaSetDevice(db_.device);
    cudaStreamSynchronize(stream_);  // nothing may still be using the blocks when they go back to the cache
    for (void* p : device_) device_release(db_.device, p);
    for (void* p : pinned_) pinned_release(p);
    event_release(db_.device, evStart_); event_release(db_.device, evStop_);
}

void* PairsSearch::alloc(size_t bytes) {
    void* p = nullptr;
    if (!device_alloc(db_.device, &p, bytes)) return nullptr;
    device_.push_back(p);
    return p;
}

// One pinned block, one copy.
bool PairsSearch::upload(const std::vector<unsigned char>& block, unsigned char** dBlock, unsigned char** hBlock) {
    void* h = nullptr;
    if (!pinned_alloc(&h, block.size())) return false;
    pinned_.push_back(h);
    memcpy(h, block.data(), block.size());
    *hBlock = static_cast<unsigned char*>(h);
    if (!(*dBlock = static_cast<unsigned char*>(alloc(block.size())))) return false;
    CUDA_TRY(cudaMemcpyAsync(*dBlock, h, block.size(), cudaMemcpyHostToDevice, stream_));
    return true;
}

// Geometry and tables of one class.  The strip height is one per launch (it is a template parameter): the one the B200
// step-time model (step_cycles, three warps per partition) prices lowest over every task of the class.  Per query, the
// group size G is the smallest power of two whose G x R rows cover the query, within what shared memory holds.
bool PairsSearch::plan(int type, const std::vector<Scoring>& queries, int wantEnd, const std::vector<std::vector<int>>& byQuery,
                       const int* pos, Class* c) {
    const Scoring& s0 = queries[0];
    const int lanes = type == 0 ? 2 : 1, A = s0.A, warps = kPairsThreads / 32;
    const int flavorClass = s0.mode == kModeSW ? (wantEnd ? 0 : 1) : 2;
    const std::vector<int>& sortedLen = db_.lay->sortedLen;
    auto geometry = [&](int ri, int Q, int* G, int* passes) {
        const int R = kPairsR[ri];
        auto smem = [&](int g) { return (size_t)lanes * (A + 1) * ((g * pairs_rpad(R) + 31) / 32 * 32) * 4; };
        int g = 1;
        while (g < 32 && g * R < Q) g *= 2;
        while (g > 1 && smem(g) > (size_t)db_.smemLimit) g /= 2;
        *G = g;
        *passes = (Q + g * R - 1) / (g * R);
        return smem(g) <= (size_t)db_.smemLimit;
    };
    double bestCost = 1e300;
    c->rIndex = -1;
    for (int ri = 0; ri < 2; ri++) {
        double cost = 0;
        bool fits = true;
        for (size_t q = 0; q < byQuery.size() && fits; q++) {
            if (byQuery[q].empty()) continue;
            int G = 1, passes = 1;
            fits = geometry(ri, queries[q].Q, &G, &passes);
            double steps = 0;
            for (size_t j = 0; j < byQuery[q].size(); j += lanes) steps += sortedLen[pos[byQuery[q][j]]] + G - 1;
            cost += passes * steps * step_cycles(flavorClass, 3, kPairsR[ri]) * G / 32.0;
        }
        if (fits && cost < bestCost) { bestCost = cost; c->rIndex = ri; }
    }
    if (c->rIndex < 0) { set_error("alphabet too large for the shared-memory query profile"); return false; }
    c->type = type;
    const int R = kPairsR[c->rIndex];
    // Blocks of up to `rounds` tasks per warp: enough blocks that every SM takes several (one is resident at a time), few
    // enough that the profile build is paid for many tasks.
    long long warpTasks = 0;
    for (size_t q = 0; q < byQuery.size(); q++) {
        int G = 1, passes = 1;
        geometry(c->rIndex, queries[q].Q, &G, &passes);
        warpTasks += ((long long)byQuery[q].size() + lanes * (32 / G) - 1) / (lanes * (32 / G));
    }
    const int rounds = (int)std::max<long long>(1, std::min<long long>(4, warpTasks / ((long long)db_.numSMs * warps * 8)));
    long long col = 32, bnd = 0, queryOff = 0;
    std::vector<double> work;
    for (size_t q = 0; q < byQuery.size(); q++) {
        const std::vector<int>& ks = byQuery[q];
        const long long off = queryOff;
        queryOff += std::max(queries[q].Q, 0);
        if (ks.empty()) continue;
        PairQuery pq;
        pq.Q = queries[q].Q;
        geometry(c->rIndex, pq.Q, &pq.G, &pq.passes);
        pq.padTop = s0.mode == kModeNW ? 0 : pq.passes * pq.G * R - pq.Q;  // HW / OV: the last query row at the bottom of the last pass
        pq.queryOff = off;
        const int qIndex = (int)c->queryTab.size();
        c->queryTab.push_back(pq);
        c->maxG = std::max(c->maxG, pq.G);
        c->maxPasses = std::max(c->maxPasses, pq.passes);
        const int firstTask = (int)c->tasks.size();
        for (size_t j = 0; j < ks.size(); j += lanes) {
            PairTask tk;
            const bool two = lanes == 2 && j + 1 < ks.size();
            tk.slot[0] = ks[j]; tk.slot[1] = two ? ks[j + 1] : -1;
            tk.tgt[0] = pos[ks[j]]; tk.tgt[1] = two ? pos[ks[j + 1]] : pos[ks[j]];
            tk.T[0] = sortedLen[tk.tgt[0]]; tk.T[1] = two ? sortedLen[tk.tgt[1]] : 0;
            tk.col = type == 0 ? col : 0;
            if (type == 0) col += tk.T[0] + 32;
            tk.bnd = pq.passes > 1 ? bnd : 0;
            if (pq.passes > 1) bnd += tk.T[0];
            c->tasks.push_back(tk);
        }
        const int nt = (int)c->tasks.size() - firstTask, perRound = warps * (32 / pq.G), per = perRound * rounds;
        for (int k = 0; k < nt; k += per) {
            const int cnt = std::min(per, nt - k);
            c->blocks.push_back({qIndex, firstTask + k, cnt, 0});
            work.push_back((double)pq.passes * (c->tasks[firstTask + k].T[0] + pq.G) * ((cnt + perRound - 1) / perRound));
        }
    }
    c->streamEntries = col + 32;
    c->bndWords = bnd + 32;
    // the heaviest blocks first, so that the last blocks to start are short ones
    std::vector<int> order(c->blocks.size());
    for (size_t k = 0; k < order.size(); k++) order[k] = (int)k;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return work[a] > work[b]; });
    std::vector<PairBlock> sorted(c->blocks.size());
    for (size_t k = 0; k < order.size(); k++) sorted[k] = c->blocks[order[k]];
    c->blocks.swap(sorted);
    return true;
}

// Uploads a class's tables and launches it (16 bits: after the gather of its paired stream).
bool PairsSearch::launch(const Class& c, const std::vector<Scoring>& queries, int wantEnd, const ScoreBounds& b, bool rangeTracking,
                         long long step, long long rangeLo, const Tables& d) {
    const Scoring& s0 = queries[0];
    const int mode = s0.mode, R = kPairsR[c.rIndex];
    const PairQuery* dQueryTab = d.queryTab;
    const PairTask* dTasks = d.tasks;
    const PairBlock* dBlocks = d.blocks;
    PairsParams p;
    memset(&p, 0, sizeof(p));
    if (c.type == 0) {
        uint16_t* dStream = static_cast<uint16_t*>(alloc(sizeof(uint16_t) * (size_t)c.streamEntries));
        if (!dStream) return false;
        if (!launch_gather_pairs(dTasks, (int)c.tasks.size(), db_.dResidues, db_.dOffsets, dStream, stream_)) {
            set_error("gather of the paired stream failed");
            return false;
        }
        p.stream = dStream;
    }
    if (c.maxPasses > 1) {
        p.bndHalf = c.bndWords;
        p.bndH = alloc(2 * sizeof(uint32_t) * (size_t)c.bndWords);
        p.bndF = alloc(2 * sizeof(uint32_t) * (size_t)c.bndWords);
        if (!p.bndH || !p.bndF) return false;
    }
    const int flavor = mode == kModeSW ? (wantEnd ? kFlavorSWEnd : kFlavorSWScore) : kFlavorGlobal;
    const void* fn = pairs_kernel_fn(c.rIndex, c.type, flavor);
    if (!allow_full_smem(db_.device, fn, db_.smemLimit)) return false;
    p.queries = dQueries_; p.matrix = dMatrix_;
    p.A = s0.A; p.gapOpen = s0.Go; p.gapExt = s0.Ge; p.mode = mode; p.wantEnd = wantEnd;
    p.queryTab = dQueryTab; p.blockTab = dBlocks; p.tasks = dTasks;
    p.residues = db_.dResidues; p.offsets = db_.dOffsets;
    p.outScore = dOut_; p.outEndQ = dOut_ + numPairs_; p.outEndT = dOut_ + 2 * (size_t)numPairs_;
    // as launch_group: the SW overflow limit, the "no residue" letter and the range tracking of the 16-bit sweeps
    p.overflowLimit = c.type == 0 ? 32767 - std::max(b.maxEntry, 0) - 1 : (1 << 30);
    p.padLetterScore = c.type == 0 ? (mode == kModeNW ? 0 : -16384) : 0;
    const long long margin = (long long)(R + 3) * step;
    p.rangeHi = rangeTracking ? (int)(32767 - margin) : INT_MAX;
    p.rangeLo = rangeTracking ? (int)(rangeLo + margin) : INT_MIN;
    p.one = 1;
    const size_t smem = (size_t)(c.type == 0 ? 2 : 1) * (s0.A + 1) * ((c.maxG * pairs_rpad(R) + 31) / 32 * 32) * 4;
    void* args[] = {&p};
    CUDA_TRY(cudaLaunchKernel(fn, dim3((unsigned)c.blocks.size()), dim3(kPairsThreads), args, smem, stream_));
    return true;
}

int PairsSearch::run(const std::vector<Scoring>& queries, int wantEnd, int numPairs, const int* pairQuery, const int* pairTarget,
                     const SearchOut& out, float* deviceMs, SearchStats* stats) {
    if (deviceMs) *deviceMs = 0.f;
    if (numPairs <= 0) return 0;
    CUDA_TRY_RC(cudaSetDevice(db_.device));
    const Scoring& s0 = queries[0];  // alphabet, matrix, gaps and mode are the same for every query
    const int Go = s0.Go, Ge = s0.Ge, mode = s0.mode, nq = (int)queries.size();
    const bool isSW = mode == kModeSW;
    ScoreBounds b;
    if (const int rc = s0.validate(&b)) return rc;
    if (s0.A == 256 && *db_.hMaxCode >= 255) b.args16 = false;  // code 255 cannot ride in the 16-bit stream (see search())
    // the routing rule of SearchContext::route and the range limits of SearchContext::Run, for a pair of lengths (Q, T)
    const long long step = (long long)Go + Ge + b.absEntry, rangeLo = mode == kModeNW ? -28000 : -16383;
    const bool rangeTracking = !isSW && b.args16 && 40 * step <= 6000;
    auto fits = [&](int Q, int T, long long lim) {
        const long long lo = 3LL * Go + ((long long)Q + T) * Ge + b.absEntry;
        const long long hi = (b.maxEntry > 0 ? (long long)std::min(Q, T) * b.maxEntry : 0) + Go + b.absEntry;
        return lo <= lim && hi <= lim;
    };
    auto ok16 = [&](int Q, int T) {
        if (isSW) return b.args16;
        if (!rangeTracking) return b.args16 && fits(Q, T, 16000);
        const long long border = (long long)Go + (mode == kModeNW ? (long long)std::max(Q, T) : mode == kModeHW ? (long long)Q : 0LL) * Ge;
        return -border >= rangeLo + 40 * step;
    };
    auto ok32 = [&](int Q, int T) { return isSW ? (b.maxEntry > 0 ? (long long)std::min(Q, T) * b.maxEntry : 0) < (1LL << 30) : fits(Q, T, 1LL << 30); };

    // ---- route every pair, group the classes by query (longest target first)
    std::vector<int> pos((size_t)numPairs);
    std::vector<char> fixed((size_t)numPairs, 0);
    std::vector<std::vector<int>> by16((size_t)nq), by32((size_t)nq);
    for (int k = 0; k < numPairs; k++) {
        const int q = pairQuery[k], p = db_.lay->pos[pairTarget[k]], T = db_.lay->sortedLen[p], Q = queries[q].Q;
        pos[k] = p;
        if (T == 0 || Q <= 0) fixed[k] = 1;  // nothing to align: the defined result, below
        else if (ok16(Q, T)) by16[q].push_back(k);
        else if (ok32(Q, T)) by32[q].push_back(k);
        else return OPAL_B200_ERR_OVERFLOW;
    }
    auto longest_first = [&](std::vector<int>& ks) {
        std::stable_sort(ks.begin(), ks.end(), [&](int a, int c) { return db_.lay->sortedLen[pos[a]] > db_.lay->sortedLen[pos[c]]; });
    };
    bool any16 = false, any32 = false;
    for (int q = 0; q < nq; q++) {
        longest_first(by16[q]); longest_first(by32[q]);
        any16 |= !by16[q].empty(); any32 |= !by32[q].empty();
    }
    SearchStats st;
    numPairs_ = numPairs;
    if (any16 || any32) {
        Class c16;
        if (any16 && !plan(0, queries, wantEnd, by16, pos.data(), &c16)) return OPAL_B200_ERR_CUDA;
        // ---- one upload: [matrix | queries | the 16-bit class's query table, tasks, blocks]
        std::vector<unsigned char> block;
        auto put = [&](const void* src, size_t bytes) {
            const size_t at = block.size();
            block.resize((at + bytes + 15) / 16 * 16, 0);
            if (bytes) memcpy(block.data() + at, src, bytes);
            return at;
        };
        const size_t atMatrix = put(s0.entries, sizeof(int) * (size_t)s0.num_entries());
        const size_t atQueries = block.size();
        for (const Scoring& s : queries)
            if (s.Q > 0) block.insert(block.end(), s.query, s.query + s.Q);  // back to back: PairQuery::queryOff
        put(nullptr, 0);
        // (every part starts on a 16-byte boundary: the tables are found at the offsets put() returns)
        auto put_tables = [&](const Class& c) {
            return std::array<size_t, 3>{put(c.queryTab.data(), sizeof(PairQuery) * c.queryTab.size()),
                                         put(c.tasks.data(), sizeof(PairTask) * c.tasks.size()),
                                         put(c.blocks.data(), sizeof(PairBlock) * c.blocks.size())};
        };
        auto tables_at = [](const unsigned char* dBase, const std::array<size_t, 3>& at) {
            return Tables{reinterpret_cast<const PairQuery*>(dBase + at[0]), reinterpret_cast<const PairTask*>(dBase + at[1]),
                          reinterpret_cast<const PairBlock*>(dBase + at[2])};
        };
        const std::array<size_t, 3> at16 = put_tables(c16);
        unsigned char *dBlock = nullptr, *hBlock = nullptr;
        int* hOut = nullptr;
        if (!event_acquire(db_.device, &evStart_) || !event_acquire(db_.device, &evStop_)) return OPAL_B200_ERR_CUDA;
        if (!upload(block, &dBlock, &hBlock)) return OPAL_B200_ERR_CUDA;
        dMatrix_ = reinterpret_cast<const int*>(dBlock + atMatrix);
        dQueries_ = dBlock + atQueries;
        const size_t outInts = 4 * (size_t)numPairs + 1;
        if (!(dOut_ = static_cast<int*>(alloc(sizeof(int) * outInts)))) return OPAL_B200_ERR_CUDA;
        if (!pinned_alloc((void**)&hOut, sizeof(int) * outInts)) return OPAL_B200_ERR_CUDA;
        pinned_.push_back(hOut);
        int* dCount = dOut_ + 3 * (size_t)numPairs;
        CUDA_TRY_RC(cudaMemsetAsync(dOut_, 0, sizeof(int) * (3 * (size_t)numPairs + 1), stream_));  // (0 is never "re-run me")
        CUDA_TRY_RC(cudaEventRecord(evStart_, stream_));
        // ---- 16 bits, then the collection of what they could not hold
        if (any16) {
            if (!launch(c16, queries, wantEnd, b, rangeTracking, step, rangeLo, tables_at(dBlock, at16))) return OPAL_B200_ERR_CUDA;
            st.kernelLaunches += 2;
            st.R = kPairsR[c16.rIndex]; st.G = c16.maxG; st.passes = c16.maxPasses; st.warpsPerPartition = 3; st.groups = 1;
            collect_flagged_kernel<<<std::min(db_.numSMs * 4, (numPairs + 255) / 256), 256, 0, stream_>>>(dOut_, numPairs, dCount + 1, dCount);
            CUDA_TRY_RC(cudaGetLastError());
            CUDA_TRY_RC(cudaMemcpyAsync(hOut, dCount, sizeof(int), cudaMemcpyDeviceToHost, stream_));
            CUDA_TRY_RC(cudaStreamSynchronize(stream_));
            const int flagged = hOut[0];
            if (flagged > 0) {
                CUDA_TRY_RC(cudaMemcpyAsync(hOut, dCount + 1, sizeof(int) * (size_t)flagged, cudaMemcpyDeviceToHost, stream_));
                CUDA_TRY_RC(cudaStreamSynchronize(stream_));
                std::vector<char> touched((size_t)nq, 0);
                for (int f = 0; f < flagged; f++) { const int k = hOut[f]; by32[pairQuery[k]].push_back(k); touched[pairQuery[k]] = 1; }
                for (int q = 0; q < nq; q++) if (touched[q]) longest_first(by32[q]);
                any32 = true;
                st.rerun32 = flagged;
            }
        }
        // ---- 32 bits: the pairs routed there and the re-runs
        if (any32) {
            Class c32;
            if (!plan(1, queries, wantEnd, by32, pos.data(), &c32)) return OPAL_B200_ERR_CUDA;
            block.clear();
            const std::array<size_t, 3> at32 = put_tables(c32);
            unsigned char *dPlan32 = nullptr, *hPlan32 = nullptr;
            if (!upload(block, &dPlan32, &hPlan32)) return OPAL_B200_ERR_CUDA;
            if (!launch(c32, queries, wantEnd, b, rangeTracking, step, rangeLo, tables_at(dPlan32, at32))) return OPAL_B200_ERR_CUDA;
            st.kernelLaunches++;
        }
        CUDA_TRY_RC(cudaEventRecord(evStop_, stream_));
        // ---- the per-pair results back in one copy
        CUDA_TRY_RC(cudaMemcpyAsync(hOut, dOut_, sizeof(int) * (wantEnd ? 3 : 1) * (size_t)numPairs, cudaMemcpyDeviceToHost, stream_));
        CUDA_TRY_RC(cudaStreamSynchronize(stream_));
        if (deviceMs) CUDA_TRY_RC(cudaEventElapsedTime(deviceMs, evStart_, evStop_));
        for (int k = 0; k < numPairs; k++)
            if (!fixed[k] && (hOut[k] == kScoreOverflow || hOut[k] == kScoreNone)) return OPAL_B200_ERR_OVERFLOW;
        const int *hEndQ = hOut + numPairs, *hEndT = hOut + 2 * (size_t)numPairs;
        for (int k = 0; k < numPairs; k++)
            if (!fixed[k])
                out.put(k, hOut[k], (wantEnd && hEndQ[k] != 0x7fffffff) ? hEndQ[k] : -1, (wantEnd && hEndT[k] != 0x7fffffff) ? hEndT[k] : -1);
    }
    for (int k = 0; k < numPairs; k++) {
        if (!fixed[k]) continue;
        const int Q = queries[pairQuery[k]].Q, T = db_.lay->sortedLen[pos[k]];
        int sc = 0, eq = Q - 1, et = T - 1;  // as SearchContext::route (oracle/opal_oracle.c)
        if (Q > 0 && (mode == kModeNW || mode == kModeHW)) sc = -Go - (Q - 1) * Ge;
        else if (Q <= 0 && T > 0 && mode == kModeNW) sc = -Go - (T - 1) * Ge;
        if (isSW) { eq = -1; et = -1; }
        out.put(k, sc, wantEnd ? eq : -1, wantEnd ? et : -1);
    }
    if (stats) *stats = st;
    return 0;
}

int DeviceDb::search_pairs(const std::vector<Scoring>& queries, int wantEnd, int numPairs, const int* pairQuery, const int* pairTarget,
                           const SearchOut& out, float* deviceMs) {
    if (cudaSetDevice(db_.device) != cudaSuccess) { set_error("cudaSetDevice failed"); return OPAL_B200_ERR_CUDA; }
    if (!ensure_uploaded()) return OPAL_B200_ERR_CUDA;
    SearchStats st;
    int rc;
    {
        PairsSearch ps(db_, stream());
        rc = ps.run(queries, wantEnd, numPairs, pairQuery, pairTarget, out, deviceMs, &st);
    }
    contexts_[0]->stats_ = st;
    return rc;
}

// ------------------------------------------------------------------ DPX roofline probe
double measure_dpx_peak(int device, int mix, double* threadInstrPerSec, float* msOut) {
    constexpr int ILP = 8;
    const int iters = 4096;
    if (cudaSetDevice(device) != cudaSuccess) { set_error("cudaSetDevice failed"); return 0.0; }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    const int blocks = prop.multiProcessorCount * 2;
    uint32_t* out = nullptr;
    if (cudaMalloc(&out, sizeof(uint32_t) * blocks * 512) != cudaSuccess) { set_error("cudaMalloc failed"); return 0.0; }
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(a);
        if (mix == 0) dpx_peak_kernel<ILP, 0><<<blocks, 512>>>(out, iters, 12345u + rep);
        else dpx_peak_kernel<ILP, 1><<<blocks, 512>>>(out, iters, 12345u + rep);
        cudaEventRecord(b);
        cudaEventSynchronize(b);
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        if (rep > 0) best = std::min(best, ms);
    }
    const cudaError_t e = cudaGetLastError();
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(out);
    if (e != cudaSuccess) { set_error(cudaGetErrorString(e)); return 0.0; }
    const double perPair = mix == 0 ? 6.0 : 5.0;  // packed instructions per cell pair: SW / NW-HW-OV (SURVEY.md 8d)
    const double instr = perPair * ILP * (double)iters * blocks * 512;  // thread-level packed instructions
    const double ips = instr / (best * 1e-3);
    if (threadInstrPerSec) *threadInstrPerSec = ips;
    if (msOut) *msOut = best;
    return ips * 2.0 / perPair / 1e9;  // 2 cells per packed instruction
}

}  // namespace opalb200
