// api.cu -- the C ABI of libopal_b200.so: opal.h (drop-in) and opal_b200.h (resident handle).
//
// opalSearchDatabase mirrors reference src/opal.cpp:1435-1519 step by step -- skip mask from
// prefilled records, score/end search, early return on error, then either the alignment stage
// or the "no alignment" field fill -- with the SIMD passes replaced by DeviceDb::search.
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/opal.h"
#include "../../include/opal_b200.h"
#include "align.h"
#include "engine.h"

using namespace opalb200;

// The CUDA "current device" is per-thread state of the caller: entry points put it back on return.
struct DeviceGuard {
    int saved = -1;
    DeviceGuard() { if (cudaGetDevice(&saved) != cudaSuccess) saved = -1; }
    ~DeviceGuard() { if (saved >= 0) cudaSetDevice(saved); }
};

// Searches in flight (batches, slices, devices) each use streams of their own; the driver multiplexes streams onto
// CUDA_DEVICE_MAX_CONNECTIONS hardware queues (8 by default), and streams that share a queue wait for each other's
// launches -- measured on an eighth of BASELINE configs[2] with twelve searches in flight: 4,790 GCUPS with 8 queues,
// 5,190 with 32.  The variable is read when the process initialises CUDA, so it is set when the library is loaded,
// unless the host application has chosen a value itself.
__attribute__((constructor)) static void opalb200_on_load() { setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0); }

static int default_device() {
    const char* e = getenv("OPAL_B200_DEVICE");
    return e ? atoi(e) : 0;
}

// ------------------------------------------------------------------ several devices behind one call
// Every (query, target) pair is independent (SURVEY.md section 8e): a database is dealt over the devices, each device
// searches its shard on a host thread and streams of its own, results come back by per-device copies and are
// scattered into the caller's arrays by an index map.  No collective, no peer traffic.

// Devices of the drop-in entry points (they take no device argument): OPAL_B200_DEVICES = "all" or a comma-separated
// list of ordinals; otherwise the single device OPAL_B200_DEVICE (default 0).
static std::vector<int> env_devices() {
    std::vector<int> devs;
    if (const char* e = getenv("OPAL_B200_DEVICES")) {
        if (!strcmp(e, "all")) {
            int count = 0;
            if (cudaGetDeviceCount(&count) != cudaSuccess) count = 0;
            for (int d = 0; d < count; d++) devs.push_back(d);
        } else {
            for (const char* p = e; *p;) {
                char* end = nullptr;
                const long d = strtol(p, &end, 10);
                if (end == p) break;
                if (d >= 0) devs.push_back((int)d);  // an ordinal may repeat: several shards on one device (used by the tests)
                p = *end ? end + 1 : end;
            }
        }
    }
    if (devs.empty()) devs.push_back(default_device());
    return devs;
}

// fn(s) for every shard, each on a host thread of its own (the caller runs shard 0); returns the first non-zero
// code in shard order and leaves that shard's error text with the calling thread.
template <class F>
static int on_shards(int parts, F fn) {
    if (parts == 1) return fn(0);
    std::vector<int> rc((size_t)parts, 0);
    std::vector<std::string> err((size_t)parts);
    std::vector<std::thread> th;
    for (int s = 1; s < parts; s++)
        th.emplace_back([&, s] {
            DeviceGuard guard;
            rc[s] = fn(s);
            if (rc[s]) err[s] = last_error();
        });
    rc[0] = fn(0);
    if (rc[0]) err[0] = last_error();
    for (auto& t : th) t.join();
    for (int s = 0; s < parts; s++)
        if (rc[s]) { set_error(err[s]); return rc[s]; }
    return 0;
}

// The object behind an OpalB200Db handle: one resident shard per device.
struct DbHandle {
    std::vector<DeviceDb*> shards;
    std::vector<std::vector<int>> index;  // [shard][local index] -> caller index; empty when one shard holds everything
    int n = 0;
    long long residues = 0;
    SearchStats stats;  // last search: launches / re-runs summed over the shards, geometry of shard 0
    ~DbHandle() { for (DeviceDb* d : shards) delete d; }
    int parts() const { return (int)shards.size(); }
    int caller_index(int s, int local) const { return index.empty() ? local : index[s][local]; }
    void collect_stats() {
        stats = shards[0]->stats();
        for (size_t s = 1; s < shards.size(); s++) {
            stats.kernelLaunches += shards[s]->stats().kernelLaunches;
            stats.rerun32 += shards[s]->stats().rerun32;
            stats.foldedTasks += shards[s]->stats().foldedTasks;
            stats.chainedTasks += shards[s]->stats().chainedTasks;
        }
    }
};

// Shards of `n` scattered sequences on `devices`: NULL (error text set) on failure.
static DbHandle* create_handle(unsigned char* const* db, int n, const int* lens, const std::vector<int>& devices,
                               const int* callerIndex = nullptr) {
    DbHandle* h = new DbHandle();
    h->n = n;
    const int parts = (int)std::max<size_t>(1, std::min<size_t>(devices.size(), (size_t)std::max(n / 2, 1)));
    h->shards.assign((size_t)parts, nullptr);
    if (parts == 1 && !callerIndex) {
        h->shards[0] = DeviceDb::create(db, n, lens, devices[0]);
        if (!h->shards[0]) { delete h; return nullptr; }
        h->residues = h->shards[0]->residues();
        return h;
    }
    std::shared_ptr<const Layout> lay = layout_for(lens, nullptr, n, false, nullptr);
    if (!lay) { delete h; return nullptr; }
    h->index = *lay->parts(parts, 1);  // dealt in length order: equal residue counts, equal length mix (engine.cu, Layout::parts)
    if (callerIndex)  // keep every shard in ascending CALLER index (ties between equal scores are broken by it, on the device too)
        for (auto& v : h->index) std::sort(v.begin(), v.end(), [&](int a, int b) { return callerIndex[a] < callerIndex[b]; });
    const int rc = on_shards(parts, [&](int s) -> int {
        const std::vector<int>& idx = h->index[s];
        std::vector<unsigned char*> ptr(idx.size());
        std::vector<int> len(idx.size());
        for (size_t k = 0; k < idx.size(); k++) { ptr[k] = db[idx[k]]; len[k] = lens[idx[k]]; }
        h->shards[s] = DeviceDb::create(ptr.data(), (int)idx.size(), len.data(), devices[s]);
        return h->shards[s] ? 0 : OPAL_ERR_NO_SIMD_SUPPORT;
    });
    if (rc) { delete h; return nullptr; }
    for (DeviceDb* d : h->shards) h->residues += d->residues();
    if (callerIndex)  // the sequences came in an order of their own (packed database): translate to the caller's
        for (auto& v : h->index)
            for (int& i : v) i = callerIndex[i];
    return h;
}

extern "C" {

void opalInitSearchResult(OpalSearchResult* r) {  // reference src/opal.cpp:1549-1555
    r->scoreSet = 0;
    r->startLocationTarget = r->startLocationQuery = -1;
    r->endLocationTarget = r->endLocationQuery = -1;
    r->alignment = NULL;
    r->alignmentLength = 0;
}

int opalSearchResultIsEmpty(const OpalSearchResult r) { return !r.scoreSet; }  // :1557-1559

void opalSearchResultSetScore(OpalSearchResult* r, int score) {  // :1561-1564
    r->scoreSet = 1;
    r->score = score;
}

// Orders the database uploads of the slices of one device (see opalSearchDatabase).
struct CreateGate {
    std::mutex mu;
    std::condition_variable cv;
    int next = 0;
    void enter(int ticket) { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return next == ticket; }); }
    void leave() { { std::lock_guard<std::mutex> lk(mu); next++; } cv.notify_all(); }
};

// The body of opalSearchDatabase once the database is (or can be made) resident.  `ddb` may be NULL: it is
// then created from db / dbSeqLengths if any entry needs work.  db / dbSeqLengths may be NULL for handle calls.
static int search_into_results(DeviceDb* ddb, const Scoring& s, unsigned char* const* db, int dbLength, const int* dbSeqLengths,
                               OpalSearchResult* results[], const int searchType, int device, CreateGate* gate = nullptr, int ticket = 0) {
    if (!valid_mode(s.mode)) return OPAL_ERR_INVALID_MODE;  // :1469-1473, results untouched
    if (dbLength <= 0) return 0;

    // Entries that already hold what this search level needs are not recomputed (:1446-1451).
    // (The loops over all records run on the host pool for large databases: half a million 40-byte records cost
    // milliseconds per pass on one core.)
    std::vector<unsigned char> skip(dbLength);
    std::atomic<bool> anyWorkFlag(false);
    parallel_for(dbLength, 65536, [&](long long lo, long long hi) {
        bool any = false;
        for (long long i = lo; i < hi; i++) {
            const OpalSearchResult* r = results[i];
            skip[i] = r->scoreSet && (searchType == OPAL_SEARCH_SCORE || (r->endLocationQuery >= 0 && r->endLocationTarget >= 0));
            any |= !skip[i];
        }
        if (any) anyWorkFlag.store(true);
    });
    const bool anyWork = anyWorkFlag.load();
    const int wantEnd = searchType != OPAL_SEARCH_SCORE;
    const bool trace = getenv("OPAL_B200_TRACE") != nullptr;  // phase timings of the call on stderr
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::milli>(b - a).count();
    };
    const auto t0 = now();
    DeviceDb* owned = nullptr;
    if (gate) gate->enter(ticket);  // slices of one device stage and upload in order: the first one's data must land first
    if (!ddb && (anyWork || searchType == OPAL_SEARCH_ALIGNMENT)) ddb = owned = DeviceDb::create(db, dbLength, dbSeqLengths, device);
    if (gate) gate->leave();
    if (!ddb && (anyWork || searchType == OPAL_SEARCH_ALIGNMENT)) return OPAL_ERR_NO_SIMD_SUPPORT;
    const auto t1 = now();
    int status = 0;
    if (anyWork)  // results go straight into the records (same pass also sets the no-alignment fields, :1508-1515)
        status = ddb->search(s, wantEnd, skip.data(), SearchOut::into(results, searchType != OPAL_SEARCH_ALIGNMENT), nullptr);
    const auto t2 = now();
    if (status == 0 && searchType == OPAL_SEARCH_ALIGNMENT)
        status = align_database(ddb, {{&s, results, dbLength, nullptr}}, db, dbSeqLengths);
    const auto t3 = now();
    delete owned;
    if (trace)
        fprintf(stderr, "[opal-b200] pack+upload %.3f ms, search %.3f ms, alignment %.3f ms, release %.3f ms\n", ms(t0, t1), ms(t1, t2),
                ms(t2, t3), ms(t3, now()));
    if (status) return status;  // :1473
    if (searchType != OPAL_SEARCH_ALIGNMENT) {  // :1508-1515: every entry, skipped ones included (the others were done above)
        parallel_for(dbLength, 65536, [&](long long lo, long long hi) {
            for (long long i = lo; i < hi; i++) {
                if (anyWork && !skip[i]) continue;
                results[i]->alignment = NULL;
                results[i]->alignmentLength = -1;
                results[i]->startLocationQuery = -1;
                results[i]->startLocationTarget = -1;
            }
        });
    }
    return 0;
}

int opalSearchDatabase(unsigned char query[], int queryLength, unsigned char* db[], int dbLength, int dbSeqLengths[],
                       int gapOpen, int gapExt, int* scoreMatrix, int alphabetLength, OpalSearchResult* results[],
                       const int searchType, int mode, int overflowMethod) {
    DeviceGuard guard;
    (void)overflowMethod;  // OPAL_OVERFLOW_SIMPLE / _BUCKETS only schedule the reference's passes; results are equal
    const std::vector<int> devices = env_devices();
    const int D = (int)std::min<size_t>(devices.size(), (size_t)std::max(dbLength / 2, 1));
    const bool modeOk = valid_mode(mode);
    const Scoring scoring = Scoring::with_matrix(query, queryLength, scoreMatrix, alphabetLength, gapOpen, gapExt, mode);
    // A large database is cut into a few SLICES per device (longest sequences first) that are staged, uploaded and
    // searched as databases of their own, each on a host thread and streams of its own: the first slice is being
    // searched while the others are still on their way, and a slice's records are written while the next one's kernels
    // run -- per call, the staging, the copies and the result writes then overlap the kernels instead of preceding
    // and following them.
    long long total = 0;
    for (int i = 0; i < dbLength && modeOk; i++) total += dbSeqLengths[i] > 0 ? dbSeqLengths[i] : 0;
    // Measured on BASELINE configs[2] (60 calls, 16 host threads): the whole database on one device (207 M residues) gains
    // 9 % from four slices; half of it (104 M) is indifferent; a quarter (52 M) LOSES 13 % with three and an eighth 33 %
    // with two -- every slice is a search of its own (plans, passes, launches), which a short search does not win back.
    int K = total / std::max(D, 1) >= (144LL << 20) ? 4 : 1;
    if (const char* e = getenv("OPAL_B200_SLICES")) K = std::max(1, std::min(atoi(e), 16));
    K = std::min(K, std::max(dbLength / (2 * std::max(D, 1)), 1));
    if (D * K <= 1 || !modeOk)
        return search_into_results(nullptr, scoring, db, dbLength, dbSeqLengths, results, searchType, devices[0]);
    // One call = the whole database (reference src/opal.h:150-154), on every listed device: each searches the parts
    // dealt to it and fills the caller's records of those parts; the alignment stage stays on the owning device.
    std::shared_ptr<const Layout> lay = layout_for(dbSeqLengths, nullptr, dbLength, false, nullptr);
    if (!lay) return OPAL_ERR_NO_SIMD_SUPPORT;
    const std::shared_ptr<const std::vector<std::vector<int>>> parts = lay->parts(D, K);
    std::vector<CreateGate> gates((size_t)D);
    return on_shards(D * K, [&](int s) -> int {
        const int d = s / K, k = s % K;
        const std::vector<int>& idx = (*parts)[(size_t)s];
        if (idx.empty()) {  // nothing dealt to this slice: let the next one through
            if (K > 1) { gates[d].enter(k); gates[d].leave(); }
            return 0;
        }
        std::vector<unsigned char*> ptr(idx.size());
        std::vector<int> len(idx.size());
        std::vector<OpalSearchResult*> res(idx.size());
        for (size_t j = 0; j < idx.size(); j++) { ptr[j] = db[idx[j]]; len[j] = dbSeqLengths[idx[j]]; res[j] = results[idx[j]]; }
        set_thread_overlapped(k + 1 < K);  // other slices follow on this device: plan for throughput, not for the last task's end
        const int rc = search_into_results(nullptr, scoring, ptr.data(), (int)idx.size(), len.data(), res.data(), searchType, devices[d],
                                           K > 1 ? &gates[d] : nullptr, k);
        set_thread_overlapped(false);
        return rc;
    });
}

int opalSearchDatabaseRescore(unsigned char query[], int queryLength, unsigned char* db[], int dbLength, int dbSeqLengths[],
                              int gapOpen, int gapExt, int* scoreMatrix, int alphabetLength, OpalSearchResult* results[],
                              const int searchType, int mode, int overflowMethod) {
    return opalSearchDatabase(query, queryLength, db, dbLength, dbSeqLengths, gapOpen, gapExt, scoreMatrix, alphabetLength,
                              results, searchType, mode, overflowMethod);
}

int opalSearchDatabaseCharSW(unsigned char query[], int queryLength, unsigned char** db, int dbLength, int dbSeqLengths[],
                             int gapOpen, int gapExt, int* scoreMatrix, int alphabetLength, OpalSearchResult* results[]) {
    DeviceGuard guard;
    // reference src/opal.cpp:1522-1546: SW scores that fit 8 bits; the others come back unset (-1).
    if (dbLength <= 0) return 0;
    bool argsFit = !(gapOpen < -128 || 127 < gapOpen || gapExt < -128 || 127 < gapExt);  // :178-180
    for (int i = 0; argsFit && i < alphabetLength * alphabetLength; i++)
        if (scoreMatrix[i] < -128 || 127 < scoreMatrix[i]) argsFit = false;               // :188-193
    std::vector<int> sc(dbLength, -1);
    int rc = argsFit ? 0 : OPAL_ERR_OVERFLOW;
    if (argsFit) {
        DeviceDb* ddb = DeviceDb::create(db, dbLength, dbSeqLengths, env_devices()[0]);
        if (!ddb) return OPAL_ERR_NO_SIMD_SUPPORT;
        const int st = ddb->search(Scoring::with_matrix(query, queryLength, scoreMatrix, alphabetLength, gapOpen, gapExt, OPAL_MODE_SW), 0,
                                   nullptr, SearchOut::arrays(sc.data(), nullptr, nullptr), nullptr);
        delete ddb;
        if (st == OPAL_ERR_NO_SIMD_SUPPORT) return st;
        if (st) std::fill(sc.begin(), sc.end(), -1);
    }
    for (int i = 0; i < dbLength; i++) {
        if (argsFit && sc[i] >= 0 && sc[i] <= 127) {
            opalSearchResultSetScore(results[i], sc[i]);
            results[i]->endLocationQuery = results[i]->endLocationTarget = -1;  // :423-426
        } else {
            results[i]->score = -1;  // :1538-1541
            results[i]->scoreSet = 0;
            rc = OPAL_ERR_OVERFLOW;
        }
    }
    return rc;
}

// ------------------------------------------------------------------ opal_b200.h
// Arguments only the PSSM entry points have: the PSSM itself, and -- for OPAL_SEARCH_ALIGNMENT -- the residues it was
// built for, which label the diagonal steps of an alignment MATCH / MISMATCH.  0 or OPAL_ERR_INVALID_ARGUMENT.
static int check_pssm_args(const int* pssm, const unsigned char* query, int queryLength, int alphabetLength, int searchType) {
    if (!pssm && queryLength > 0) { set_error("pssm is NULL"); return OPAL_ERR_INVALID_ARGUMENT; }
    if (searchType == OPAL_SEARCH_ALIGNMENT && queryLength > 0) {
        if (!query) { set_error("OPAL_SEARCH_ALIGNMENT with a PSSM needs the query residues"); return OPAL_ERR_INVALID_ARGUMENT; }
        for (int r = 0; r < queryLength; r++)
            if (query[r] >= alphabetLength) { set_error("query holds residue codes >= alphabetLength"); return OPAL_ERR_INVALID_ARGUMENT; }
    }
    return 0;
}

int opalb200_device_count(void) {
    int n = 0;
    return cudaGetDeviceCount(&n) == cudaSuccess ? n : 0;
}

const char* opalb200_last_error(void) { return last_error(); }

void opalb200_trim_cache(void) {
    DeviceGuard guard;
    trim_cache();
    trim_layouts();
}

OpalB200Db* opalb200_db_create(unsigned char* db[], int dbLength, const int dbSeqLengths[], int device) {
    DeviceGuard guard;
    if (dbLength < 0 || (dbLength > 0 && (!db || !dbSeqLengths))) { set_error("invalid database"); return nullptr; }
    const std::vector<int> devices = device >= 0 ? std::vector<int>(1, device) : env_devices();
    return reinterpret_cast<OpalB200Db*>(create_handle(db, dbLength, dbSeqLengths, devices));
}

OpalB200Db* opalb200_db_create_multi(unsigned char* db[], int dbLength, const int dbSeqLengths[], const int devices[], int numDevices) {
    DeviceGuard guard;
    if (dbLength < 0 || (dbLength > 0 && (!db || !dbSeqLengths))) { set_error("invalid database"); return nullptr; }
    std::vector<int> devs;
    for (int k = 0; devices && k < numDevices; k++) devs.push_back(devices[k]);  // an ordinal may repeat (several shards on one device)
    if (devs.empty()) devs = env_devices();
    return reinterpret_cast<OpalB200Db*>(create_handle(db, dbLength, dbSeqLengths, devs));
}

OpalB200Db* opalb200_db_create_sorted(const unsigned char* residues, const int sortedLengths[], const int order[], int dbLength,
                                      int device) {
    DeviceGuard guard;
    if (dbLength < 0 || (dbLength > 0 && (!residues || !sortedLengths))) { set_error("invalid packed database"); return nullptr; }
    const std::vector<int> devices = device >= 0 ? std::vector<int>(1, device) : env_devices();
    if (devices.size() == 1) {
        DeviceDb* d = DeviceDb::create_sorted(residues, sortedLengths, order, dbLength, devices[0]);
        if (!d) return nullptr;
        DbHandle* h = new DbHandle();
        h->shards.push_back(d); h->n = dbLength; h->residues = d->residues();
        return reinterpret_cast<OpalB200Db*>(h);
    }
    // several devices: the packed sequences are dealt like scattered ones (pointers into the packed buffer)
    std::vector<unsigned char*> ptr((size_t)dbLength);
    size_t off = 0;
    for (int p = 0; p < dbLength; p++) {
        if (sortedLengths[p] < 0 || (p > 0 && sortedLengths[p] > sortedLengths[p - 1])) { set_error("packed database is not sorted longest first"); return nullptr; }
        ptr[p] = const_cast<unsigned char*>(residues) + off;
        off += (size_t)sortedLengths[p];
    }
    if (order) {  // must be a permutation of 0..n-1
        std::vector<char> seen((size_t)std::max(dbLength, 1), 0);
        for (int p = 0; p < dbLength; p++) {
            if (order[p] < 0 || order[p] >= dbLength || seen[order[p]]) { set_error("packed database: order[] is not a permutation"); return nullptr; }
            seen[order[p]] = 1;
        }
    }
    return reinterpret_cast<OpalB200Db*>(create_handle(ptr.data(), dbLength, sortedLengths, devices, order));
}

void opalb200_db_destroy(OpalB200Db* h) {
    DeviceGuard guard;
    delete reinterpret_cast<DbHandle*>(h);
}

int opalb200_db_length(const OpalB200Db* h) { return reinterpret_cast<const DbHandle*>(h)->n; }

long long opalb200_db_residues(const OpalB200Db* h) { return reinterpret_cast<const DbHandle*>(h)->residues; }

int opalb200_db_devices(const OpalB200Db* h) { return reinterpret_cast<const DbHandle*>(h)->parts(); }

static int db_search(OpalB200Db* hh, const Scoring& scoring, int searchType, const unsigned char* skip, int* scores, int* endQuery,
                     int* endTarget, float* deviceMs) {
    if (!hh || !scores) return OPAL_ERR_NO_SIMD_SUPPORT;
    DeviceGuard guard;
    DbHandle* h = reinterpret_cast<DbHandle*>(hh);
    const int wantEnd = searchType != OPAL_SEARCH_SCORE && endQuery && endTarget;
    if (h->index.empty()) {
        const int rc = h->shards[0]->search(scoring, wantEnd, skip, SearchOut::arrays(scores, endQuery, endTarget), deviceMs);
        h->collect_stats();
        return rc;
    }
    std::vector<float> ms((size_t)h->parts(), 0.f);
    const int rc = on_shards(h->parts(), [&](int s) -> int {
        const std::vector<int>& idx = h->index[s];
        const size_t m = idx.size();
        std::vector<int> sc(m), eq(m, -1), et(m, -1);
        std::vector<unsigned char> sk;
        if (skip) { sk.resize(m); for (size_t k = 0; k < m; k++) sk[k] = skip[idx[k]]; }
        const int r = h->shards[s]->search(scoring, wantEnd, skip ? sk.data() : nullptr, SearchOut::arrays(sc.data(), eq.data(), et.data()),
                                           &ms[s]);
        if (r) return r;
        for (size_t k = 0; k < m; k++) {
            if (skip && sk[k]) continue;
            scores[idx[k]] = sc[k];
            if (endQuery) endQuery[idx[k]] = eq[k];
            if (endTarget) endTarget[idx[k]] = et[k];
        }
        return 0;
    });
    if (deviceMs) *deviceMs = *std::max_element(ms.begin(), ms.end());  // the devices run concurrently
    h->collect_stats();
    return rc;
}

int opalb200_db_search(OpalB200Db* hh, const unsigned char query[], int queryLength, int gapOpen, int gapExt,
                       const int* scoreMatrix, int alphabetLength, int searchType, int mode, const unsigned char* skip,
                       int* scores, int* endQuery, int* endTarget, float* deviceMs) {
    return db_search(hh, Scoring::with_matrix(query, queryLength, scoreMatrix, alphabetLength, gapOpen, gapExt, mode), searchType, skip,
                     scores, endQuery, endTarget, deviceMs);
}

int opalb200_db_search_pssm(OpalB200Db* hh, const int* pssm, int queryLength, int alphabetLength, int gapOpen, int gapExt,
                            int searchType, int mode, const unsigned char* skip, int* scores, int* endQuery, int* endTarget,
                            float* deviceMs) {
    if (deviceMs) *deviceMs = 0.f;
    if (const int rc = check_pssm_args(pssm, nullptr, queryLength, alphabetLength, OPAL_SEARCH_SCORE)) return rc;
    return db_search(hh, Scoring::with_pssm(nullptr, pssm, queryLength, alphabetLength, gapOpen, gapExt, mode), searchType, skip, scores,
                     endQuery, endTarget, deviceMs);
}

// The batch entry points once their searches are built: outputs are [search][caller index].
static int db_search_batch(OpalB200Db* hh, const std::vector<Scoring>& searches, int searchType, int* scores, int* endQuery,
                           int* endTarget, int inFlight, float* batchMs) {
    if (!hh || !scores) return OPAL_ERR_NO_SIMD_SUPPORT;
    DeviceGuard guard;
    DbHandle* h = reinterpret_cast<DbHandle*>(hh);
    const int wantEnd = searchType != OPAL_SEARCH_SCORE && endQuery && endTarget;
    const int fl = inFlight <= 0 ? 3 : inFlight;
    if (h->index.empty()) {
        const int rc = h->shards[0]->search_batch(searches, wantEnd, scores, endQuery, endTarget, fl, batchMs);
        h->collect_stats();
        return rc;
    }
    std::vector<float> ms((size_t)h->parts(), 0.f);
    const size_t n = (size_t)h->n;
    const int rc = on_shards(h->parts(), [&](int s) -> int {
        const std::vector<int>& idx = h->index[s];
        const size_t m = idx.size(), all = m * searches.size();
        std::vector<int> sc(all), eq(wantEnd ? all : 0), et(wantEnd ? all : 0);
        const int r = h->shards[s]->search_batch(searches, wantEnd, sc.data(), wantEnd ? eq.data() : nullptr, wantEnd ? et.data() : nullptr,
                                                 fl, &ms[s]);
        if (r) return r;
        for (size_t q = 0; q < searches.size(); q++)
            for (size_t k = 0; k < m; k++) {
                const size_t to = q * n + (size_t)idx[k], from = q * m + k;
                scores[to] = sc[from];
                if (endQuery) endQuery[to] = wantEnd ? eq[from] : -1;
                if (endTarget) endTarget[to] = wantEnd ? et[from] : -1;
            }
        return 0;
    });
    if (batchMs) *batchMs = *std::max_element(ms.begin(), ms.end());
    h->collect_stats();
    return rc;
}

int opalb200_db_search_batch(OpalB200Db* hh, int numQueries, const unsigned char* const queries[], const int queryLengths[],
                             int gapOpen, int gapExt, const int* scoreMatrix, int alphabetLength, int searchType, int mode,
                             int* scores, int* endQuery, int* endTarget, int inFlight, float* batchMs) {
    if (numQueries > 0 && (!queries || !queryLengths)) return OPAL_ERR_NO_SIMD_SUPPORT;
    std::vector<Scoring> searches;
    for (int q = 0; q < numQueries; q++)
        searches.push_back(Scoring::with_matrix(queries[q], queryLengths[q], scoreMatrix, alphabetLength, gapOpen, gapExt, mode));
    return db_search_batch(hh, searches, searchType, scores, endQuery, endTarget, inFlight, batchMs);
}

int opalb200_db_search_batch_modes(OpalB200Db* hh, int numSearches, const unsigned char* const queries[], const int queryLengths[],
                                   const int modes[], int gapOpen, int gapExt, const int* scoreMatrix, int alphabetLength,
                                   int searchType, int* scores, int* endQuery, int* endTarget, int inFlight, float* batchMs) {
    if (numSearches > 0 && !modes) return OPAL_ERR_INVALID_MODE;
    for (int q = 0; q < numSearches; q++)
        if (!valid_mode(modes[q])) return OPAL_ERR_INVALID_MODE;
    if (numSearches > 0 && (!queries || !queryLengths)) return OPAL_ERR_NO_SIMD_SUPPORT;
    std::vector<Scoring> searches;
    for (int q = 0; q < numSearches; q++)
        searches.push_back(Scoring::with_matrix(queries[q], queryLengths[q], scoreMatrix, alphabetLength, gapOpen, gapExt, modes[q]));
    return db_search_batch(hh, searches, searchType, scores, endQuery, endTarget, inFlight, batchMs);
}

int opalb200_db_search_batch_pssm(OpalB200Db* hh, int numSearches, const int* const pssms[], const int queryLengths[], const int modes[],
                                  int alphabetLength, int gapOpen, int gapExt, int searchType, int* scores, int* endQuery,
                                  int* endTarget, int inFlight, float* batchMs) {
    if (batchMs) *batchMs = 0.f;
    if (numSearches > 0 && !modes) return OPAL_ERR_INVALID_MODE;
    if (numSearches > 0 && (!pssms || !queryLengths)) { set_error("pssms / queryLengths is NULL"); return OPAL_ERR_INVALID_ARGUMENT; }
    for (int q = 0; q < numSearches; q++)
        if (!valid_mode(modes[q])) return OPAL_ERR_INVALID_MODE;
    std::vector<Scoring> searches;
    for (int q = 0; q < numSearches; q++) {
        if (const int rc = check_pssm_args(pssms[q], nullptr, queryLengths[q], alphabetLength, OPAL_SEARCH_SCORE)) return rc;
        searches.push_back(Scoring::with_pssm(nullptr, pssms[q], queryLengths[q], alphabetLength, gapOpen, gapExt, modes[q]));
    }
    return db_search_batch(hh, searches, searchType, scores, endQuery, endTarget, inFlight, batchMs);
}

static int db_search_results(OpalB200Db* hh, const Scoring& scoring, OpalSearchResult* results[], int searchType) {
    if (!hh || !results) return OPAL_ERR_NO_SIMD_SUPPORT;
    DeviceGuard guard;
    DbHandle* h = reinterpret_cast<DbHandle*>(hh);
    if (h->index.empty())
        return search_into_results(h->shards[0], scoring, nullptr, h->n, nullptr, results, searchType, h->shards[0]->device());
    if (!valid_mode(scoring.mode)) return OPAL_ERR_INVALID_MODE;
    return on_shards(h->parts(), [&](int s) -> int {
        const std::vector<int>& idx = h->index[s];
        std::vector<OpalSearchResult*> res(idx.size());
        for (size_t k = 0; k < idx.size(); k++) res[k] = results[idx[k]];
        return search_into_results(h->shards[s], scoring, nullptr, (int)idx.size(), nullptr, res.data(), searchType, h->shards[s]->device());
    });
}

int opalb200_db_search_results(OpalB200Db* hh, const unsigned char query[], int queryLength, int gapOpen, int gapExt,
                               const int* scoreMatrix, int alphabetLength, OpalSearchResult* results[], int searchType, int mode) {
    return db_search_results(hh, Scoring::with_matrix(query, queryLength, scoreMatrix, alphabetLength, gapOpen, gapExt, mode), results,
                             searchType);
}

int opalb200_db_search_results_pssm(OpalB200Db* hh, const unsigned char query[], const int* pssm, int queryLength, int alphabetLength,
                                    int gapOpen, int gapExt, OpalSearchResult* results[], int searchType, int mode) {
    if (const int rc = check_pssm_args(pssm, query, queryLength, alphabetLength, searchType)) return rc;
    return db_search_results(hh, Scoring::with_pssm(query, pssm, queryLength, alphabetLength, gapOpen, gapExt, mode), results, searchType);
}

// Score -> top-k -> alignment for a batch of searches; indices / results are [search][k] (row q starts at q * k).  Every
// search is checked before any runs (the PSSM argument rule, then -- when anything is selected -- Scoring::validate and
// the database's residue codes), in search order, so a fault reports the code of the lowest-index search that has one
// and writes nothing.  Every shard searches and selects ITS k best of every search on the device (DeviceDb::search_batch_topk:
// only k records per search and shard come back, not every score); the candidates are merged here: score descending,
// caller index ascending among equals.  At OPAL_SEARCH_ALIGNMENT every shard then aligns the hits it owns, of all
// searches in the same launches.
static int db_search_batch_topk(OpalB200Db* hh, const std::vector<Scoring>& searches, int searchType, int k, int* indices,
                                OpalSearchResult* results[], int* found, int inFlight) {
    if (found) *found = 0;
    if (!hh || !indices || !results || k < 0) return OPAL_ERR_NO_SIMD_SUPPORT;
    DeviceGuard guard;
    DbHandle* h = reinterpret_cast<DbHandle*>(hh);
    const int n = h->n, kk = std::min(k, n), parts = h->parts(), ns = (int)searches.size();
    const int wantEnd = searchType != OPAL_SEARCH_SCORE;
    for (const Scoring& sc : searches) {
        if (sc.byPssm)
            if (const int rc = check_pssm_args(sc.entries, sc.query, sc.Q, sc.A, searchType)) return rc;
        for (int s = 0; s < parts && kk > 0; s++)
            if (const int rc = h->shards[s]->check(sc)) return rc;
    }
    if (kk <= 0 || ns == 0) {
        if (found) *found = kk;
        return 0;
    }
    struct Hit { int score, index, endQ, endT, shard, local; };
    std::vector<std::vector<Hit>> perShard((size_t)parts);  // [shard]: ks candidates of every search
    auto shard_k = [&](int s) { return std::min(kk, h->shards[s]->size()); };
    int status = on_shards(parts, [&](int s) -> int {
        const size_t all = (size_t)ns * (size_t)shard_k(s);
        std::vector<int> li(all), sc(all), eq(all), et(all);
        const int* map = h->index.empty() ? nullptr : h->index[s].data();
        const int r = h->shards[s]->search_batch_topk(searches, wantEnd, shard_k(s), map, li.data(), sc.data(), eq.data(), et.data(),
                                                      inFlight <= 0 ? 3 : inFlight);
        if (r) return r;
        for (size_t j = 0; j < all; j++) perShard[s].push_back({sc[j], h->caller_index(s, li[j]), eq[j], et[j], s, li[j]});
        return 0;
    });
    h->collect_stats();
    if (status) return status;
    auto better = [](const Hit& a, const Hit& b) { return a.score != b.score ? a.score > b.score : a.index < b.index; };
    std::vector<Hit> hits;  // [search][kk]
    for (int q = 0; q < ns; q++) {
        std::vector<Hit> cand;
        for (int s = 0; s < parts; s++) {
            const auto from = perShard[s].begin() + (size_t)q * shard_k(s);
            cand.insert(cand.end(), from, from + shard_k(s));
        }
        std::sort(cand.begin(), cand.end(), better);
        hits.insert(hits.end(), cand.begin(), cand.begin() + kk);
    }
    auto slot = [&](int q, int j) { return (size_t)q * (size_t)k + (size_t)j; };
    for (int q = 0; q < ns; q++)
        for (int j = 0; j < kk; j++) {
            const Hit& hit = hits[(size_t)q * kk + j];
            OpalSearchResult* r = results[slot(q, j)];
            indices[slot(q, j)] = hit.index;
            opalInitSearchResult(r);
            opalSearchResultSetScore(r, hit.score);
            r->endLocationQuery = wantEnd ? hit.endQ : -1;
            r->endLocationTarget = wantEnd ? hit.endT : -1;
            r->alignmentLength = -1;  // as opalSearchDatabase leaves it below OPAL_SEARCH_ALIGNMENT (:1508-1515)
        }
    if (found) *found = kk;
    if (searchType == OPAL_SEARCH_ALIGNMENT)  // start + alignment on the device that owns the target
        status = on_shards(parts, [&](int s) -> int {
            std::vector<std::vector<int>> subset((size_t)ns);
            std::vector<std::vector<OpalSearchResult*>> res((size_t)ns);
            for (int q = 0; q < ns; q++)
                for (int j = 0; j < kk; j++) {
                    const Hit& hit = hits[(size_t)q * kk + j];
                    if (hit.shard == s) { subset[q].push_back(hit.local); res[q].push_back(results[slot(q, j)]); }
                }
            std::vector<AlignSet> sets;
            for (int q = 0; q < ns; q++)
                if (!subset[q].empty()) sets.push_back({&searches[q], res[q].data(), (int)subset[q].size(), subset[q].data()});
            return sets.empty() ? 0 : align_database(h->shards[s], sets);
        });
    return status;
}

int opalb200_db_search_topk(OpalB200Db* hh, const unsigned char query[], int queryLength, int gapOpen, int gapExt,
                            const int* scoreMatrix, int alphabetLength, int searchType, int mode, int k, int* indices,
                            OpalSearchResult* results[], int* found) {
    return db_search_batch_topk(hh, {Scoring::with_matrix(query, queryLength, scoreMatrix, alphabetLength, gapOpen, gapExt, mode)},
                                searchType, k, indices, results, found, 1);
}

int opalb200_db_search_topk_pssm(OpalB200Db* hh, const unsigned char query[], const int* pssm, int queryLength, int alphabetLength,
                                 int gapOpen, int gapExt, int searchType, int mode, int k, int* indices, OpalSearchResult* results[],
                                 int* found) {
    return db_search_batch_topk(hh, {Scoring::with_pssm(query, pssm, queryLength, alphabetLength, gapOpen, gapExt, mode)}, searchType, k,
                                indices, results, found, 1);
}

int opalb200_db_search_batch_topk(OpalB200Db* hh, int numSearches, const unsigned char* const queries[], const int queryLengths[],
                                  const int modes[], int gapOpen, int gapExt, const int* scoreMatrix, int alphabetLength,
                                  int searchType, int k, int* indices, OpalSearchResult* results[], int* found, int inFlight) {
    if (found) *found = 0;
    if (numSearches > 0 && !modes) return OPAL_ERR_INVALID_MODE;
    if (numSearches > 0 && (!queries || !queryLengths)) return OPAL_ERR_NO_SIMD_SUPPORT;
    std::vector<Scoring> searches;
    for (int q = 0; q < numSearches; q++)
        searches.push_back(Scoring::with_matrix(queries[q], queryLengths[q], scoreMatrix, alphabetLength, gapOpen, gapExt, modes[q]));
    return db_search_batch_topk(hh, searches, searchType, k, indices, results, found, inFlight);
}

int opalb200_db_search_batch_topk_pssm(OpalB200Db* hh, int numSearches, const unsigned char* const queries[], const int* const pssms[],
                                       const int queryLengths[], const int modes[], int alphabetLength, int gapOpen, int gapExt,
                                       int searchType, int k, int* indices, OpalSearchResult* results[], int* found, int inFlight) {
    if (found) *found = 0;
    if (numSearches > 0 && !modes) return OPAL_ERR_INVALID_MODE;
    if (numSearches > 0 && (!pssms || !queryLengths)) { set_error("pssms / queryLengths is NULL"); return OPAL_ERR_INVALID_ARGUMENT; }
    std::vector<Scoring> searches;
    for (int q = 0; q < numSearches; q++)
        searches.push_back(Scoring::with_pssm(queries ? queries[q] : nullptr, pssms[q], queryLengths[q], alphabetLength, gapOpen, gapExt,
                                              modes[q]));
    return db_search_batch_topk(hh, searches, searchType, k, indices, results, found, inFlight);
}

void opalb200_db_last_stats(const OpalB200Db* h, int* kernelLaunches, int* rerun32, int* G, int* R, int* passes,
                            int* warpsPerPartition, int* groups) {
    const SearchStats& s = reinterpret_cast<const DbHandle*>(h)->stats;
    if (kernelLaunches) *kernelLaunches = s.kernelLaunches;
    if (rerun32) *rerun32 = s.rerun32;
    if (G) *G = s.G;
    if (R) *R = s.R;
    if (passes) *passes = s.passes;
    if (warpsPerPartition) *warpsPerPartition = s.warpsPerPartition;
    if (groups) *groups = s.groups;
}

int opalb200_db_last_folded(const OpalB200Db* h) { return reinterpret_cast<const DbHandle*>(h)->stats.foldedTasks; }

int opalb200_db_last_chained(const OpalB200Db* h) { return reinterpret_cast<const DbHandle*>(h)->stats.chainedTasks; }

double opalb200_measure_dpx_peak(int device, double* threadInstrPerSec, float* ms) {
    DeviceGuard guard;
    return measure_dpx_peak(device, 0, threadInstrPerSec, ms);
}

double opalb200_measure_dpx_peak_mix(int device, int mix, double* threadInstrPerSec, float* ms) {
    DeviceGuard guard;
    return measure_dpx_peak(device, mix != 0 ? 1 : 0, threadInstrPerSec, ms);
}

}  // extern "C"
