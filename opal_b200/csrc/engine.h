// engine.h -- host-side engine of opal-b200: resident database, geometry choice, pass scheduling.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/opal.h"

#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

namespace opalb200 {

// Return codes shared with opal.h (OPAL_ERR_OVERFLOW / _NO_SIMD_SUPPORT / _INVALID_MODE).
constexpr int OPAL_B200_ERR_OVERFLOW = 1, OPAL_B200_ERR_CUDA = 2, OPAL_B200_ERR_MODE = 3, OPAL_B200_ERR_ARGUMENT = 4;
// Folded stream: at most this many of the longest targets, none shorter than kFoldMinLength.
constexpr int kFoldTargets = 128, kFoldMinLength = 256;

// Kernel registry: one translation unit per strip height R (kernels_inst.cu compiled with
// -DOPAL_R=<R>), each exporting a table indexed [type * 4 + flavor]; type 0 = Packed16, 1 = Scalar32.
struct KernelTable {
    int R;
    const void* const* fn;
    const void* const* chainFn;  // chained-pass variants [type * 4 + flavor]; entries are null for most strip heights
};
const std::vector<KernelTable>& kernel_tables();

struct Geometry {
    int G = 1, R = 0, tableIndex = 0, passes = 1, Rpad = 0, rowStride = 0, padTop = 0, warpsPerPartition = 4;
    size_t smemBytes = 0;
    bool folded = false;  // one target per warp in both half-words (SearchParams::folded)
    bool chain = false;   // all passes of a task in one launch, a warp per pass (SearchParams::chain)
};

struct SearchStats {
    int kernelLaunches = 0, rerun32 = 0, G = 0, R = 0, passes = 0, warpsPerPartition = 0, groups = 0, foldedTasks = 0, chainedTasks = 0;
};

constexpr int kMaxDevices = 64;  // devices the per-device resource cache is sized for (larger ordinals are rejected)
// Device memory from the per-device block cache (engine.cu): recycled, not returned to the driver (until trim_cache()).
bool device_alloc(int device, void** p, size_t bytes);
void device_release(int device, void* p);
void trim_cache();
void trim_layouts();

// body(lo, hi) over [0, n) in parts of at least `grain`, on the persistent host pool (the caller takes part).
void parallel_for(long long n, long long grain, const std::function<void(long long, long long)>& body);

void set_error(const std::string& msg);
const char* last_error();

inline bool valid_mode(int mode) { return mode == OPAL_MODE_NW || mode == OPAL_MODE_HW || mode == OPAL_MODE_OV || mode == OPAL_MODE_SW; }

// What decides the widths that can carry a search (Scoring::bounds).
struct ScoreBounds {
    int maxEntry = 0, minEntry = 0;       // over every entry that can score a cell (0 when there is none)
    long long absEntry = 0, gapMax = 0;   // largest |entry|; larger of |Go| and |Ge|
    bool args16 = false, args32 = false;  // entries and penalties fit the 16-bit / the 32-bit passes
};

// How one search scores: the query, the gap penalties and the mode, and either the A x A substitution matrix (cell
// (r, y) = matrix[query[r] * A + y]) or a Q x A position-specific scoring matrix (cell (r, y) = pssm[r * A + y]).  With
// a PSSM the query residues (codes < A) only label the diagonal steps of an alignment MATCH / MISMATCH: the score and
// end searches do not read them, and they may be NULL there.
struct Scoring {
    const unsigned char* query = nullptr;
    int Q = 0, A = 0, Go = 0, Ge = 0, mode = 0;
    const int* entries = nullptr;  // the matrix or the PSSM (may be NULL when it has no entries)
    bool byPssm = false;

    static Scoring with_matrix(const unsigned char* query, int Q, const int* matrix, int A, int Go, int Ge, int mode) {
        return {query, Q, A, Go, Ge, mode, matrix, false};
    }
    static Scoring with_pssm(const unsigned char* query, const int* pssm, int Q, int A, int Go, int Ge, int mode) {
        return {query, Q, A, Go, Ge, mode, pssm, true};
    }
    long long num_entries() const { return byPssm ? (long long)Q * A : (long long)A * A; }
    int cell(int r, int y) const { return byPssm ? entries[(size_t)r * A + y] : entries[query[r] * A + y]; }
    ScoreBounds bounds() const;
    // The argument checks of a search (reference src/opal.cpp:183-198, 615-630), in the order that decides the code of
    // a call with several faults, and its bounds: 0, or an OPAL_B200_ERR_* code (with an error text where the reference
    // has none).  Entries are read only once the alphabet length has passed.
    int validate(ScoreBounds* b) const;
};

// Where the results of one search go: the caller's arrays (caller order, -1 = unset; endQ / endT may be NULL), the
// caller's OpalSearchResult records, or nowhere yet -- left in HBM for the device-side selection of search_topk.
struct SearchOut {
    int *scores = nullptr, *endQ = nullptr, *endT = nullptr;
    // Records: one pass over half a million 40-byte records instead of two; noAlignmentFill also gives every computed
    // record the fields opalSearchDatabase sets below OPAL_SEARCH_ALIGNMENT (reference src/opal.cpp:1508-1515).
    OpalSearchResult* const* records = nullptr;
    bool noAlignmentFill = false;
    int* dSelect = nullptr;  // on the device: selection scratch [count | flagged positions (n) | k records]

    static SearchOut arrays(int* scores, int* endQ, int* endT) { return {scores, endQ, endT}; }
    static SearchOut into(OpalSearchResult* const* records, bool noAlignmentFill) { return {nullptr, nullptr, nullptr, records, noAlignmentFill}; }
    static SearchOut on_device(int* dSelect) { return {nullptr, nullptr, nullptr, nullptr, false, dSelect}; }
    void put(int i, int score, int endQuery, int endTarget) const;  // the result of caller index i
};

// Task lengths of one class (longest first) with strided prefix sums, so that the planner can price any
// contiguous range of tasks under any group size in O(1).
struct TaskLens {
    std::vector<int> len;
    std::vector<double> prefix[6];  // prefix[s][k] = sum of len[i] over i = 0, g, 2g, ... < k*g with g = 1 << s
    void build();
    // sum of len[i] for i = lo, lo+g, ... < hi  (lo must be a multiple of g = 1 << sh), and how many terms
    double strided(int sh, size_t lo, size_t hi, double* terms) const {
        const size_t g = (size_t)1 << sh, a = lo / g, b = (hi + g - 1) / g;
        *terms = (double)(b - a);
        return prefix[sh][b] - prefix[sh][a];
    }
};

// What depends on the sequence lengths alone (engine.cu, "layouts"): shared by every database built from the same
// length array, immutable once built.
struct Layout {
    std::vector<int> lens;                   // the caller's length array (the cache key)
    std::vector<int> order, pos, sortedLen;  // sorted position -> caller index, its inverse, lengths longest first
    std::vector<long long> offsets, copyOff; // residue offset of sorted position p / of copy position i (n + 1 entries)
    std::vector<long long> pairOff, foldOff; // first entry of every pair / folded target in its stream
    long long total = 0, entries = 0, foldEntries = 0;
    int numPairs = 0, numFold = 0, nonEmpty = 0;  // nonEmpty: sorted positions [0, nonEmpty) have at least one residue
    const TaskLens& pair_lens() const;       // planner prefix sums over all non-empty pairs / targets, built on first use
    const TaskLens& target_lens() const;
    // The database cut into devices x perDevice parts (engine.cu: Layout::parts): caller indices of every part,
    // ascending; part d * perDevice + k is slice k of device d.  Built on first use, remembered with the layout.
    std::shared_ptr<const std::vector<std::vector<int>>> parts(int devices, int perDevice) const;
private:
    mutable std::once_flag pairOnce_, targetOnce_;
    mutable TaskLens pairLens_, targetLens_;
    mutable std::mutex partsMu_;
    mutable std::vector<std::pair<std::pair<int, int>, std::shared_ptr<const std::vector<std::vector<int>>>>> parts_;
};
// The layout of a database: from the cache, or built (and remembered when the database is scattered).
std::shared_ptr<const Layout> layout_for(const int* lens, const int* order, int n, bool packed, bool* cached);
// The calling thread's searches are followed by others on the same device (batches, slices): plans are priced by the
// SM time they hold rather than by when their last task ends.
void set_thread_overlapped(bool on);
struct PhaseTrace;  // phase timings on stderr with OPAL_B200_TRACE=1 (engine.cu)

// A length-sorted (longest first) database resident in one device's HBM, built by DeviceDb::build and read-only once
// its upload has finished.  It is the only owner of these allocations; search contexts read them through a const
// reference.
struct DbArrays {
    int device = 0, n = 0, numSMs = 0, smemLimit = 0;
    long long totalResidues = 0;
    std::shared_ptr<const Layout> lay;
    unsigned char *hBlock = nullptr, *dBlock = nullptr;  // offsets | pair offsets | fold offsets | lengths | max code | residues (pinned / device)
    uint8_t *hResidues = nullptr, *dResidues = nullptr;  // views: the pinned host copy and the device copy
    long long *dOffsets = nullptr, *dPairOffsets = nullptr, *dFoldOffsets = nullptr;
    int *dLengths = nullptr, *dMaxCode = nullptr;
    uint16_t* dPairStream = nullptr;
    uint16_t* dFoldStream = nullptr;  // folded stream of the numFold longest targets
    int numPairs = 0, numFold = 0;
    int* hMaxCode = nullptr;  // pinned: the largest residue code, copied back by the upload (read once it has finished)
    int* dOrder = nullptr;    // device copy of lay->order (sorted position -> caller index), made by DeviceDb::ensure_order

    DbArrays() = default;
    DbArrays(const DbArrays&) = delete;
    DbArrays& operator=(const DbArrays&) = delete;
    ~DbArrays();
};

// One search in flight on a resident database: its stream and events, result and argument blocks, boundary rows and
// chained-launch scratch.  It reads the database arrays and owns none of them.
class SearchContext {
public:
    explicit SearchContext(const DbArrays& db) : db_(db) {}
    SearchContext(const SearchContext&) = delete;
    ~SearchContext();
    bool alloc_search_buffers();
    // Blocks until the database upload issued on this context's stream has finished (nothing to wait for elsewhere).
    bool ensure_uploaded();
    // Score / score+end for every non-skipped target, into `out`.  Stages: Scoring::validate, route (every target to
    // the 16- or the 32-bit class), upload_args, ladder (16 bits, then 32 bits for what 16 could not hold).
    int search(const Scoring& s, int wantEnd, const unsigned char* skip, const SearchOut& out, float* deviceMs);
    // Score [+ end] search followed by the selection of the k best targets: score descending, then smallest
    // map[caller index] (map NULL: the caller index itself).  Writes k (<= n) caller indices and their records.  Reads
    // the index map made by DeviceDb::ensure_order.
    int search_topk(const Scoring& s, int wantEnd, int k, const int* map, int* outIndex, int* outScore, int* outEndQ, int* outEndT);

private:
    friend class DeviceDb;  // build() uploads on the first context's stream; in_flight() reads every context's stats and timing
    struct Group;
    struct Run;     // the search in progress (engine.cu)
    struct Routes;  // its targets by precision class
    int route(const Run& run, const unsigned char* skip, const SearchOut& out, Routes* routes);
    bool upload_args(Run* run);
    bool ladder(const Run& run, Routes& routes, const SearchOut& out, float* deviceMs, PhaseTrace& trace, int* rc);
    bool fetch(int wantEnd, PhaseTrace& trace);
    bool publish(const std::vector<int>& list, int wantEnd, const SearchOut& out, std::vector<int>* overflowed);
    bool collect(int* dSelect, int emptyFrom, std::vector<int>* flagged);
    bool plan_class(int type, const std::vector<int>& list, const Run& run, std::vector<Group>* groups, double deadline = 0);
    bool launch_group(const Group& grp, int* taskListDevice, cudaStream_t stream, const Run& run);
    int run_classes(const std::vector<std::pair<int, const std::vector<int>*>>& classes, const Run& run);
    bool ensure_boundary();

    const DbArrays& db_;
    bool uploadPending_ = false;  // the database upload was issued on stream_ and has not been waited for
    int *dResults_ = nullptr, *hResults_ = nullptr;  // [score | endQ | endT | task list] device block, [score | endQ | endT] pinned
    int *dScore_ = nullptr, *dEndQ_ = nullptr, *dEndT_ = nullptr, *dTaskList_ = nullptr;  // views
    int *hScore_ = nullptr, *hEndQ_ = nullptr, *hEndT_ = nullptr;  // views into hResults_
    uint32_t *dBndH_ = nullptr, *dBndF_ = nullptr;
    unsigned char *dArgs_ = nullptr, *hArgs_ = nullptr;  // launch counters | score matrix | query, or counters | PSSM (device / pinned)
    size_t argsCapacity_ = 0;
    cudaStream_t stream_ = nullptr;
    cudaEvent_t evStart_ = nullptr, evStop_ = nullptr, evFork_ = nullptr;
    std::vector<cudaStream_t> auxStreams_;
    std::vector<cudaEvent_t> auxEvents_;
    SearchStats stats_;
    std::vector<void*> chainScratch_;  // device blocks of chained launches (boundary rows, flags), released by the next search
    bool startRecorded_ = false;
};

// The pairs path: many queries, each scored against its own list of database entries (pairs_kernel.cuh).  It reads the
// database arrays through a const reference and owns only the buffers of its call, which it releases when it goes.
// Stages: route every pair (the defined result of an empty query or target, or the 16- or the 32-bit class), group the
// classes' pairs by query and plan their geometry, one upload of [matrix | queries | tables], the 16-bit launch, the
// device-side collection of what 16 bits could not hold, the 32-bit launch, one copy of the per-pair results back.
struct PairTask;
struct PairQuery;
struct PairBlock;
class PairsSearch {
public:
    PairsSearch(const DbArrays& db, cudaStream_t stream) : db_(db), stream_(stream) {}
    PairsSearch(const PairsSearch&) = delete;
    ~PairsSearch();
    // Pair k scores queries[pairQuery[k]] against database entry pairTarget[k] (the database's caller index); its result
    // goes to out.put(k, ...).  The queries share the alphabet, the matrix, the gap penalties and the mode, and have
    // passed DeviceDb::check.  0 or an OPAL_B200_ERR_* code (nothing is written unless it is 0).
    int run(const std::vector<Scoring>& queries, int wantEnd, int numPairs, const int* pairQuery, const int* pairTarget,
            const SearchOut& out, float* deviceMs, SearchStats* stats);

private:
    struct Class;  // the pairs of one precision class, grouped and planned (engine.cu)
    struct Tables { const PairQuery* queryTab; const PairTask* tasks; const PairBlock* blocks; };  // a class's tables on the device
    bool plan(int type, const std::vector<Scoring>& queries, int wantEnd, const std::vector<std::vector<int>>& byQuery,
              const int* pos, Class* c);
    bool launch(const Class& c, const std::vector<Scoring>& queries, int wantEnd, const ScoreBounds& b, bool rangeTracking,
                long long step, long long rangeLo, const Tables& d);
    bool upload(const std::vector<unsigned char>& block, unsigned char** dBlock, unsigned char** hBlock);
    void* alloc(size_t bytes);

    const DbArrays& db_;
    cudaStream_t stream_;
    std::vector<void*> device_, pinned_;  // this call's blocks
    cudaEvent_t evStart_ = nullptr, evStop_ = nullptr;
    const int* dMatrix_ = nullptr;
    const uint8_t* dQueries_ = nullptr;
    int *dOut_ = nullptr;  // [score | endQ | endT | flagged count | flagged slots], numPairs each
    int numPairs_ = 0;
};
bool launch_gather_pairs(const PairTask* tasks, int numTasks, const uint8_t* residues, const long long* offsets, uint16_t* stream,
                         cudaStream_t st);
const void* pairs_kernel_fn(int rIndex, int type, int flavor);  // pairs.cu: [strip height index][Packed16 / Scalar32][flavor]

// A resident database and the search contexts that run on it.
class DeviceDb {
public:
    static DeviceDb* create(unsigned char* const* db, int n, const int* lens, int device);
    // Database that is already packed: residues contiguous, longest sequence first; order[p] = caller index of
    // sorted position p (NULL = identity).  This is the in-memory form of the on-disk format (cli/packed_db.h).
    static DeviceDb* create_sorted(const unsigned char* residues, const int* sortedLens, const int* order, int n, int device);

    // Several queries against the resident database, up to `inFlight` of them on the device at a time (each on a
    // search context of its own: streams, result and scratch buffers), so that the tail of one query overlaps the
    // bulk of the next and host-side planning / publishing overlaps kernels.  Outputs are [search][caller index].
    int search_batch(const std::vector<Scoring>& searches, int wantEnd, int* scores, int* endQ, int* endT, int inFlight,
                     float* batchMs);
    // Blocks until the upload issued by create() has finished (create() returns with it in flight).
    bool ensure_uploaded() { return contexts_[0]->ensure_uploaded(); }

    // SearchContext::search on the first context.
    int search(const Scoring& s, int wantEnd, const unsigned char* skip, const SearchOut& out, float* deviceMs) {
        return contexts_[0]->search(s, wantEnd, skip, out, deviceMs);
    }

    // For every search: the score [+ end] search followed by the selection of the k best targets (score descending,
    // then smallest map[caller index]; map NULL: the caller index itself), up to `inFlight` of them on the device at
    // a time (as search_batch); k <= size().  Outputs are [search][k] caller indices and their records.  0, or the
    // code of the lowest-index search that failed.
    int search_batch_topk(const std::vector<Scoring>& searches, int wantEnd, int k, const int* map, int* outIndex, int* outScore,
                          int* outEndQ, int* outEndT, int inFlight);
    // The checks a search makes before it sweeps: Scoring::validate, then (for a search that sweeps at all) the
    // database's residue codes against the alphabet length.  0 or an OPAL_B200_ERR_* code.
    int check(const Scoring& s);
    // PairsSearch::run on the first context's stream, once the upload has finished; the call's statistics become stats().
    int search_pairs(const std::vector<Scoring>& queries, int wantEnd, int numPairs, const int* pairQuery, const int* pairTarget,
                     const SearchOut& out, float* deviceMs);

    int size() const { return db_.n; }
    long long residues() const { return db_.totalResidues; }
    const SearchStats& stats() const { return contexts_[0]->stats_; }
    int device() const { return db_.device; }
    // What the alignment stage reads: the database arrays, and the stream of the first context to run on.
    const DbArrays& arrays() const { return db_; }
    cudaStream_t stream() const { return contexts_[0]->stream_; }

private:
    DeviceDb() {}
    static DeviceDb* build(unsigned char* const* db, const unsigned char* packed, const int* lens, const int* order, int n, int device);
    bool ensure_order();
    // job(context, q) for every q in [0, num), up to inFlight at a time, each context on a host thread of its own.
    int in_flight(int num, int inFlight, const std::function<int(SearchContext&, int)>& job, float* batchMs);

    DbArrays db_;
    // [0]: made with the database, which is uploaded on its stream; in_flight adds more.  Declared after db_, so every
    // context has synchronized its streams and released its blocks before the database arrays go.
    std::vector<std::unique_ptr<SearchContext>> contexts_;
};

double measure_dpx_peak(int device, int mix, double* threadInstrPerSec, float* ms);  // mix 0 = SW recurrence, 1 = NW / HW / OV

}  // namespace opalb200
