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

// A length-sorted (longest first) database resident in one device's HBM.
class DeviceDb {
public:
    static DeviceDb* create(unsigned char* const* db, int n, const int* lens, int device);
    // Database that is already packed: residues contiguous, longest sequence first; order[p] = caller index of
    // sorted position p (NULL = identity).  This is the in-memory form of the on-disk format (cli/packed_db.h).
    static DeviceDb* create_sorted(const unsigned char* residues, const int* sortedLens, const int* order, int n, int device);
    ~DeviceDb();

    // Several queries against the resident database, up to `inFlight` of them on the device at a time (each on a
    // search context of its own: streams, result and scratch buffers), so that the tail of one query overlaps the
    // bulk of the next and host-side planning / publishing overlaps kernels.  Outputs are [search][caller index].
    int search_batch(const std::vector<Scoring>& searches, int wantEnd, int* scores, int* endQ, int* endT, int inFlight,
                     float* batchMs);
    // Blocks until the upload issued by create() has finished (create() returns with it in flight).
    bool ensure_uploaded();

    // Score / score+end for every non-skipped target, into `out`.  Stages: Scoring::validate, route (every target to
    // the 16- or the 32-bit class), upload_args, ladder (16 bits, then 32 bits for what 16 could not hold).
    int search(const Scoring& s, int wantEnd, const unsigned char* skip, const SearchOut& out, float* deviceMs);

    // Score [+ end] search followed by the selection of the k best targets: score descending, then smallest
    // map[caller index] (map NULL: the caller index itself).  Writes k (<= size()) caller indices and their records.
    int search_topk(const Scoring& s, int wantEnd, int k, const int* map, int* outIndex, int* outScore, int* outEndQ, int* outEndT);
    // search_topk of every search, up to `inFlight` of them on the device at a time (as search_batch); k <= size().
    // Outputs are [search][k].  0, or the code of the lowest-index search that failed.
    int search_batch_topk(const std::vector<Scoring>& searches, int wantEnd, int k, const int* map, int* outIndex, int* outScore,
                          int* outEndQ, int* outEndT, int inFlight);
    // The checks a search makes before it sweeps: Scoring::validate, then (for a search that sweeps at all) the
    // database's residue codes against the alphabet length.  0 or an OPAL_B200_ERR_* code.
    int check(const Scoring& s);

    int size() const { return n_; }
    long long residues() const { return totalResidues_; }
    const SearchStats& stats() const { return stats_; }
    int device() const { return device_; }
    cudaStream_t stream() const { return stream_; }
    // sorted position -> caller index, and device-side views (used by the alignment stage)
    const std::vector<int>& order() const { return lay_->order; }
    const std::vector<int>& sorted_position() const { return lay_->pos; }
    const uint8_t* d_residues() const { return dResidues_; }
    const long long* d_offsets() const { return dOffsets_; }
    const std::vector<long long>& offsets() const { return lay_->offsets; }
    const std::vector<int>& sorted_lengths() const { return lay_->sortedLen; }
    const uint8_t* h_residues() const { return hResidues_; }  // pinned host copy, sorted order

private:
    DeviceDb() {}
    static DeviceDb* build(unsigned char* const* db, const unsigned char* packed, const int* lens, const int* order, int n, int device);
    DeviceDb* clone_context();
    bool ensure_order();
    // job(context, q) for every q in [0, num), up to inFlight at a time, each context on a host thread of its own.
    int in_flight(int num, int inFlight, const std::function<int(DeviceDb*, int)>& job, float* batchMs);
    bool alloc_search_buffers();
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

    int device_ = 0, n_ = 0, numSMs_ = 0, smemLimit_ = 0;
    long long totalResidues_ = 0;
    std::shared_ptr<const Layout> lay_;
    bool ownsDb_ = true, uploaded_ = false;  // search contexts made by clone_context() borrow the database arrays
    std::vector<DeviceDb*> contexts_;
    uint8_t* hResidues_ = nullptr;
    uint8_t* dResidues_ = nullptr;
    long long* dOffsets_ = nullptr;
    int* dLengths_ = nullptr;
    int *dResults_ = nullptr, *hResults_ = nullptr;  // [score | endQ | endT | task list] device block, [score | endQ | endT] pinned
    int *dScore_ = nullptr, *dEndQ_ = nullptr, *dEndT_ = nullptr, *dTaskList_ = nullptr;  // views
    uint32_t *dBndH_ = nullptr, *dBndF_ = nullptr;
    uint16_t* dPairStream_ = nullptr;
    long long* dPairOffsets_ = nullptr;
    uint16_t* dFoldStream_ = nullptr;    // folded stream of the numFold_ longest targets
    long long* dFoldOffsets_ = nullptr;
    int numFold_ = 0;
    int *dMaxCode_ = nullptr, *hMaxCode_ = nullptr;
    unsigned char *hBlock_ = nullptr, *dBlock_ = nullptr;  // offsets | pair offsets | lengths | max code | residues (pinned / device)
    int numPairs_ = 0, maxCode_ = 0;
    unsigned char *dArgs_ = nullptr, *hArgs_ = nullptr;  // launch counters | score matrix | query, or counters | PSSM (device / pinned)
    size_t argsCapacity_ = 0;
    int *hScore_ = nullptr, *hEndQ_ = nullptr, *hEndT_ = nullptr;  // views into hResults_
    cudaStream_t stream_ = nullptr;
    cudaEvent_t evStart_ = nullptr, evStop_ = nullptr, evFork_ = nullptr;
    std::vector<cudaStream_t> auxStreams_;
    std::vector<cudaEvent_t> auxEvents_;
    SearchStats stats_;
    std::vector<void*> chainScratch_;  // device blocks of chained launches (boundary rows, flags), released by the next search
    bool startRecorded_ = false;
    int* dOrder_ = nullptr;       // device copy of order_ (sorted position -> caller index), made by the first top-k search, borrowed by the contexts
};

double measure_dpx_peak(int device, int mix, double* threadInstrPerSec, float* ms);  // mix 0 = SW recurrence, 1 = NW / HW / OV

}  // namespace opalb200
