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
    // bulk of the next and host-side planning / publishing overlaps kernels.  Outputs are [query][caller index].
    // pssms: one position-specific scoring matrix per query (see search()); queries / matrix are then unused.
    int search_batch(int numQueries, const unsigned char* const* queries, const int* queryLengths, int Go, int Ge,
                     const int* matrix, int A, int wantEnd, int mode, int* scores, int* endQ, int* endT, int inFlight,
                     float* batchMs, const int* modes = nullptr,  // modes: one per query (NULL: `mode` for all)
                     const int* const* pssms = nullptr);
    // Blocks until the upload issued by create() has finished (create() returns with it in flight).
    bool ensure_uploaded();

    // Score / score+end for every non-skipped target; outputs in caller order (-1 = unset).
    // With `records` the results go straight into the caller's OpalSearchResult records instead of the three arrays
    // (one pass over half a million 40-byte records instead of two); noAlignmentFill also gives every computed record
    // the fields opalSearchDatabase sets below OPAL_SEARCH_ALIGNMENT (reference src/opal.cpp:1508-1515).
    // With `pssm` (Q x A ints, row r = scores of query position r against every letter) the query is scored by it
    // instead of by matrix rows of query letters; query and matrix are then unused (either may be NULL).
    int search(const unsigned char* query, int Q, int Go, int Ge, const int* matrix, int A, int wantEnd, int mode,
               const unsigned char* skip, int* scores, int* endQ, int* endT, float* deviceMs,
               OpalSearchResult* const* records = nullptr, bool noAlignmentFill = false, const int* pssm = nullptr);

    // Score [+ end] search followed by the selection of the k best targets: score descending, then smallest
    // map[caller index] (map NULL: the caller index itself).  Writes k (<= size()) caller indices and their records.
    int search_topk(const unsigned char* query, int Q, int Go, int Ge, const int* matrix, int A, int wantEnd, int mode, int k,
                    const int* map, int* outIndex, int* outScore, int* outEndQ, int* outEndT, const int* pssm = nullptr);

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
    bool alloc_search_buffers();
    struct Group;
    bool plan_class(int type, const std::vector<int>& list, int Q, int A, int mode, int wantEnd, std::vector<Group>* groups,
                    double deadline = 0);
    bool launch_group(const Group& grp, int* taskListDevice, cudaStream_t stream, const unsigned char* dQuery, const int* dMatrix,
                      int Q, int Go, int Ge, int A, int wantEnd, int mode, int maxScore, int* launchSlot);
    int run_classes(const std::vector<std::pair<int, const std::vector<int>*>>& classes, const unsigned char* dQuery,
                    const int* dMatrix, int Q, int Go, int Ge, int A, int wantEnd, int mode, int maxScore, int* launchSlot);
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
    int *dScore_ = nullptr, *dEndQ_ = nullptr, *dEndT_ = nullptr, *dTaskList_ = nullptr, *dCounters_ = nullptr;  // views
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
    const int* dPssm_ = nullptr;  // the PSSM of the search in progress in dArgs_ (NULL: matrix search)
    size_t argsCapacity_ = 0;
    int *hScore_ = nullptr, *hEndQ_ = nullptr, *hEndT_ = nullptr;  // views into hResults_
    cudaStream_t stream_ = nullptr;
    cudaEvent_t evStart_ = nullptr, evStop_ = nullptr, evFork_ = nullptr;
    std::vector<cudaStream_t> auxStreams_;
    std::vector<cudaEvent_t> auxEvents_;
    SearchStats stats_;
    std::vector<void*> chainScratch_;  // device blocks of chained launches (boundary rows, flags), released by the next search
    bool startRecorded_ = false;
    bool keepOnDevice_ = false;   // search_topk: results stay in HBM, the ladder's hand-over list is gathered there
    int* dSelect_ = nullptr;      // search_topk scratch: [count | flagged positions (n) | k records]
    int* dOrder_ = nullptr;       // device copy of order_ (sorted position -> caller index), made by the first search_topk
    int absScore_ = 0;            // largest |score matrix entry| of the search in progress
    bool rangeTracking_ = false;  // its 16-bit NW / HW / OV class is guarded by the kernel's range tracking
};

double measure_dpx_peak(int device, int mix, double* threadInstrPerSec, float* ms);  // mix 0 = SW recurrence, 1 = NW / HW / OV

}  // namespace opalb200
