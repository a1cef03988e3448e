// align.cu -- the OPAL_SEARCH_ALIGNMENT stage on the GPU: start location + operation string.
//
// Reference behaviour being reproduced (src/opal.cpp:1475-1507 and findAlignment, :1236-1431):
// for every database entry the query prefix [0, endQ] and the target prefix [0, endT] are reversed,
// a banded, NW-anchored Gotoh DP runs over them until the first column in which a cell that the mode
// allows as an alignment end reaches the known score, and a traceback with the fixed preference
// E, then F, then the diagonal yields the operations.  start = end - (stop cell).
//
// B200 design: no 12-byte Cell matrix.  Kernel 1 (one warp per target, 8 query rows per thread,
// the same systolic wavefront as the search kernel but in exact 32-bit arithmetic) sweeps the reversed
// rectangle once and stores 4 decision bits per cell -- H==E, H==F, "E opened here", "F opened here" --
// i.e. one 32-bit word per (thread, column), plus one byte per word naming the first row whose H
// equals the known score.  It also finds the stop column with the mode's eligibility rule.  Kernel 2
// (one thread per target) walks the decision bits from the stop cell back to the origin and emits the
// operations, which come out directly in alignment order (start -> end).  Only the operation strings
// and four ints per target travel back to the host.
//
// The band (calculateBandBorders, src/opal.cpp:1046-1179) is restated on the host; cells outside it
// are -infinity exactly as in the reference.  Where the reference's own result would be inconsistent
// (its HW/OV stop rule reads the last IN-BAND row as if it were the last row, SURVEY.md 8c Q9) the
// replay check below fails and the target is redone with the full band, which is always correct.
#include "align.h"

#include <algorithm>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace opalb200 {

namespace {

constexpr int kNegInf = -(1 << 30);
constexpr int kRows = 8;  // query rows per thread: 8 cells x 4 bits = one flag word per column

struct AlignTask {
    long long targetOffset;  // residue offset of the target in the sorted device buffer
    long long flagOffset;    // first flag word of this task
    long long eqOffset;      // first eq byte
    long long opsOffset;     // first op byte
    long long bndOffset;     // first boundary int (2 per column)
    int Qp, Tp;              // reversed-problem sizes: endQ + 1, endT + 1
    int endQ, endT;
    int score;
    int bottom, top;         // band
    int rowBlocks;           // ceil(Qp / 8)
    int search;              // its entry in the search table
};

// What the tasks of one search share (device pointers): the query, the entries (the A x A matrix, or with byPssm the
// Q x A PSSM), the mode and the gap penalties.  One launch holds the tasks of every search in the table.
struct AlignSearch {
    const uint8_t* query;
    const int* entries;
    int A, Go, Ge, mode, byPssm;
};

struct AlignOut {
    int stopCol;   // first column reaching the score (INT_MAX if none)
    int endRow;    // row of the stop cell in the reversed problem
    int opsLen;
    int status;    // 0 ok, 1 no stop cell found
};

__device__ __forceinline__ int sat_sub(int x, int g) { return max(x - g, kNegInf); }

// ---------------------------------------------------------------- kernel 1: DP + decision bits
// With a PSSM (pssm non-NULL, Q x A) reversed row r is scored by PSSM row endQ - r instead of the matrix row of its query
// letter; `matrixInSmem` then means that a pass's 32 x kRows rows of it are staged in shared memory.
__global__ void __launch_bounds__(32) align_dp_kernel(const AlignTask* tasks, const AlignSearch* searches, AlignOut* outs,
                                                      const uint8_t* residues, uint32_t* flags, uint8_t* eqRows, int* bnd, int matrixInSmem) {
    extern __shared__ int smemMatrix[];
    const AlignTask task = tasks[blockIdx.x];
    const AlignSearch sr = searches[task.search];
    const uint8_t* query = sr.query;
    const int *matrix = sr.entries, *pssm = sr.byPssm ? sr.entries : nullptr;
    const int A = sr.A, Go = sr.Go, Ge = sr.Ge, mode = sr.mode;
    const int t = threadIdx.x;
    const int* S = pssm ? pssm : matrix;
    if (matrixInSmem && !pssm) {
        for (int i = t; i < A * A; i += 32) smemMatrix[i] = matrix[i];
        __syncwarp();
        S = smemMatrix;
    }
    const int Qp = task.Qp, Tp = task.Tp, bottom = task.bottom, top = task.top, score = task.score;
    const uint8_t* tgt = residues + task.targetOffset;
    const int passes = (Qp + 32 * kRows - 1) / (32 * kRows);
    int stopCol = INT_MAX;
    int* bndH = bnd + task.bndOffset;
    int* bndF = bndH + Tp;

    for (int pass = 0; pass < passes; pass++) {
        const int row0 = (pass * 32 + t) * kRows;  // first reversed-query row of this thread
        const int passRow0 = pass * 32 * kRows;
        if (pssm && matrixInSmem) {  // this pass's PSSM rows, reversed: staged row i = PSSM row endQ - passRow0 - i
            const int n = min(32 * kRows, Qp - passRow0) * A;
            for (int i = t; i < n; i += 32) smemMatrix[i] = pssm[(size_t)(task.endQ - passRow0 - i / A) * A + i % A];
            __syncwarp();
            S = smemMatrix;
        }
        int H[kRows], E[kRows], qoff[kRows];
#pragma unroll
        for (int j = 0; j < kRows; j++) {
            const int r = row0 + j;
            H[j] = -Go - r * Ge;  // column -1 (src/opal.cpp:1266-1269)
            E[j] = kNegInf;
            if (!pssm) qoff[j] = (r < Qp) ? (int)query[task.endQ - r] * A : 0;
            else qoff[j] = (r < Qp) ? (matrixInSmem ? r - passRow0 : task.endQ - r) * A : 0;
        }
        int diag = (row0 == 0) ? 0 : -Go - (row0 - 1) * Ge;  // H[row0-1][-1]; the corner is 0
        int outH = kNegInf, outF = kNegInf;
        const bool lastPass = pass == passes - 1;
        const int steps = Tp + 31;
        for (int s = 0; s < steps; s++) {
            int upH = __shfl_up_sync(0xffffffffu, outH, 1);
            int upF = __shfl_up_sync(0xffffffffu, outF, 1);
            const int c = s - t;
            if (t == 0) {
                if (pass == 0) { upH = -Go - c * Ge; upF = kNegInf; }  // row -1 (src/opal.cpp:1283-1286)
                else if (c < Tp) { upH = bndH[c]; upF = bndF[c]; }
            }
            if (c < 0 || c >= Tp || row0 >= Qp) continue;
            const int y = tgt[task.endT - c];
            int uH = upH, uF = upF, d = diag;
            diag = upH;
            uint32_t word = 0;
            int eq = 255;
            const int r1 = min(Qp - 1, c + bottom);  // last in-band row of this column
#pragma unroll
            for (int j = 0; j < kRows; j++) {
                const int r = row0 + j;
                const bool inBand = r < Qp && r >= c - top && r <= c + bottom;
                const int hl = H[j];
                int e = kNegInf, f = kNegInf, h = kNegInf;
                if (inBand) {
                    e = max(sat_sub(hl, Go), sat_sub(E[j], Ge));
                    f = max(sat_sub(uH, Go), sat_sub(uF, Ge));
                    const int dg = (d <= kNegInf) ? kNegInf : d + S[qoff[j] + y];
                    h = max(max(e, f), dg);
                    if (h < kNegInf / 2) h = kNegInf;  // built from -infinity only
                    if (e < kNegInf / 2) e = kNegInf;
                    if (f < kNegInf / 2) f = kNegInf;
                }
                uint32_t nib = 0;
                if (h == e) nib |= 1u;
                if (h == f) nib |= 2u;
                if (e == hl - Go) nib |= 4u;  // E opened from H of the previous column
                if (f == uH - Go) nib |= 8u;  // F opened from H of the previous row
                word |= nib << (4 * j);
                if (inBand) {
                    if (h == score && eq == 255) eq = j;
                    bool eligible;
                    if (mode == OPAL_MODE_SW) eligible = true;
                    else if (mode == OPAL_MODE_OV) eligible = (r == r1) || (c == Tp - 1);
                    else if (mode == OPAL_MODE_HW) eligible = (r == r1);
                    else eligible = false;
                    if (eligible && h >= score) stopCol = min(stopCol, c);
                }
                uF = f; uH = h; d = hl;
                H[j] = h; E[j] = e;
            }
            outH = uH; outF = uF;
            const long long w = (long long)c * task.rowBlocks + (pass * 32 + t);
            flags[task.flagOffset + w] = word;
            eqRows[task.eqOffset + w] = (uint8_t)eq;
            if (!lastPass && t == 31) { bndH[c] = outH; bndF[c] = outF; }
        }
        __syncwarp();
    }
    // first column in which an eligible cell reaches the score (src/opal.cpp:1275)
    for (int o = 16; o > 0; o >>= 1) stopCol = min(stopCol, __shfl_xor_sync(0xffffffffu, stopCol, o));
    if (mode == OPAL_MODE_NW) stopCol = Tp - 1;
    if (t == 0) {
        AlignOut o;
        o.stopCol = stopCol; o.endRow = -1; o.opsLen = 0; o.status = (stopCol == INT_MAX) ? 1 : 0;
        outs[blockIdx.x] = o;
    }
}

// ---------------------------------------------------------------- kernel 2: traceback
__global__ void align_traceback_kernel(const AlignTask* tasks, const AlignSearch* searches, AlignOut* outs, int numTasks,
                                       const uint8_t* residues, const uint32_t* flags, const uint8_t* eqRows, uint8_t* ops) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= numTasks) return;
    const AlignTask task = tasks[i];
    AlignOut o = outs[i];
    if (o.status != 0) return;
    const uint8_t* query = searches[task.search].query;
    const int mode = searches[task.search].mode;
    const int ce = o.stopCol;
    int re;
    if (mode == OPAL_MODE_NW || mode == OPAL_MODE_HW) re = task.Qp - 1;  // src/opal.cpp:1341-1350
    else {  // SW, OV: first row of the stop column whose H equals the score (:1351-1358)
        re = -1;
        for (int b = 0; b < task.rowBlocks && re < 0; b++) {
            const int e = eqRows[task.eqOffset + (long long)ce * task.rowBlocks + b];
            if (e != 255) re = b * kRows + e;
        }
        if (re < 0) { o.status = 1; outs[i] = o; return; }
    }
    const uint8_t* tgt = residues + task.targetOffset;
    uint8_t* out = ops + task.opsOffset;
    int n = 0, ri = re, ci = ce, field = 0;  // 0 = H, 1 = E, 2 = F
    while (ri >= 0 && ci >= 0) {  // src/opal.cpp:1372-1399
        const uint32_t word = flags[task.flagOffset + (long long)ci * task.rowBlocks + (ri >> 3)];
        const uint32_t nib = (word >> (4 * (ri & 7))) & 15u;
        if (field == 0) {
            if (nib & 1u) field = 1;
            else if (nib & 2u) field = 2;
            else {
                out[n++] = (query[task.endQ - ri] == tgt[task.endT - ci]) ? OPAL_ALIGN_MATCH : OPAL_ALIGN_MISMATCH;
                ci--; ri--;
            }
        } else if (field == 1) {
            field = (nib & 4u) ? 0 : 1;
            out[n++] = OPAL_ALIGN_INS; ci--;
        } else {
            field = (nib & 8u) ? 0 : 2;
            out[n++] = OPAL_ALIGN_DEL; ri--;
        }
    }
    while (ri >= 0) { out[n++] = OPAL_ALIGN_DEL; ri--; }  // :1402-1405
    while (ci >= 0) { out[n++] = OPAL_ALIGN_INS; ci--; }  // :1406-1409
    o.endRow = re; o.opsLen = n;
    outs[i] = o;
}

// ---------------------------------------------------------------- band (host), src/opal.cpp:1046-1179
typedef long long i64;
int gap_penalty(int len, int Go, int Ge) { return len > 0 ? Go + Ge * (len - 1) : 0; }
int tdiv(i64 num, i64 den, bool* bad) {
    if (den == 0) { *bad = true; return 0; }
    i64 v = num / den;
    return (int)std::max<i64>(INT_MIN, std::min<i64>(INT_MAX, v));
}
int bottom_ov(int k, int Q, int T, int Go, int Ge, int M, bool* bad) {  // :1057-1070
    int border = std::max(0, std::min(Q - T, tdiv(-1 * ((i64)k + Go - Ge - (i64)M * T), Ge, bad)));
    const int cand = tdiv(-1 * ((i64)k - (i64)M * Q + Go - Ge), (i64)Ge + M, bad);
    if (cand > Q - T) border = std::max(border, cand);
    return std::min(border, Q - 1);
}
int top_hw(int k, int Q, int T, int Go, int Ge, int M, bool* bad) {  // :1072-1085
    const int v = tdiv(-1 * ((i64)k - (i64)M * Q + Go), Ge, bad);
    int border = std::max(0, std::min(T - Q, v == INT_MAX ? v : v + 1));
    const int cand = tdiv(-1 * ((i64)k - (i64)T * M + 2 * (i64)Go + (i64)Ge * (Q - T - 2)), 2 * (i64)Ge + M, bad);
    if (cand > T - Q) border = std::max(border, cand);
    return std::min(border, T - 1);
}
int bottom_hw(int k, int Q, int T, int Go, int Ge, int M, bool* bad) {  // :1087-1102
    int border = 0;
    const int cand = tdiv(-1 * ((i64)k + Go - Ge - (i64)Q * M), (i64)Ge + M, bad);
    if (cand >= Q - T) border = std::max(border, cand);
    if (-2 * (i64)Go - (i64)Ge * (Q - T - 2) + (i64)M * T >= k) border = std::max(border, Q - T - 1);
    return std::min(border, Q - 1);
}
int bottom_nw(int k, int Q, int T, int Go, int Ge, int M, bool* bad) {  // :1104-1124
    int border = 0;
    const int cand = tdiv(-1 * ((i64)k + 2 * (i64)Go - (i64)M * Q + (i64)Ge * (T - Q - 2)), 2 * (i64)Ge + M, bad);
    if (cand > Q - T) border = std::max(border, cand);
    if (Q - T <= tdiv(-1 * ((i64)k + Go - (i64)M * T - Ge), Ge, bad)) border = std::max(border, Q - T);
    if (-2 * (i64)Go - (i64)Ge * (Q - T - 2) + (i64)M * T >= k) border = std::max(border, Q - T - 1);
    return std::min(border, Q - 1);
}
// Returns false when the reference would have no band (or would divide by zero): use the full matrix.
bool band_borders(int k, int mode, int Q, int T, int Go, int Ge, int M, int* bottom, int* top) {  // :1151-1179
    bool bad = false;
    const int m = std::min(Q, T);
    if (mode == OPAL_MODE_OV || mode == OPAL_MODE_SW) {
        if ((i64)M * m < k) return false;
        *bottom = bottom_ov(k, Q, T, Go, Ge, M, &bad);
        *top = bottom_ov(k, T, Q, Go, Ge, M, &bad);
    } else if (mode == OPAL_MODE_HW) {
        if ((i64)M * m - gap_penalty(Q - m, Go, Ge) < k) return false;
        *bottom = bottom_hw(k, Q, T, Go, Ge, M, &bad);
        *top = top_hw(k, Q, T, Go, Ge, M, &bad);
    } else {
        if ((i64)M * m - gap_penalty(std::abs(Q - T), Go, Ge) < k) return false;
        *bottom = bottom_nw(k, Q, T, Go, Ge, M, &bad);
        *top = bottom_nw(k, T, Q, Go, Ge, M, &bad);
    }
    return !bad && *bottom >= 0 && *bottom < Q && *top >= 0 && *top < T;
}

// Replay of an operation string (the check of reference src/test.cpp:348-422): does it start at
// (sq, st), end at (endQ, endT) and score exactly `score` under s?
bool replay_ok(const Scoring& s, const unsigned char* t, int T, const unsigned char* ops, int n, int sq, int st, int endQ, int endT,
               int score) {
    i64 sc = 0;
    int qi = sq, ti = st, prev = -1;
    if (qi < 0 || ti < 0) return false;
    for (int i = 0; i < n; i++) {
        const int op = ops[i];
        if ((op != OPAL_ALIGN_DEL && ti >= T) || (op != OPAL_ALIGN_INS && qi >= s.Q)) return false;
        if (op == OPAL_ALIGN_MATCH) { if (s.query[qi] != t[ti]) return false; sc += s.cell(qi, t[ti]); qi++; ti++; }
        else if (op == OPAL_ALIGN_MISMATCH) { if (s.query[qi] == t[ti]) return false; sc += s.cell(qi, t[ti]); qi++; ti++; }
        else if (op == OPAL_ALIGN_DEL) { sc -= (prev == OPAL_ALIGN_DEL ? s.Ge : s.Go); qi++; }
        else if (op == OPAL_ALIGN_INS) { sc -= (prev == OPAL_ALIGN_INS ? s.Ge : s.Go); ti++; }
        else return false;
        prev = op;
    }
    return qi - 1 == endQ && ti - 1 == endT && sc == score;
}

#define ALIGN_TRY(expr)                                                                          \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) { set_error(std::string(#expr) + ": " + cudaGetErrorString(_e)); ok = false; goto done; } \
    } while (0)

#define ALIGN_OK(expr)                      \
    do {                                    \
        if (!(expr)) { ok = false; goto done; } \
    } while (0)

}  // namespace

int align_database(DeviceDb* ddb, const std::vector<AlignSet>& sets, unsigned char* const* db, const int* lens) {
    if (!ddb || !ddb->ensure_uploaded()) return OPAL_B200_ERR_CUDA;
    const int ns = (int)sets.size();
    // target of record j of search q on the host: the caller's pointer, or (resident-handle calls) the database's own
    // sorted copy; the record describes database entry entry(q, j): all of them, or the search's subset (top-k pipelines)
    auto entry = [&](int q, int j) { return sets[q].subset ? sets[q].subset[j] : j; };
    auto target_len = [&](int q, int j) { return lens ? lens[entry(q, j)] : ddb->sorted_lengths()[ddb->sorted_position()[entry(q, j)]]; };
    auto target_ptr = [&](int q, int j) -> const unsigned char* {
        return db ? db[entry(q, j)] : ddb->h_residues() + ddb->offsets()[ddb->sorted_position()[entry(q, j)]];
    };
    std::vector<int> M((size_t)ns);  // the band's M of every search: the largest entry that can score a cell

    // ---- entries that have an alignment at all (src/opal.cpp:1479-1483)
    struct Item { int q, j; };
    std::vector<Item> todo;
    for (int q = 0; q < ns; q++) {
        const Scoring& s = *sets[q].s;
        M[q] = s.bounds().maxEntry;
        for (int j = 0; j < sets[q].n; j++) {
            OpalSearchResult* r = sets[q].results[j];
            if ((s.mode == OPAL_MODE_SW && r->score == 0) || r->endLocationQuery < 0 || r->endLocationTarget < 0 ||
                r->endLocationQuery >= s.Q || r->endLocationTarget >= target_len(q, j)) {
                r->alignment = NULL;
                r->alignmentLength = 0;
                r->startLocationQuery = r->startLocationTarget = -1;
                r->endLocationQuery = r->endLocationTarget = -1;
            } else {
                todo.push_back({q, j});
            }
        }
    }
    if (todo.empty()) return 0;

    const cudaStream_t stream = ddb->stream();
    cudaSetDevice(ddb->device());
    bool ok = true;
    unsigned char* dArgs = nullptr;  // [search table | entries and query of every search]
    AlignTask* dTasks = nullptr;
    AlignOut* dOuts = nullptr;
    uint32_t* dFlags = nullptr;
    uint8_t *dEq = nullptr, *dOps = nullptr;
    int* dBnd = nullptr;
    std::vector<unsigned char> hOps;
    std::vector<AlignOut> hOuts;
    // the table, then every search's entries (searches that share one matrix share one copy) and query: one upload
    auto up16 = [](size_t x) { return (x + 15) / 16 * 16; };
    std::vector<size_t> entOff((size_t)ns), qOff((size_t)ns);
    size_t argsBytes = up16(sizeof(AlignSearch) * (size_t)ns), smemBytes = 0;
    for (int q = 0; q < ns; q++) {
        const Scoring& s = *sets[q].s;
        entOff[q] = 0;
        for (int p = 0; p < q && !entOff[q]; p++)
            if (sets[p].s->entries == s.entries && sets[p].s->num_entries() == s.num_entries()) entOff[q] = entOff[p];
        if (!entOff[q]) { entOff[q] = argsBytes; argsBytes += up16(sizeof(int) * (size_t)s.num_entries()); }
        qOff[q] = argsBytes;
        argsBytes += up16((size_t)s.Q + 16);
        // matrix, or a pass's 32 x kRows PSSM rows, in shared memory when it fits
        smemBytes = std::max(smemBytes, sizeof(int) * (size_t)s.A * (s.byPssm ? 32 * kRows : s.A));
    }
    const int matrixInSmem = smemBytes <= 40000 ? 1 : 0;
    std::vector<unsigned char> hArgs(argsBytes, 0);
    size_t freeB = 0, totalB = 0;
    cudaMemGetInfo(&freeB, &totalB);
    const long long budgetWords = (long long)std::max<size_t>(64u << 20, std::min<size_t>(freeB / 3, (size_t)16 << 30)) / 4;

    const int dev = ddb->device();
    auto dalloc = [&](void* pp, size_t bytes) { return device_alloc(dev, (void**)pp, bytes); };
    auto release_batch = [&]() {
        device_release(dev, dTasks); device_release(dev, dOuts); device_release(dev, dFlags); device_release(dev, dEq);
        device_release(dev, dOps); device_release(dev, dBnd);
        dTasks = nullptr; dOuts = nullptr; dFlags = nullptr; dEq = nullptr; dOps = nullptr; dBnd = nullptr;
    };
    ALIGN_OK(dalloc(&dArgs, argsBytes));
    for (int q = 0; q < ns; q++) {
        const Scoring& s = *sets[q].s;
        const AlignSearch sr{dArgs + qOff[q], reinterpret_cast<const int*>(dArgs + entOff[q]), s.A, s.Go, s.Ge, s.mode, s.byPssm ? 1 : 0};
        memcpy(hArgs.data() + sizeof(AlignSearch) * q, &sr, sizeof(sr));
        if (s.num_entries() > 0) memcpy(hArgs.data() + entOff[q], s.entries, sizeof(int) * (size_t)s.num_entries());
        if (s.Q > 0 && s.query) memcpy(hArgs.data() + qOff[q], s.query, (size_t)s.Q);
    }
    ALIGN_TRY(cudaMemcpyAsync(dArgs, hArgs.data(), argsBytes, cudaMemcpyHostToDevice, stream));

    {
        // Two rounds at most: the reference's band first, the full band for entries whose replay fails.
        std::vector<Item> pending = todo;
        for (int round = 0; round < 2 && !pending.empty(); round++) {
            std::vector<Item> failed;
            size_t cursor = 0;
            while (cursor < pending.size()) {
                // ---- one batch within the memory budget
                std::vector<AlignTask> tasks;
                std::vector<Item> ids;
                long long flagWords = 0, opsBytes = 0, bndInts = 0;
                while (cursor < pending.size()) {
                    const Item it = pending[cursor];
                    const Scoring& s = *sets[it.q].s;
                    const OpalSearchResult* r = sets[it.q].results[it.j];
                    AlignTask tk;
                    tk.Qp = r->endLocationQuery + 1; tk.Tp = r->endLocationTarget + 1;
                    tk.endQ = r->endLocationQuery; tk.endT = r->endLocationTarget; tk.score = r->score;
                    tk.rowBlocks = (tk.Qp + kRows - 1) / kRows;
                    tk.search = it.q;
                    const long long words = (long long)tk.rowBlocks * tk.Tp;
                    if (!tasks.empty() && flagWords + words > budgetWords) break;
                    if (round == 0 && band_borders(tk.score, s.mode, tk.Qp, tk.Tp, s.Go, s.Ge, M[it.q], &tk.bottom, &tk.top)) {}
                    else { tk.bottom = tk.Qp - 1; tk.top = tk.Tp - 1; }
                    tk.targetOffset = ddb->offsets()[ddb->sorted_position()[entry(it.q, it.j)]];
                    tk.flagOffset = flagWords; tk.eqOffset = flagWords; tk.opsOffset = opsBytes; tk.bndOffset = bndInts;
                    flagWords += words; opsBytes += tk.Qp + tk.Tp + 8; bndInts += 2LL * tk.Tp;
                    tasks.push_back(tk); ids.push_back(it);
                    cursor++;
                }
                const int nt = (int)tasks.size();
                release_batch();  // the previous batch was synchronised before its results were read
                ALIGN_OK(dalloc(&dTasks, sizeof(AlignTask) * nt));
                ALIGN_OK(dalloc(&dOuts, sizeof(AlignOut) * nt));
                ALIGN_OK(dalloc(&dFlags, sizeof(uint32_t) * (size_t)flagWords));
                ALIGN_OK(dalloc(&dEq, (size_t)flagWords));
                ALIGN_OK(dalloc(&dOps, (size_t)opsBytes));
                ALIGN_OK(dalloc(&dBnd, sizeof(int) * (size_t)std::max<long long>(bndInts, 1)));
                ALIGN_TRY(cudaMemcpyAsync(dTasks, tasks.data(), sizeof(AlignTask) * nt, cudaMemcpyHostToDevice, stream));
                // an alignment is shorter than its slot: the unused tail travels back with the rest, so it is defined
                ALIGN_TRY(cudaMemsetAsync(dOps, 0, (size_t)opsBytes, stream));
                const AlignSearch* dSearches = reinterpret_cast<const AlignSearch*>(dArgs);
                align_dp_kernel<<<nt, 32, matrixInSmem ? smemBytes : 0, stream>>>(dTasks, dSearches, dOuts, ddb->d_residues(), dFlags, dEq,
                                                                                   dBnd, matrixInSmem);
                ALIGN_TRY(cudaGetLastError());
                align_traceback_kernel<<<(nt + 63) / 64, 64, 0, stream>>>(dTasks, dSearches, dOuts, nt, ddb->d_residues(), dFlags, dEq, dOps);
                ALIGN_TRY(cudaGetLastError());
                hOps.resize((size_t)opsBytes);
                hOuts.resize(nt);
                ALIGN_TRY(cudaMemcpyAsync(hOps.data(), dOps, (size_t)opsBytes, cudaMemcpyDeviceToHost, stream));
                ALIGN_TRY(cudaMemcpyAsync(hOuts.data(), dOuts, sizeof(AlignOut) * nt, cudaMemcpyDeviceToHost, stream));
                ALIGN_TRY(cudaStreamSynchronize(stream));
                for (int k = 0; k < nt; k++) {
                    const Item it = ids[k];
                    OpalSearchResult* r = sets[it.q].results[it.j];
                    const AlignOut& o = hOuts[k];
                    const AlignTask& tk = tasks[k];
                    const unsigned char* ops = hOps.data() + tk.opsOffset;
                    const int sq = tk.endQ - o.endRow, st = tk.endT - o.stopCol;  // src/opal.cpp:1499-1500
                    const bool good = o.status == 0 && replay_ok(*sets[it.q].s, target_ptr(it.q, it.j), target_len(it.q, it.j), ops, o.opsLen, sq,
                                                                 st, tk.endQ, tk.endT, tk.score);
                    if (!good && round == 0 && (tk.bottom != tk.Qp - 1 || tk.top != tk.Tp - 1)) { failed.push_back(it); continue; }
                    if (o.status != 0) {  // prefilled score / end inconsistent with the sequences: no alignment exists
                        r->alignment = NULL; r->alignmentLength = 0;
                        r->startLocationQuery = r->startLocationTarget = -1;
                        continue;
                    }
                    r->startLocationQuery = sq;
                    r->startLocationTarget = st;
                    r->alignmentLength = o.opsLen;
                    r->alignment = (unsigned char*)malloc((size_t)std::max(o.opsLen, 1));
                    memcpy(r->alignment, ops, (size_t)o.opsLen);
                }
            }
            pending.swap(failed);
        }
    }
done:
    cudaStreamSynchronize(stream);  // nothing may still be using the blocks when they go back to the cache
    device_release(dev, dArgs);
    release_batch();
    return ok ? 0 : OPAL_B200_ERR_CUDA;
}

}  // namespace opalb200
