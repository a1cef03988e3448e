// search_kernel.cuh -- the score / score+end kernel of opal-b200 (sm_100a).
//
// Replaces the reference's inter-sequence SIMD passes
//   searchDatabaseSW_<SimdSW<T>>      (reference src/opal.cpp:164-470)
//   searchDatabase_<Simd<T>, MODE>    (reference src/opal.cpp:594-977)
// with one kernel template.  It is not a port of the lane-per-sequence column sweep: a GROUP of G
// threads (G = 1..32, a power of two) owns one target pair and sweeps it as a systolic wavefront.
//
//   * thread t of the group holds R consecutive query rows in registers (H - gapOpen and E per
//     row), so a group covers G*R query rows per pass; longer queries take several passes with
//     the boundary row (H, F per target column) parked in HBM between passes;
//   * at step s thread t computes target column s - t; the bottom (H, F) of its strip travels
//     to thread t+1 with one rotating __shfl_sync per value, so no DP state ever leaves registers
//     within a pass (the rotation also serves the folded sweep, SearchParams::folded, in which one
//     target fills both 16-bit lanes of a warp and thread 31's low lane feeds thread 0's high lane);
//   * the two 16-bit halves of every register hold two DIFFERENT targets (Rognes/Opal style), and
//     the recurrence is issued as packed DPX instructions: VIADDMNMX.S16x2 (E, F, diagonal+max),
//     VIMNMX.S16x2, VIADD.16x2;  the 32-bit re-run uses the s32 forms of the same instructions;
//   * substitution scores come from a query profile in shared memory laid out thread-major
//     (each thread's R rows contiguous, thread stride an odd number of 16-byte units) in two
//     planes -- scores in the low half-word / in the high half-word -- so a packed score is
//     LDS.128 + LDS.128 + one IMAD-pipe add per 4 rows, bank-conflict free for any residues.
//
// Arithmetic notes (all integer):
//   HG = H - gapOpen is what is stored; the profile is pre-biased by +gapOpen, so
//   diag + P == HG_diag + P'.  DPX adds wrap (they do not saturate), therefore 16-bit safety is
//   established by bounds: SW flags a target whose best exceeds 32767 - maxScore - 1 (it is then
//   re-run in 32 bits, mirroring the reference's char -> short -> int ladder, src/opal.cpp:512-530);
//   NW/HW/OV targets are routed by an a-priori bound on the host (engine.cu).
//
// End-location key (reference src/opal.h:43-45 and SURVEY.md section 0 fact 3): maximal score, then
// smallest target index, then smallest query index -- tracked per thread with strict improvements
// in column-major order and merged across threads / passes with that key.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <type_traits>

namespace opalb200 {

// Threads per block the kernels are compiled for = 128 x the warps that may share a scheduler partition.  Three
// warps per partition (cap of 170 registers) give 6 - 20 % more throughput than two (tools/steptime_probe.py); a
// fourth adds nothing and would need a 128-register cap.  The NW/HW/OV flavor at the tallest strips wants more
// than 170 registers: it is compiled twice, uncapped for one or two warps per partition (where the cap costs up to
// 25 %) and capped for three (+10 % throughput over two uncapped).
constexpr int launch_bound_for(int flavor, int R) { return (flavor == 2 && R > 24) ? 256 : 384; }
constexpr int kModeNW = 0, kModeHW = 1, kModeOV = 2, kModeSW = 3;
// NW / HW / OV sweeps handle their rare per-column events (result cell, last-column scan, start of the high half-words
// of a folded task) behind ONE compare per step against the nearest event.  Measured on B200 this form is 13 % faster
// than separate compares at 18 rows and 3 - 7 % SLOWER at 24 - 33 (the event block inflates the loop; register
// allocation at the 170-register cap), so the tall strips keep the separate compares -- and do not take folded
// NW / HW / OV tasks.
__host__ __device__ constexpr bool single_event_compare(int R) { return R <= 18; }
constexpr int kFlavorSWScore = 0, kFlavorSWEnd = 1, kFlavorGlobal = 2, kFlavorSWEndFast = 3;
constexpr int kRowBits = 6;  // kFlavorSWEndFast: low bits of the tracked key hold 63 - row (latch_key_s16x2 spells the mask out)
static_assert(kRowBits == 6, "latch_key_s16x2 saturates the row bits with 0x003f003f");
constexpr int kScoreNone = INT32_MIN;          // "no candidate yet" in the running-result arrays
constexpr int kScoreOverflow = INT32_MIN + 1;  // 16-bit pass: re-run this target in 32 bits

struct SearchParams {
    // query side
    const uint8_t* query;  // Q alphabet indices
    const int* matrix;     // score rows read by the profile build: A*A, row = query letter (PSSM search: the PSSM, row = query row)
    int Q, A, gapOpen, gapExt, mode, wantEnd;
    // geometry of this pass
    int G, rowBase, padTop, pass, numPasses, rowStride, Rpad;
    // database, device resident, length-sorted (longest first):
    //   plain:  residues back to back + offsets/lengths per target          (32-bit class, alignment stage)
    //   paired: targets 2p and 2p+1 interleaved column by column as uint16 = (res0 + 1) | (res1 + 1) << 8,
    //           0 = "no residue"; every pair is preceded and followed by >= 32 zero entries, so a
    //           wavefront may read 31 columns before / after a pair without bounds checks
    const uint8_t* residues;
    const long long* offsets;
    const int* lengths;
    const uint16_t* pairStream;
    const long long* pairOffsets;
    int numTargets;       // targets in the database (the last pair may have one member)
    // work: Packed16 tasks are pair indices, Scalar32 tasks are target indices (taskList null = 0..numTasks-1)
    const int* taskList;
    int taskBase;         // first task when taskList is null
    int numTasks;
    int* counter;
    // boundary row between passes, indexed by residue offset of the task's first target + column; a pass
    // reads the previous pass's rows from bndIn* and writes its own to bndOut* (ping-pong, so that a warp may
    // sweep a task twice)
    const void* bndInH;
    const void* bndInF;
    void* bndOutH;
    void* bndOutF;
    // running results, indexed by sorted-target index
    int* outScore;
    int* outEndQ;
    int* outEndT;
    int overflowLimit;  // SW: largest best that is still provably exact at this width
    int padLetterScore; // profile value of the pad letter (before the +gapOpen bias)
    int one;            // the constant 1, opaque to the compiler (see vimax_track_s16x2)
    int keyScale;       // 1 << kRowBits, opaque to the compiler so that the key is built by an IMAD (FMA pipe)
    int fastEndLimit;   // kFlavorSWEndFast: tracked scores at or above this are re-run by the exact flavor
    // Folded tasks (Packed16, G = 32, one pass): ONE target occupies both half-words.  The low halves of the
    // warp hold query rows [0, 32 R), the high halves rows [32 R, 64 R) of the SAME target 32 columns behind, so
    // the warp is a 64-deep wavefront: what leaves the low half of thread 31 enters the high half of thread 0 one
    // step later.  Half the rows per thread means a much shorter step -- this is how the longest targets of a
    // database, which bound the time of a search (each is swept by one warp), are finished sooner.  Tasks are
    // sorted-target indices; pairStream / pairOffsets then point at the folded stream, whose entry c of a
    // target is (res[c] + 1) | (res[c - 32] + 1) << 8 over T + 32 columns, padded like a pair.
    int folded;
    // NW / HW / OV at 16 bits: H of every strip's last row is sampled in every column; a target whose samples leave
    // [rangeLo, rangeHi] is flagged and re-run at 32 bits (see range tracking in the sweep).
    int rangeHi, rangeLo;
    // Chained passes (the latency class of a query that takes several passes): ALL passes of a task run in one launch,
    // each on a warp of its own -- block b sweeps pass b % numPasses of the tasks of quad b / numPasses -- and the
    // boundary row travels from the warp of pass p to the warp of pass p + 1 through HBM / L2 while both are sweeping.
    // The rows start out filled with a value no cell can take (kChainEmpty); the consumer reads them 32 columns at a
    // time, two chunks ahead of its first thread, and waits while a chunk still holds that value -- no fence, no
    // counter: a 32-bit store is atomic, and the producer writes every entry exactly once.
    // The longest target of a database then costs its length in steps ONCE instead of once per pass.
    // bndOutH / bndOutF hold numPasses rows of chainStride entries, chainOffsets[task] is a task's place in a row.
    int chain;
    int chainStride;
    const int* chainOffsets;
    int* chainDone;       // [task * numPasses + pass]: that pass has written its results
    int* chainTicket;     // blocks take their place in the chain in the order they START (so a producer is never behind its consumer)
    // Position-specific scoring matrix, Q x A row-major (row r = scores of query position r against every target letter),
    // or NULL.  When set, `matrix` points at it as well and the profile build takes row r for query row r instead of the
    // row of query letter query[r]; `query` is unused.  (Last member: the sweep's parameter offsets stay where they were.)
    const int* pssm;
};
// Chained passes: "not written yet" in a boundary row.  Both half-words -32768 (or INT_MIN at 32 bits) lies outside
// every range the kernels guarantee; a sweep that has already left that range (its target is flagged and re-run at 32
// bits anyway) could still produce the pattern by accident, so the producer never stores it (it stores the pattern + 1).
constexpr uint32_t kChainEmpty = 0x80008000u;
constexpr uint32_t kChainEmpty32 = 0x80000000u;
constexpr int kFoldLag = 32;  // columns between the two halves of a folded task = depth of one warp's wavefront

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t addr) {
    uint2 v;
    asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// One residue code of the paired stream, zero-extended by the load itself (a 16-bit load of both codes costs
// a mask, a second mask and a shift on the integer pipe per step; two byte loads cost nothing there).
__device__ __forceinline__ uint32_t ldg_u8(const uint8_t* p) {
    uint32_t v;
    asm("ld.global.nc.u8 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// Chained passes: loads that must see what another SM has just written (L1 is not coherent), and the flag accesses.
__device__ __forceinline__ uint32_t ld_cg_u32(const void* p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_gpu_u32(void* p, uint32_t v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

// a * m + b with m a run-time 0 / 1: a select issued as one IMAD on the FMA pipe instead of a compare and a
// SEL on the integer pipe, where they would compete with the DPX instructions.
__device__ __forceinline__ uint32_t blend_fma(uint32_t a, uint32_t m, uint32_t b) { return a * m + b; }

// kFlavorSWEndFast, end of a column: where a half-word of `best` changed, latch the column and the key (its low
// bits name the row); then saturate the row bits.  Two LOP3 with predicate outputs, four SEL and one OR (ptxas turns
// predicated moves and multiplies alike into SEL); the row is extracted from the latched key once, after the sweep.
__device__ __forceinline__ uint32_t latch_key_s16x2(uint32_t best, uint32_t before, int c, int& colLo, int& colHi,
                                                    uint32_t& keyLo, uint32_t& keyHi) {
    uint32_t out;
    asm("{.reg .pred pl, ph;\n\t"
        ".reg .b32 x, l, h;\n\t"
        "xor.b32 x, %5, %6;\n\t"
        "and.b32 l, x, 0xffff;\n\t"
        "and.b32 h, x, 0xffff0000;\n\t"
        "setp.ne.u32 pl, l, 0;\n\t"
        "setp.ne.u32 ph, h, 0;\n\t"
        "@pl mov.b32 %1, %7;\n\t"
        "@ph mov.b32 %2, %7;\n\t"
        "@pl mov.b32 %3, %5;\n\t"
        "@ph mov.b32 %4, %5;\n\t"
        "or.b32 %0, %5, 0x003f003f;}\n\t"
        : "=&r"(out), "+r"(colLo), "+r"(colHi), "+r"(keyLo), "+r"(keyHi)
        : "r"(best), "r"(before), "r"(c));
    return out;
}

// Packed max with per-half "a is still the max" predicates (a >= b).
// CUDA 12.9's __vibmax_s16x2 (crt/device_functions.hpp:964-983) declares its result "=r" without an
// early clobber and re-reads operand a after writing it, so `x = __vibmax_s16x2(x, ...)` can be
// assigned one register for both and then always reports "no improvement".  Same PTX, but the
// result goes through a private temporary and the outputs are written last; ptxas still fuses it
// into one VIMNMX.S16x2 with two predicate destinations.
__device__ __forceinline__ uint32_t vibmax_s16x2(uint32_t a, uint32_t b, bool* pred_hi, bool* pred_lo) {
    uint32_t val, ph, pl;
    asm("{.reg .pred pu, pv;\n\t"
        ".reg .s16 rs0, rs1, rs2, rs3;\n\t"
        ".reg .b32 t;\n\t"
        "max.s16x2 t, %3, %4;\n\t"
        "mov.b32 {rs0, rs1}, t;\n\t"
        "mov.b32 {rs2, rs3}, %3;\n\t"
        "setp.eq.s16 pv, rs0, rs2;\n\t"
        "setp.eq.s16 pu, rs1, rs3;\n\t"
        "selp.b32 %1, 1, 0, pu;\n\t"
        "selp.b32 %2, 1, 0, pv;\n\t"
        "mov.b32 %0, t;}\n\t"
        : "=&r"(val), "=&r"(ph), "=&r"(pl)
        : "r"(a), "r"(b));
    *pred_hi = (bool)ph;
    *pred_lo = (bool)pl;
    return val;
}

// best = max(best, x) per half-word; where a half strictly improves, its row register takes `row`.
// One VIMNMX.S16x2 with two predicate outputs plus two predicated IMADs: `one` is a run-time 1, so the
// row update is a multiply on the FMA pipe instead of a SEL competing with the DPX work on the integer pipe.
__device__ __forceinline__ uint32_t vimax_track_s16x2(uint32_t best, uint32_t x, int& rowLo, int& rowHi, int row, int one) {
    uint32_t val;
    asm("{.reg .pred pu, pv;\n\t"
        ".reg .s16 rs0, rs1, rs2, rs3;\n\t"
        ".reg .b32 t;\n\t"
        "max.s16x2 t, %3, %4;\n\t"
        "mov.b32 {rs0, rs1}, t;\n\t"
        "mov.b32 {rs2, rs3}, %3;\n\t"
        "setp.eq.s16 pv, rs0, rs2;\n\t"
        "setp.eq.s16 pu, rs1, rs3;\n\t"
        "@!pv mul.lo.s32 %1, %6, %5;\n\t"
        "@!pu mul.lo.s32 %2, %6, %5;\n\t"
        "mov.b32 %0, t;}\n\t"
        : "=&r"(val), "+r"(rowLo), "+r"(rowHi)
        : "r"(best), "r"(x), "r"(row), "r"(one));
    return val;
}

// ---------------------------------------------------------------- arithmetic traits
struct Packed16 {
    typedef uint32_t reg;
    static constexpr int LANES = 2;
    static constexpr int NEG = -30000;
    static __device__ __forceinline__ reg splat(int v) { uint32_t u = (uint32_t)v & 0xffffu; return u | (u << 16); }
    static __device__ __forceinline__ reg pack(int lo, int hi) { return ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16); }
    static __device__ __forceinline__ int lane(reg v, int l) { return l ? ((int)v >> 16) : (int)(short)(v & 0xffffu); }
    static __device__ __forceinline__ reg addmax(reg a, reg b, reg c) { return __viaddmax_s16x2(a, b, c); }
    static __device__ __forceinline__ reg addmax_relu(reg a, reg b, reg c) { return __viaddmax_s16x2_relu(a, b, c); }
    static __device__ __forceinline__ reg vmax(reg a, reg b) { return __vmaxs2(a, b); }
    static __device__ __forceinline__ reg vmin(reg a, reg b) { return __vmins2(a, b); }
    static __device__ __forceinline__ reg vmax3(reg a, reg b, reg c) { return __vimax3_s16x2(a, b, c); }
    static __device__ __forceinline__ reg add(reg a, reg b) { return __vadd2(a, b); }
    static __device__ __forceinline__ reg bmax(reg a, reg b, bool* phi, bool* plo) { return vibmax_s16x2(a, b, phi, plo); }
    static __device__ __forceinline__ reg track(reg best, reg x, int& rowLo, int& rowHi, int row, int one) { return vimax_track_s16x2(best, x, rowLo, rowHi, row, one); }
    static __device__ __forceinline__ reg combine(uint32_t lo, uint32_t hi) { return lo + hi; }
    static __device__ __forceinline__ reg blend(reg a, uint32_t m, reg b) { return blend_fma(a, m, b); }
};

struct Scalar32 {
    typedef int reg;
    static constexpr int LANES = 1;
    static constexpr int NEG = -1500000000;
    static __device__ __forceinline__ reg splat(int v) { return v; }
    static __device__ __forceinline__ reg pack(int lo, int) { return lo; }
    static __device__ __forceinline__ int lane(reg v, int) { return v; }
    static __device__ __forceinline__ reg addmax(reg a, reg b, reg c) { return __viaddmax_s32(a, b, c); }
    static __device__ __forceinline__ reg addmax_relu(reg a, reg b, reg c) { return __viaddmax_s32_relu(a, b, c); }
    static __device__ __forceinline__ reg vmax(reg a, reg b) { return max(a, b); }
    static __device__ __forceinline__ reg vmin(reg a, reg b) { return min(a, b); }
    static __device__ __forceinline__ reg vmax3(reg a, reg b, reg c) { return __vimax3_s32(a, b, c); }
    static __device__ __forceinline__ reg add(reg a, reg b) { return a + b; }
    static __device__ __forceinline__ reg bmax(reg a, reg b, bool* phi, bool* plo) { *phi = true; return __vibmax_s32(a, b, plo); }
    static __device__ __forceinline__ reg track(reg best, reg x, int& rowLo, int&, int row, int) {
        bool keep;
        const reg v = __vibmax_s32(best, x, &keep);
        if (!keep) rowLo = row;
        return v;
    }
    static __device__ __forceinline__ reg combine(uint32_t lo, uint32_t) { return (int)lo; }
    static __device__ __forceinline__ reg blend(reg a, uint32_t m, reg b) { return (int)blend_fma((uint32_t)a, m, (uint32_t)b); }
};

// Column -1 of the DP matrix (reference src/opal.cpp:247-249 for SW, :671-679 for the others);
// rows above the query (padding, r < 0) and the corner behave as H = 0.
__device__ __forceinline__ int border_h(int mode, int r, int Go, int Ge) {
    if (mode == kModeSW || mode == kModeOV || r < 0) return 0;
    return -Go - r * Ge;
}

// Lexicographic "is candidate (s, c, r) better than (S, C, R)" under the end-location key.
__device__ __forceinline__ bool better(int s, int c, int r, int S, int C, int R) {
    if (s != S) return s > S;
    if (c != C) return c < C;
    return r < R;
}

// ---------------------------------------------------------------- the kernel
// Shared memory: plane LO = (A+1) rows x rowStride words, then plane HI likewise (Packed16 only).
// Row 0 is the "no residue" letter, row y+1 is target letter y.  Word (row, t*Rpad + j) of plane LO
// holds the biased score of padded query row rowBase + t*R + j against that letter in its low
// half-word (sign bits cleared); plane HI holds it shifted left by 16.
// CHAIN: the variant for chained passes (SearchParams::chain), compiled for a few strip heights and for one warp per
// scheduler partition only; the other instantiations carry none of its code (the pointers and marks it keeps live
// across the sweep cost the capped 384-thread kernels a fifth of their speed when they were a run-time branch).
constexpr bool chain_strip_height(int R) { return R == 6 || R == 9 || R == 12 || R == 17 || R == 24 || R == 33; }
template <int R, int FLAVOR, class TR, int MAXT = launch_bound_for(FLAVOR, R), bool CHAIN = false>
__global__ void __launch_bounds__(MAXT, 1) search_kernel(const SearchParams p) {
    typedef typename TR::reg reg;
    constexpr int LANES = TR::LANES;
    constexpr bool kSW = FLAVOR != kFlavorGlobal;
    extern __shared__ __align__(16) uint32_t smem[];

    const int G = p.G, Go = p.gapOpen, Ge = p.gapExt, A = p.A, mode = p.mode;
    const int planeWords = (A + 1) * p.rowStride;
    // which pass over the query this block sweeps: the launch's (one launch per pass), or -- chained passes -- its own
    int pass = p.pass, rowBase = p.rowBase, chainQuad = 0;
    if (CHAIN) {
        if (threadIdx.x == 0) smem[0] = (uint32_t)atomicAdd(p.chainTicket, 1);  // (the profile is built over it below)
        __syncthreads();
        const int ticket = (int)smem[0];
        __syncthreads();
        pass = ticket % p.numPasses;
        chainQuad = ticket / p.numPasses;
        rowBase = pass * G * R;
    }

    // ---- build the query profile for this pass.  One thread per profile COLUMN (a padded query row of some thread's
    // strip): it reads its query letter once -- the only load with global-memory latency -- and then walks down the
    // A + 1 target letters of that column, reading one row of the score matrix (a few cache lines).  (The earlier form,
    // one thread per profile WORD, paid the query load and its dependent matrix load for every word: ~40 us per launch
    // at 32 x 33 rows, which is 6 % of a BASELINE configs[1] search and 1 - 2 % of every pass on a database shard.)
    // With a PSSM the column reads its own row of it.  (Written so that the sweep compiles to the same SASS as without
    // PSSM support: a select of the row base here changed the register allocation of the R = 32 step.)
    const bool byRow = p.pssm != nullptr;
    for (int pos = threadIdx.x; pos < p.rowStride; pos += blockDim.x) {
        const int t = pos / p.Rpad, j = pos - t * p.Rpad;
        int q = -1, q2 = -1;  // rows of `matrix` (query letters, or query rows) of the low / high half-word rows; -1 = padding
        const bool used = t < G && j < R;
        if (used) {
            const int r = rowBase + t * R + j - p.padTop;
            if (r >= 0 && r < p.Q) q = byRow ? r : p.query[r];
            q2 = q;
            if (LANES == 2 && p.folded) {  // high half-words: the rows 32 R further down
                const int r2 = r + 32 * R;
                q2 = (r2 >= 0 && r2 < p.Q) ? (byRow ? r2 : (int)p.query[r2]) : -1;
            }
        }
        // padding rows score 0 against everything (keeps H = 0 above the query); letter 0 is "no residue"
        const int* mrow = p.matrix + (q >= 0 ? q : 0) * A;
        const int* mrow2 = p.matrix + (q2 >= 0 ? q2 : 0) * A;
        for (int row = 0; row <= A; row++) {
            int sc = Go, scHi = Go;
            if (used) {
                if (row == 0) sc = scHi = p.padLetterScore + Go;
                if (q >= 0 && row > 0) sc = mrow[row - 1] + Go;
                if (q2 >= 0 && row > 0) scHi = mrow2[row - 1] + Go;
                if (!(LANES == 2 && p.folded)) scHi = sc;
            }
            const int idx = row * p.rowStride + pos;
            if (LANES == 2) {
                smem[idx] = (uint32_t)sc & 0xffffu;
                smem[planeWords + idx] = (uint32_t)scHi << 16;
            } else {
                smem[idx] = (uint32_t)sc;
            }
        }
    }
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int t = lane & (G - 1);
    const int groupInWarp = lane / G;
    const int groupsPerWarp = 32 / G;
    const uint32_t smemBase = (uint32_t)__cvta_generic_to_shared(smem);
    uint32_t myLo = smemBase + 4u * (uint32_t)(t * p.Rpad);
    uint32_t myHi = myLo + 4u * (uint32_t)planeWords;
    uint32_t rowBytes = 4u * (uint32_t)p.rowStride;
    // opaque to the compiler: it otherwise re-derives them from the CTA id, t and the launch parameters in every step
    // (six instructions of the sweep loop, measured in the executed SASS of the R = 32 bulk kernel)
    // (NW / HW / OV only: the SW loops are laid out differently and were measured no shorter with it)
    // (and only the tall strips: at R = 18 the pinned form measured 4.6 % slower, 4920 against 5160 GCUPS at Q = 144)
    constexpr bool kTightStep = !kSW && !single_event_compare(R);
    if constexpr (kTightStep) asm volatile("" : "+r"(myLo), "+r"(myHi), "+r"(rowBytes));
    const reg negGe = TR::splat(-Ge), negGo = TR::splat(-Go), negGmin = TR::splat(-min(Ge, Go));
    const reg NEGV = TR::splat(TR::NEG);
    // (Keeping P[] live across steps and reloading each chunk for the next column right after its use was
    // measured slower on B200: 0.83 vs 0.75 ms on BASELINE configs[1], extra registers and no shorter step.)
    // rows 4v .. 4v+3 (fewer at the tail) of one profile column: LDS.128 / .64 / .32 per plane
    auto load_chunk = [&](reg* P, uint32_t plo, uint32_t phi, int v) {
        const int j0 = v * 4;
        if (j0 + 4 <= R) {
            const uint4 a = lds128(plo + 4 * j0);
            uint4 b = a;
            if (LANES == 2) b = lds128(phi + 4 * j0);
            P[j0] = TR::combine(a.x, b.x); P[j0 + 1] = TR::combine(a.y, b.y);
            P[j0 + 2] = TR::combine(a.z, b.z); P[j0 + 3] = TR::combine(a.w, b.w);
        } else {
            int j = j0;
            if (R - j >= 2) {
                const uint2 a = lds64(plo + 4 * j);
                uint2 b = a;
                if (LANES == 2) b = lds64(phi + 4 * j);
                P[j] = TR::combine(a.x, b.x); P[j + 1] = TR::combine(a.y, b.y);
                j += 2;
            }
            if (R - j >= 1) P[j] = TR::combine(lds32(plo + 4 * j), LANES == 2 ? lds32(phi + 4 * j) : 0u);
        }
    };
    const bool firstPass = pass == 0, lastPass = pass == p.numPasses - 1;
    const bool firstPassOfLaunch = firstPass;  // (the sweep shadows firstPass with its compile-time copy)
    const int myRow0 = rowBase + t * R - p.padTop;  // query row of this thread's register 0
    // NW keeps padding at the bottom, so its last query row sits at a run-time position.
    const int lastRowPadded = p.Q - 1 + p.padTop;
    const int tLast = (lastRowPadded - rowBase) / R, jLast = (lastRowPadded - rowBase) % R;
    // Thread 0 of a group has no thread above it: what enters its strip is row -1 of the matrix (first pass) or
    // the previous pass's boundary row.  notFirst = 0 / 1 blends that in with an IMAD (see blend_fma); the value
    // blended in is kept at 0 in every other thread.
    // Folded tasks: thread 0 takes the low half-word of thread 31 (delivered by the same rotating shuffle) into its
    // high half-word -- a multiplication by 65536 -- and the boundary value only into its low half-word.
    const bool folded = LANES == 2 && p.folded != 0;
    const uint32_t notFirst = t != 0 ? (uint32_t)p.one : (folded ? 65536u * (uint32_t)p.one : 0u);
    const uint32_t synMask = (t == 0 && folded) ? 0xffffu : 0xffffffffu;
    const reg synIdle = t == 0 ? (reg)((uint32_t)(kSW ? negGo : NEGV) & synMask) : TR::splat(0);  // boundary row beyond the target's end
    const int srcLane = (lane & ~(G - 1)) | ((t - 1) & (G - 1));  // the thread above; thread 0 reads the last thread
    const int foldRows = folded ? 32 * R : 0;

    // Work distribution: tasks are ordered longest first.  The first task of every warp is static and
    // strided so that the longest targets land on different SMs / scheduler partitions (warp w of
    // block b takes task w * gridDim.x + b); afterwards warps pull from a global counter (LPT order).
    const int totalWarps = gridDim.x * (blockDim.x >> 5);
    bool firstTask = true;
    for (;;) {
        int w = 0;
        if (firstTask) {
            w = (threadIdx.x >> 5) * gridDim.x + blockIdx.x;
            if (CHAIN) w = chainQuad * (blockDim.x >> 5) + (threadIdx.x >> 5);  // one task per warp: its pass of this quad
            firstTask = false;
        } else if (CHAIN) {
            break;
        } else {
            if (lane == 0) w = totalWarps + atomicAdd(p.counter, 1);
            w = __shfl_sync(0xffffffffu, w, 0);
        }
        if ((long long)w * groupsPerWarp >= p.numTasks) break;

        // ---- this group's task: a target pair (Packed16) or one target (Scalar32)
        const int taskIdx = w * groupsPerWarp + groupInWarp;
        int tgt[2] = {-1, -1}, T[2] = {0, 0};
        const uint16_t* ps = p.pairStream + 32;  // groups without a task read leading padding only
        const uint8_t* seq0 = p.residues;
        long long off0 = 0;
        if (taskIdx < p.numTasks) {
            const int task = p.taskList ? p.taskList[taskIdx] : p.taskBase + taskIdx;
            if (LANES == 2) {
                tgt[0] = folded ? task : 2 * task;
                tgt[1] = (!folded && 2 * task + 1 < p.numTargets) ? 2 * task + 1 : -1;
                ps = p.pairStream + p.pairOffsets[task];
            } else {
                tgt[0] = task;
            }
            T[0] = p.lengths[tgt[0]];
            if (tgt[1] >= 0) T[1] = p.lengths[tgt[1]];
            off0 = p.offsets[tgt[0]];
            seq0 = p.residues + off0;
        }
        const int Tmax = T[0] + ((folded && T[0] > 0) ? kFoldLag : 0);  // pairs are (longer, shorter); columns of the stream
        const int steps = __reduce_max_sync(0xffffffffu, Tmax > 0 ? Tmax + G - 1 : 0);

        // ---- per-thread DP state and tracking state; (re)initialised by init_state() to column -1
        reg HG[R], E[R];
        reg diag, outH, outF;  // outH/outF: bottom of this strip = (H - Go of its last row, F entering the row below)
        reg best;              // SW: running max of H (fast flavor: of the key H << 6 | 63 - row); global: H - Go of the last row
        int rowLo, rowHi, colLo, colHi;          // SW end / HW-OV last-row column
        uint32_t keyLo, keyHi;                   // kFlavorSWEndFast: `best` as it was when the half-word last improved
        int nwScore[2], lcScore[2], lcRow[2];    // NW final cell; OV last column
        // Range tracking (NW / HW / OV, 16 bits).  DPX adds wrap, and unlike SW these modes have no running maximum
        // that would notice: instead H - Go of the strip's LAST row is sampled in every column (two instructions per
        // column, not per cell).  Neighbouring cells differ by at most D = gapOpen + gapExt + max |score| in any
        // direction, so while every sample stays (R + 3) D inside the representable range no cell of the strip -- nor
        // of the next column -- can have left it; the first sample that does not flags the target for the 32-bit
        // class, as the reference's short pass hands over to its int pass (src/opal.cpp:802-813, 1000-1017).
        constexpr bool kRange = FLAVOR == kFlavorGlobal && LANES == 2;
        reg hiTrack, loTrack;
        const reg* bH = reinterpret_cast<const reg*>(p.bndInH) + off0;  // boundary rows of the previous pass
        const reg* bF = reinterpret_cast<const reg*>(p.bndInF) + off0;
        reg* oH = reinterpret_cast<reg*>(p.bndOutH) + off0;  // ... and of this pass
        reg* oF = reinterpret_cast<reg*>(p.bndOutF) + off0;
        if (CHAIN) {  // this pass's row and the previous pass's row of the chained launch
            const long long at = (taskIdx < p.numTasks ? p.chainOffsets[taskIdx] : 0);
            oH = reinterpret_cast<reg*>(p.bndOutH) + (long long)pass * p.chainStride + at;
            oF = reinterpret_cast<reg*>(p.bndOutF) + (long long)pass * p.chainStride + at;
            bH = oH - p.chainStride;
            bF = oF - p.chainStride;
        }
        // opaque to the compiler: otherwise it re-derives base + (off0 + c) * 4 in every step with seven integer-pipe
        // instructions, stores predicated off or not; as plain pointers the address is one IMAD.WIDE each
        asm volatile("" : "+l"(oH), "+l"(oF));
        // Chained passes, later pass: the previous pass's row arrives 32 columns at a time, lane i holding column
        // 32 k + i of the chunk in use (cur) and of the next one (nxt); thread 0 -- at column s in step s -- takes
        // its column by shuffle.  A chunk is complete when none of its entries is kChainEmpty any more.
        constexpr uint32_t kEmpty = LANES == 2 ? kChainEmpty : kChainEmpty32;
        const reg idleV = kSW ? negGo : NEGV;   // boundary row beyond the target's end
        reg curH = idleV, curF = idleV, nxtH = idleV, nxtF = idleV;
        bool chainBroken = false;  // a wait was given up: the task's results are not to be trusted (flagged for the 32-bit class)
        auto load_boundary_chunk = [&](int k, reg& h, reg& f) {
            h = idleV; f = idleV;
            if (32 * k >= Tmax) return;
            const int col = 32 * k + lane;
            bool ok;
            unsigned polls = 0;
            do {
                if (col < Tmax) { h = (reg)ld_cg_u32(bH + col); f = (reg)ld_cg_u32(bF + col); }
                ok = col >= Tmax || ((uint32_t)h != kEmpty && (uint32_t)f != kEmpty);
                if (++polls == (1u << 24)) {  // seconds: the producer is gone (must not happen); leave instead of hanging the device
                    if (lane == 0) printf("opal-b200: chained pass %d of task %d gave up waiting for columns %d.. of %d\n", pass, taskIdx, 32 * k, Tmax);
                    chainBroken = true;
                    break;
                }
            } while (!__all_sync(0xffffffffu, ok));
            if (col >= Tmax) { h = idleV; f = idleV; }
        };
        const uint32_t firstThreadOnly = t == 0 ? 0xffffffffu : 0u;
        reg nextBH, nextBF;
        auto init_state = [&](bool keyTracking) {
#pragma unroll
            for (int j = 0; j < R; j++) {
                HG[j] = TR::splat(border_h(mode, myRow0 + j, Go, Ge) - Go);
                E[j] = NEGV;
            }
            diag = TR::splat(border_h(mode, myRow0 - 1, Go, Ge) - Go);
            outH = kSW ? negGo : NEGV; outF = outH;
            best = TR::splat(keyTracking ? (1 << kRowBits) - 1 : (kSW ? 0 : TR::NEG));
            rowLo = rowHi = colLo = colHi = -1;
            keyLo = keyHi = 0;
            nwScore[0] = nwScore[1] = lcScore[0] = lcScore[1] = kScoreNone;
            lcRow[0] = lcRow[1] = -1;
            hiTrack = TR::splat(TR::NEG); loTrack = TR::splat(32767);
            nextBH = synIdle; nextBF = synIdle;
            if (!CHAIN && !firstPass && t == 0 && Tmax > 0) { nextBH = bH[0]; nextBF = bF[0]; }
        };
        unsigned storeLimit = (!lastPass && t == G - 1) ? (unsigned)Tmax : 0u;  // columns whose bottom row is parked
        // Rare events of a NW / HW / OV sweep, each at the END of one column of this thread (-2 = never):
        //   OV: last-column scan of the pair's shorter member (see below; folded: of the low half-words, whose last
        //       column is overwritten by idle columns before the sweep ends);
        //   NW: the column(s) whose cell in the last query row is the result; only the thread that holds that row looks;
        //   folded: column 31, after which the high half-words -- idle so far -- are set to their column -1.
        // The sweep tests ONE column per step, the nearest event still ahead (kept opaque so that the test stays one
        // integer-pipe compare instead of being re-derived from pass, thread, mode and lengths).
        constexpr bool kOneCompare = single_event_compare(R);
        const bool foldedGlobal = kOneCompare && folded && FLAVOR == kFlavorGlobal;
        int ovScanCol = (FLAVOR == kFlavorGlobal && mode == kModeOV && LANES == 2 && T[1] != T[0]) ? T[1] - 1 : -2;
        const int ovScanLane = foldedGlobal ? 0 : 1;
        int nwCol[2] = {-2, -2};
        int jLastTask = jLast;
        if (FLAVOR == kFlavorGlobal && mode == kModeNW && lastPass) {
            if (!foldedGlobal) {
                if (t == tLast) { nwCol[0] = T[0] - 1; nwCol[1] = T[1] - 1; }
            } else {  // the last query row sits in the low or in the high half-words
                const int pos = lastRowPadded - rowBase, half = pos >= foldRows ? 1 : 0, posIn = pos - half * foldRows;
                jLastTask = posIn % R;
                if (t == posIn / R) nwCol[half] = T[0] - 1 + half * kFoldLag;
            }
        }
        if (foldedGlobal && mode == kModeOV) ovScanCol = T[0] - 1;
        // Tall strips (separate compares): the only event INSIDE a sweep is the last column of the shorter member of a pair
        // of unequal lengths -- OV scans it, NW reads its result cell there.  The longer member's last column (and the
        // shorter one's when the lengths are equal, the usual case in a sorted database) is still in HG[] when the sweep
        // ends and is read there.  One column, one compare per step.
        int evCol = -2;
        if (!kOneCompare && FLAVOR == kFlavorGlobal && LANES == 2 && T[1] != T[0]) {
            if (mode == kModeOV) evCol = T[1] - 1;
            else if (mode == kModeNW && lastPass && t == tLast) evCol = T[1] - 1;
        }
        const int foldInitCol = foldedGlobal ? kFoldLag - 1 : -2;
        auto next_event = [&](int after) {
            int e = 0x7fffffff;
            if (ovScanCol > after) e = min(e, ovScanCol);
            if (nwCol[0] > after) e = min(e, nwCol[0]);
            if (nwCol[1] > after) e = min(e, nwCol[1]);
            if (foldInitCol > after) e = min(e, foldInitCol);
            return e == 0x7fffffff ? -2 : e;
        };
        int nextEvent = next_event(-1);
        if (kOneCompare) asm volatile("" : "+r"(storeLimit), "+r"(nextEvent));
        else asm volatile("" : "+r"(storeLimit), "+r"(evCol));

        // OV: best cell of the last target column among this thread's rows (first row on ties), half-word l
        auto scan_last_column = [&](int l) {
#pragma unroll
            for (int j = 0; j < R; j++) {
                const int r = myRow0 + j + (l == 1 ? foldRows : 0);
                const int v = TR::lane(HG[j], l) + Go;
                if (r >= 0 && r < p.Q && v > lcScore[l]) { lcScore[l] = v; lcRow[l] = r; }
            }
        };
        // residues of column cc as y0 + 1 and y1 + 1, 0 = none.  The paired stream is padded, so
        // only the upper clamp is needed (a group may idle while longer groups of its warp finish).
        struct Letters { uint32_t lo, hi; };
        auto fetch = [&](int cc) -> Letters {
            Letters w;
            if (LANES == 2) {
                const uint8_t* q = reinterpret_cast<const uint8_t*>(ps + min(cc, Tmax));
                w.lo = ldg_u8(q); w.hi = ldg_u8(q + 1);
            } else {
                w.lo = (cc >= 0 && cc < Tmax) ? (uint32_t)seq0[cc] + 1u : 0u; w.hi = 0;
            }
            return w;
        };
        // One sweep of the task with tracking flavor TRACK (kFlavorSWEndFast tasks whose score leaves the exact
        // range of the key are swept a second time with kFlavorSWEnd, see below).
        auto sweep_pass = [&](auto trackTag, auto firstTag) {
            constexpr int TRACK = decltype(trackTag)::value;
            // first pass or a later one, as a compile-time property of the loop: what enters thread 0's strip is produced
            // in different ways, and selecting between them inside the step costs a compare, a branch and four moves
            // (NW / HW / OV at the tall strips; the other kernels keep the run-time test: firstTag = 2)
            constexpr int kFirst = decltype(firstTag)::value;
            const bool firstPass = kFirst == 2 ? firstPassOfLaunch : kFirst == 1;
            int c = -t;
            Letters wnext = fetch(c);
            reg P[R];
            if (CHAIN && !firstPass) { load_boundary_chunk(0, curH, curF); load_boundary_chunk(1, nxtH, nxtF); }
            // row -1 of the matrix as seen by thread 0 (reference src/opal.cpp:716-732; all zeros for SW); NW's
            // -Go - c * Ge walks down by Ge per column
            reg synRow = TR::splat(0), synStep = TR::splat(0);
            if (t == 0) {
                synRow = (reg)((uint32_t)negGo & synMask);  // H = 0 in row -1 (SW, HW, OV)
                if (!kSW && mode == kModeNW) { synRow = (reg)((uint32_t)TR::splat(-Go - Go) & synMask); synStep = (reg)((uint32_t)negGe & synMask); }
            }
            if constexpr (kTightStep) asm volatile("" : "+r"(synStep));  // (a register, not eight instructions per step re-deriving it from t, mode and folded)

#ifdef OPAL_UNROLL2
#pragma unroll 2
#endif
            for (int s = 0; s < steps; s++, c++) {
                // ---- (H - Go, F) handed down by the row above, for column c
                reg upH = __shfl_sync(0xffffffffu, outH, srcLane);
                reg upF = __shfl_sync(0xffffffffu, outF, srcLane);
                {   // thread 0 has no thread above: row -1 of the matrix (first pass) or the previous pass's
                    // boundary row.  Written as selects / predicated loads: a per-step divergent branch here
                    // costs more than the whole exchange.
                    reg synH, synF;
                    if (firstPass) {
                        synH = synRow;
                        synF = synH;  // F entering row 0 = max(-inf - Ge, H[-1][c] - Go)
                        if (!kSW) synRow = TR::add(synRow, synStep);
                    } else if (CHAIN) {
                        // thread 0 is at column s: lane s mod 32 of the chunk in use holds it (zero for the other threads,
                        // whose value comes from the thread above)
                        synH = (reg)((uint32_t)__shfl_sync(0xffffffffu, curH, s & 31) & firstThreadOnly);
                        synF = (reg)((uint32_t)__shfl_sync(0xffffffffu, curF, s & 31) & firstThreadOnly);
                        if ((s & 31) == 31) {  // on to the next chunk; fetch the one after it (two chunks ahead of thread 0)
                            curH = nxtH; curF = nxtF;
                            load_boundary_chunk((s >> 5) + 2, nxtH, nxtF);
                        }
                    } else {
                        synH = nextBH; synF = nextBF;
                        nextBH = synIdle; nextBF = synIdle;
                        if (t == 0 && c + 1 < Tmax) { nextBH = bH[c + 1]; nextBF = bF[c + 1]; }
                    }
                    upH = TR::blend(upH, notFirst, synH);
                    upF = TR::blend(upF, notFirst, synF);
                }
                const Letters wcur = wnext;
                wnext = fetch(c + 1);
                const bool active = (unsigned)c < (unsigned)Tmax;
                // SW runs its idle columns too: with the "no residue" letter they leave a state that is
                // equivalent to the initial one (H = 0, negative E/F never matter) and cannot raise best.
                if (!kSW && !active) continue;

                // ---- one target column for this thread's R query rows.
                // Per cell (Gotoh, reference src/opal.cpp:280-328 / :748-772), with X = max(diag + P, E [, 0]):
                //   H = max(X, F);  F' = max(F - Ge, H - Go) = max(F - min(Ge, Go), X - Go).
                // So the only value carried from row to row is F (one VIADDMNMX per row on the critical
                // path); E, X and X - Go of every row depend on the previous column only.  Row j+1's X is
                // issued before row j's H is written back, which lets H - Go be updated in place.
                // Profile values of this column.  Short strips (R <= 20) keep P[] live across steps and reload each
                // 4-row chunk for the NEXT column as soon as it has been consumed, which takes the shared-memory
                // latency off the critical path of a warp that runs alone on its scheduler partition.
                const uint32_t plo = myLo + wcur.lo * rowBytes, phi = myHi + wcur.hi * rowBytes;
                load_chunk(P, plo, phi, 0);
                auto consumed = [&](int row) {  // P[row] has just been used
                    if (row % 4 == 3 && row + 1 < R) load_chunk(P, plo, phi, row / 4 + 1);
                };
                reg f = upF;
                const reg dIn = diag;
                diag = upH;
                const reg bestBefore = best;
                reg e0 = TR::addmax(E[0], negGe, HG[0]);
                E[0] = e0;
                reg X = kSW ? TR::addmax_relu(dIn, P[0], e0) : TR::addmax(dIn, P[0], e0);
                consumed(0);
    #pragma unroll
                for (int j = 0; j < R; j++) {
                    reg Xn = 0;
                    if (j + 1 < R) {
                        const reg e1 = TR::addmax(E[j + 1], negGe, HG[j + 1]);
                        E[j + 1] = e1;
                        Xn = kSW ? TR::addmax_relu(HG[j], P[j + 1], e1) : TR::addmax(HG[j], P[j + 1], e1);
                    }
                    if (j + 1 < R) consumed(j + 1);
                    if (TRACK == kFlavorSWScore) {
                        best = TR::vmax(best, X);  // ptxas pairs these into VIMNMX3.S16x2 (0.5 instruction per cell)
                    } else if (TRACK == kFlavorSWEnd) {
                        best = TR::track(best, X, rowLo, rowHi, j, p.one);
                    } else if (TRACK == kFlavorSWEndFast) {
                        // key = H << 6 | (63 - row) in both half-words: one IMAD (FMA pipe) and one VIMNMX.  Exact while
                        // H < 512; larger scores are detected at the end (fastEndLimit) and re-run by kFlavorSWEnd.
                        const uint32_t rowBits = (uint32_t)((1 << kRowBits) - 1 - j) * 0x00010001u;
                        best = TR::vmax(best, (reg)((uint32_t)X * (uint32_t)p.keyScale + rowBits));
                    }
                    const reg XG = TR::add(X, negGo);
                    HG[j] = TR::addmax(f, negGo, XG);   // H - Go = max(X, F) - Go
                    f = TR::addmax(f, negGmin, XG);     // F of the next row
                    X = Xn;
                }
                const reg u = HG[R - 1];
                outH = u; outF = f;
                if constexpr (kRange) { hiTrack = TR::vmax(hiTrack, u); loTrack = TR::vmin(loTrack, u); }

                if (TRACK == kFlavorSWEnd) {
                    const reg ch = best ^ bestBefore;
                    if (LANES == 2) { if (ch & 0xffffu) colLo = c; if (ch >> 16) colHi = c; }
                    else if (ch) colLo = c;
                }
                if (TRACK == kFlavorSWEndFast) {
                    // A changed half-word means a strictly larger (score, first row) in THIS column: latch row and
                    // column, then saturate the row bits so that equal scores of later columns cannot win.
                    if constexpr (LANES == 2)
                        best = latch_key_s16x2(best, bestBefore, c, colLo, colHi, keyLo, keyHi);
                }
                if (FLAVOR == kFlavorGlobal) {
                    auto track_last_row = [&]() {
                        // last query row (HW, OV): register R-1 of thread G-1 in the last pass.  Every thread runs the
                        // three instructions (only thread G-1's result is read), which is cheaper than branching
                        // around them.  The shorter member of a pair needs no mask in the columns past its end: a
                        // cell there is reached through a horizontal gap from its last real column, so it is
                        // strictly below the value that column already contributed.
                        // (Earlier passes run it as well; their result is never read.)
                        bool ph, pl;
                        best = TR::bmax(best, u, &ph, &pl);
                        if (!pl) colLo = c;
                        if (LANES == 2 && !ph) colHi = c;
                    };
                    if constexpr (!kOneCompare) {
                        track_last_row();  // (NW never reads it; testing the mode here would cost more than the three instructions)
                        if (c == evCol) {  // rare: last column of the shorter member of an unequal pair
                            if (mode == kModeNW) {
                                reg v = HG[0];
    #pragma unroll
                                for (int j = 1; j < R; j++) if (j == jLast) v = HG[j];
                                nwScore[1] = TR::lane(v, 1) + Go;
                            } else {
                                scan_last_column(1);
                            }
                        }
                    } else {
                    if (mode != kModeNW) track_last_row();
                    if (c == nextEvent) {  // rare: see the list of events above
                        if (mode == kModeNW) {
    #pragma unroll
                            for (int l = 0; l < LANES; l++)
                                if (c == nwCol[l]) {
                                    reg v = HG[0];
    #pragma unroll
                                    for (int j = 1; j < R; j++) if (j == jLastTask) v = HG[j];
                                    nwScore[l] = TR::lane(v, l) + Go;
                                }
                        }
                        // last target column (OV): every real row of this thread.  Only the shorter member of a
                        // pair of unequal lengths is scanned here, where each thread meets that column at a step
                        // of its own (one active thread per scan); the longer member -- and the shorter one when
                        // the lengths are equal, the usual case in a large sorted database -- is still sitting in
                        // HG[] when the sweep ends and is scanned there by all threads at once.
                        if (c == ovScanCol) scan_last_column(ovScanLane);
                        if constexpr (LANES == 2) {
                            if (c == foldInitCol) {
                                // The high half-words have swept 32 idle columns (whatever they tracked is dropped);
                                // their real column 0 is next: column -1 of rows 32 R ... (reference src/opal.cpp:671-679).
                                const uint32_t lo = 0xffffu, hi = 0xffff0000u;
    #pragma unroll
                                for (int j = 0; j < R; j++) {
                                    HG[j] = (HG[j] & lo) | ((uint32_t)TR::splat(border_h(mode, myRow0 + foldRows + j, Go, Ge) - Go) & hi);
                                    E[j] = (E[j] & lo) | ((uint32_t)NEGV & hi);
                                }
                                diag = (diag & lo) | ((uint32_t)TR::splat(border_h(mode, myRow0 + foldRows - 1, Go, Ge) - Go) & hi);
                                best = (best & lo) | ((uint32_t)TR::splat(TR::NEG) & hi);
                                hiTrack = (hiTrack & lo) | ((uint32_t)TR::splat(TR::NEG) & hi);  // samples of the idle columns are dropped
                                loTrack = (loTrack & lo) | ((uint32_t)TR::splat(32767) & hi);
                                colHi = -1;
                            }
                        }
                        nextEvent = next_event(c);
                    }
                    }
                }
                if ((unsigned)c < storeLimit) {  // last thread of a group, every pass but the last: park the bottom row
                    reg sH = outH, sF = outF;
                    if (CHAIN) {  // never the "not written yet" pattern (see kChainEmpty)
                        if ((uint32_t)sH == kEmpty) sH = (reg)(kEmpty + 1u);
                        if ((uint32_t)sF == kEmpty) sF = (reg)(kEmpty + 1u);
                    }
                    if (CHAIN) {  // read by another SM while this sweep goes on: stores at device scope
                        st_gpu_u32(oH + c, (uint32_t)sH);
                        st_gpu_u32(oF + c, (uint32_t)sF);
                    } else {
                        asm volatile("st.global.b32 [%0], %1;" :: "l"(oH + c), "r"(sH) : "memory");
                        asm volatile("st.global.b32 [%0], %1;" :: "l"(oF + c), "r"(sF) : "memory");
                    }
                }
            }

        };
        auto sweep = [&](auto trackTag) {
            if constexpr (!kTightStep) sweep_pass(trackTag, std::integral_constant<int, 2>());
            else if (firstPass) sweep_pass(trackTag, std::integral_constant<int, 1>());
            else sweep_pass(trackTag, std::integral_constant<int, 0>());
        };

        // ---- reduce the group's candidates (key: score desc, target index asc, query index asc)
        int fsc[2], fcc[2], frr[2];
        bool outOfRange[2] = {false, false};
        auto reduce = [&](bool keyTracking) {
            if constexpr (kRange) {  // did any thread's samples leave the safe range?  (bit l = half-word l)
                unsigned bad = 0;
#pragma unroll
                for (int l = 0; l < LANES; l++)
                    if (TR::lane(hiTrack, l) + Go > p.rangeHi || TR::lane(loTrack, l) + Go < p.rangeLo) bad |= 1u << l;
                for (int o = 1; o < G; o <<= 1) bad |= __shfl_xor_sync(0xffffffffu, bad, o);
                if (folded) bad = bad ? 3u : 0u;  // one target in both half-words
                outOfRange[0] = bad & 1u; outOfRange[1] = (bad >> 1) & 1u;
            }
#pragma unroll
            for (int l = 0; l < LANES; l++) {
                int sc = kScoreNone, cc = 0x7fffffff, rr = 0x7fffffff;  // this thread's candidate
                if (kSW) {
                    sc = TR::lane(best, l);
                    if (keyTracking) sc >>= kRowBits;
                    if ((FLAVOR == kFlavorSWEnd || FLAVOR == kFlavorSWEndFast) && sc > 0) {
                        cc = l ? colHi : colLo;
                        const int mask = (1 << kRowBits) - 1;
                        rr = myRow0 + (keyTracking ? mask - (int)(((l ? keyHi >> 16 : keyLo)) & mask) : (l ? rowHi : rowLo));
                        if (l == 1) { cc -= folded ? kFoldLag : 0; rr += foldRows; }  // folded: same target, 32 columns behind, 32 R rows down
                    }
                } else if (mode == kModeNW) {
                    sc = nwScore[l]; cc = (foldedGlobal ? T[0] : T[l]) - 1; rr = p.Q - 1;
                } else {
                    // last query row: the last register of the last thread (folded: of its high half-word, whose
                    // columns are 32 behind)
                    const int Tl = foldedGlobal ? T[0] : T[l];
                    if (lastPass && t == G - 1 && Tl > 0 && (!foldedGlobal || l == 1)) {
                        sc = TR::lane(best, l) + Go; cc = (l ? colHi : colLo) - (foldedGlobal ? kFoldLag : 0); rr = p.Q - 1;
                    }
                    if (mode == kModeOV && lcScore[l] != kScoreNone && better(lcScore[l], Tl - 1, lcRow[l], sc, cc, rr)) {
                        sc = lcScore[l]; cc = Tl - 1; rr = lcRow[l];
                    }
                }
                for (int o = 1; o < G; o <<= 1) {
                    const int s2 = __shfl_xor_sync(0xffffffffu, sc, o);
                    const int c2 = __shfl_xor_sync(0xffffffffu, cc, o);
                    const int r2 = __shfl_xor_sync(0xffffffffu, rr, o);
                    if (better(s2, c2, r2, sc, cc, rr)) { sc = s2; cc = c2; rr = r2; }
                }
                fsc[l] = sc; fcc[l] = cc; frr[l] = rr;
            }
            if (LANES == 2 && folded && better(fsc[1], fcc[1], frr[1], fsc[0], fcc[0], frr[0])) { fsc[0] = fsc[1]; fcc[0] = fcc[1]; frr[0] = frr[1]; }
        };

        if (FLAVOR == kFlavorSWEndFast) {
            // Key tracking is exact while scores stay below fastEndLimit.  A half-word that left that range may
            // also have spilled into its neighbour, so if any pair of this warp is affected the warp sweeps its
            // tasks once more with the exact per-cell predicate tracking (same registers, second code path).
            init_state(true);
            sweep(std::integral_constant<int, kFlavorSWEndFast>());
            reduce(true);
            bool inexact = false;
#pragma unroll
            for (int l = 0; l < LANES; l++) inexact |= fsc[l] >= p.fastEndLimit;
            if (__any_sync(0xffffffffu, inexact)) {
                if (CHAIN) storeLimit = 0;  // the boundary row is already out (the re-sweep computes the same values)
                init_state(false);
                sweep(std::integral_constant<int, kFlavorSWEnd>());
                reduce(false);
            }
        } else {
            init_state(false);
            sweep(std::integral_constant<int, FLAVOR>());
            if (FLAVOR == kFlavorGlobal && !kOneCompare && mode == kModeNW && lastPass && t == tLast && T[0] > 0) {
                // tall strips: the result cell of the longer member (of both when the lengths are equal) is read here
                reg v = HG[0];
#pragma unroll
                for (int j = 1; j < R; j++) if (j == jLast) v = HG[j];
                nwScore[0] = TR::lane(v, 0) + Go;
                if (LANES == 2 && T[1] == T[0]) nwScore[1] = TR::lane(v, 1) + Go;
            }
            if (FLAVOR == kFlavorGlobal && mode == kModeOV) {
                // threads stop updating their rows after the last column of the longer member: it is still in HG[]
                // (folded: only the high half-words; the low ones were scanned inside the sweep)
                if (T[0] > 0 && !foldedGlobal) scan_last_column(0);
                if (LANES == 2 && (foldedGlobal ? T[0] > 0 : (T[1] == T[0] && T[1] > 0))) scan_last_column(1);
            }
            reduce(false);
        }
        const bool pairInexact = false;
        if (CHAIN && !firstPass && t == 0 && taskIdx < p.numTasks) {  // the previous pass's results must be in memory
            const int* doneIn = p.chainDone + taskIdx * p.numPasses + pass - 1;
            unsigned polls = 0;
            while (ld_acquire(doneIn) == 0)
                if (++polls == (1u << 24)) { chainBroken = true; break; }  // (as above: never hang the device)
        }
#pragma unroll
        for (int l = 0; l < LANES; l++) {
            if (t == 0 && tgt[l] >= 0) {
                const int i = tgt[l];
                int sc = fsc[l], cc = fcc[l], rr = frr[l];
                bool overflow = (kSW && sc > p.overflowLimit) || pairInexact || outOfRange[l] || (CHAIN && chainBroken);
                if (!firstPass) {
                    // (volatile: with chained passes the previous pass wrote these from another SM a moment ago)
                    const int ps0 = *(volatile int*)(p.outScore + i);
                    if (ps0 == kScoreOverflow) overflow = true;
                    else if (ps0 != kScoreNone) {
                        const int pc = *(volatile int*)(p.outEndT + i), pr = *(volatile int*)(p.outEndQ + i);
                        if (sc == kScoreNone || better(ps0, pc, pr, sc, cc, rr)) { sc = ps0; cc = pc; rr = pr; }
                    }
                }
                if (overflow) sc = kScoreOverflow;
                if (sc != kScoreNone || firstPass) {
                    p.outScore[i] = sc;
                    const bool haveEnd = p.wantEnd && sc != kScoreOverflow && sc != kScoreNone && !(kSW && sc == 0);
                    p.outEndT[i] = haveEnd ? cc : (kSW || sc == kScoreNone ? 0x7fffffff : cc);
                    p.outEndQ[i] = haveEnd ? rr : (kSW || sc == kScoreNone ? 0x7fffffff : rr);
                }
            }
        }
        if (CHAIN && t == 0 && taskIdx < p.numTasks) st_release(p.chainDone + taskIdx * p.numPasses + pass, 1);
    }
}

// ---------------------------------------------------------------- DPX issue-rate probe
// Register-only loop of the cell recurrence used by bench.py to measure the integer-pipe roofline on the
// device it runs on (SURVEY.md section 8d).
// MIX 0: the SW recurrence, 6 packed instructions per 2 cells; MIX 1: NW / HW / OV, 5 (no running maximum per cell).
template <int ILP, int MIX>
__global__ void __launch_bounds__(512, 1) dpx_peak_kernel(uint32_t* out, int iters, uint32_t seed) {
    uint32_t h[ILP], e[ILP], f[ILP], b[ILP];
#pragma unroll
    for (int i = 0; i < ILP; i++) { h[i] = seed + i * 0x00010001u + threadIdx.x; e[i] = h[i] ^ 0x00050003u; f[i] = e[i] + 0x00010002u; b[i] = 0; }
    const uint32_t ng = 0xffffffffu, no = 0xfff5fff5u, pp = 0x00030002u;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < ILP; i++) {
            e[i] = __viaddmax_s16x2(e[i], ng, h[i]);
            f[i] = __viaddmax_s16x2(f[i], ng, h[i]);
            uint32_t x = MIX == 0 ? __viaddmax_s16x2_relu(h[i], pp, e[i]) : __viaddmax_s16x2(h[i], pp, e[i]);
            x = __vmaxs2(x, f[i]);
            if (MIX == 0) b[i] = __vmaxs2(b[i], x);
            h[i] = __vadd2(x, no);
        }
    }
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < ILP; i++) acc ^= b[i] ^ h[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
}

}  // namespace opalb200
