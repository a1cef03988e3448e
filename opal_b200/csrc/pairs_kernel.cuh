// pairs_kernel.cuh -- the score / score+end kernel of the pairs path (sm_100a): many queries per launch, each against
// its own list of database entries.
//
// The recurrence, the arithmetic, the profile layout and the end-location key are those of search_kernel (see the notes
// at the top of search_kernel.cuh); what differs is where the work comes from:
//   * a TASK is one (query, target) pair at 32 bits, or two pairs of the SAME query in the two 16-bit half-words -- the
//     host groups the pairs by query and, within a query, sorts them longest target first, so a task's members have
//     similar lengths and both half-words score against one profile;
//   * a BLOCK serves a run of consecutive tasks of one query (PairBlock) and builds that query's profile in shared
//     memory itself, once per pass, so one launch holds the tasks of many queries;
//   * a query longer than one strip of G x R rows takes several passes, all inside the block: the block rebuilds the
//     profile for the next G x R rows and every group sweeps the same tasks again, the boundary row (H, F per target
//     column) parked in HBM between passes (ping-pong halves, as in search_kernel);
//   * 16 bits read the two targets of a task from a per-call paired stream in pack_pairs_kernel's format,
//     (res0 + 1) | (res1 + 1) << 8 with >= 32 zero entries either side; 32 bits read the plain residues.
// Warps take their tasks statically (round k of warp w: tasks (k * warps + w) * 32 / G ...), identically in every pass,
// so the thread that parks a task's boundary row and results is the thread that reads them back.
// 16-bit safety is established as in search_kernel: SW flags a target whose best exceeds overflowLimit, NW / HW / OV
// flag a target whose sampled last-row H leaves [rangeLo, rangeHi]; flagged pairs are re-run at 32 bits by the host.
#pragma once
#include "search_kernel.cuh"

namespace opalb200 {

constexpr int kPairsThreads = 384;  // three warps per scheduler partition, one block per SM (the profile fills shared memory)
constexpr int kPairsR[2] = {8, 16};  // strip heights the pairs kernel is compiled for
__host__ __device__ constexpr int pairs_rpad(int R) { return 4 * (((R + 3) / 4) % 2 == 0 ? (R + 3) / 4 + 1 : (R + 3) / 4); }

struct PairTask {
    int slot[2];    // result slots (pair indices) of the low / high half-word; -1 = none
    int tgt[2];     // sorted positions of the targets
    int T[2];       // their lengths, T[0] >= T[1]
    long long col;  // 16 bits: the task's first entry in the paired stream
    long long bnd;  // its first entry in each half of the boundary rows (queries of several passes)
};
struct PairQuery {
    int Q, G, passes, padTop;
    long long queryOff;  // its residues in the query blob
};
struct PairBlock {
    int query, firstTask, numTasks, pad;
};

struct PairsParams {
    const uint8_t* queries;  // every query's residues, back to back
    const int* matrix;       // A x A
    int A, gapOpen, gapExt, mode, wantEnd;
    const PairQuery* queryTab;
    const PairBlock* blockTab;
    const PairTask* tasks;
    const uint8_t* residues;  // the database's plain residues (32 bits)
    const long long* offsets;
    const uint16_t* stream;   // the per-call paired stream (16 bits)
    void* bndH;               // boundary rows: two halves of bndHalf entries each
    void* bndF;
    long long bndHalf;
    int* outScore;  // by result slot
    int* outEndQ;
    int* outEndT;
    int overflowLimit, padLetterScore, rangeHi, rangeLo, one;
};

template <int R, int FLAVOR, class TR>
__global__ void __launch_bounds__(kPairsThreads, 1) pairs_kernel(const PairsParams p) {
    typedef typename TR::reg reg;
    constexpr int LANES = TR::LANES;
    constexpr bool kSW = FLAVOR != kFlavorGlobal;
    constexpr int Rpad = pairs_rpad(R);
    extern __shared__ __align__(16) uint32_t smem[];

    const PairBlock blk = p.blockTab[blockIdx.x];
    const PairQuery qi = p.queryTab[blk.query];
    const uint8_t* query = p.queries + qi.queryOff;
    const int G = qi.G, Q = qi.Q, Go = p.gapOpen, Ge = p.gapExt, A = p.A, mode = p.mode;
    const int rowStride = (G * Rpad + 31) / 32 * 32;
    const int planeWords = (A + 1) * rowStride;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    const int t = lane & (G - 1), groupInWarp = lane / G, groupsPerWarp = 32 / G;
    const int srcLane = (lane & ~(G - 1)) | ((t - 1) & (G - 1));  // the thread above; thread 0 reads the last thread
    const uint32_t smemBase = (uint32_t)__cvta_generic_to_shared(smem);
    const uint32_t myLo = smemBase + 4u * (uint32_t)(t * Rpad), myHi = myLo + 4u * (uint32_t)planeWords;
    const uint32_t rowBytes = 4u * (uint32_t)rowStride;
    const reg negGe = TR::splat(-Ge), negGo = TR::splat(-Go), negGmin = TR::splat(-min(Ge, Go));
    const reg NEGV = TR::splat(TR::NEG);
    const uint32_t notFirst = t != 0 ? (uint32_t)p.one : 0u;
    const reg synIdle = t == 0 ? (kSW ? negGo : NEGV) : TR::splat(0);  // boundary row beyond the target's end
    const int lastRowPadded = Q - 1 + qi.padTop;
    const int rounds = (blk.numTasks + warps * groupsPerWarp - 1) / (warps * groupsPerWarp);

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

    for (int pass = 0; pass < qi.passes; pass++) {
        const int rowBase = pass * G * R;
        // ---- this pass's profile (search_kernel's build: one thread per profile column, padding rows score 0)
        if (pass > 0) __syncthreads();  // every warp is through with the previous profile (and its boundary rows are out)
        for (int pos = threadIdx.x; pos < rowStride; pos += blockDim.x) {
            const int tt = pos / Rpad, j = pos - tt * Rpad;
            int q = -1;
            const bool used = tt < G && j < R;
            if (used) {
                const int r = rowBase + tt * R + j - qi.padTop;
                if (r >= 0 && r < Q) q = query[r];
            }
            const int* mrow = p.matrix + (q >= 0 ? q : 0) * A;
            for (int row = 0; row <= A; row++) {
                int sc = Go;
                if (used) {
                    if (row == 0) sc = p.padLetterScore + Go;
                    if (q >= 0 && row > 0) sc = mrow[row - 1] + Go;
                }
                const int idx = row * rowStride + pos;
                if (LANES == 2) {
                    smem[idx] = (uint32_t)sc & 0xffffu;
                    smem[planeWords + idx] = (uint32_t)sc << 16;
                } else {
                    smem[idx] = (uint32_t)sc;
                }
            }
        }
        __syncthreads();

        const bool firstPass = pass == 0, lastPass = pass == qi.passes - 1;
        const int myRow0 = rowBase + t * R - qi.padTop;  // query row of this thread's register 0
        const int tLast = (lastRowPadded - rowBase) / R, jLast = (lastRowPadded - rowBase) % R;  // (read in the last pass)
        const long long inHalf = (long long)((pass + 1) & 1) * p.bndHalf, outHalf = (long long)(pass & 1) * p.bndHalf;

        for (int round = 0; round < rounds; round++) {
            const int w = round * warps + warp;
            if (w * groupsPerWarp >= blk.numTasks) break;  // (warp-uniform)
            const int taskIdx = w * groupsPerWarp + groupInWarp;
            int slot[2] = {-1, -1}, T[2] = {0, 0};
            const uint16_t* ps = p.stream + 32;  // groups without a task read leading padding only
            const uint8_t* seq0 = p.residues;
            long long bo = 0;
            if (taskIdx < blk.numTasks) {
                const PairTask& tk = p.tasks[blk.firstTask + taskIdx];
                slot[0] = tk.slot[0]; slot[1] = tk.slot[1]; T[0] = tk.T[0]; T[1] = tk.T[1];
                if (LANES == 2) ps = p.stream + tk.col;
                else seq0 = p.residues + p.offsets[tk.tgt[0]];
                bo = tk.bnd;
            }
            const int Tmax = T[0];
            const int steps = __reduce_max_sync(0xffffffffu, Tmax > 0 ? Tmax + G - 1 : 0);

            reg HG[R], E[R];
            reg diag, outH, outF, best;
            int rowLo = -1, rowHi = -1, colLo = -1, colHi = -1;
            int nwScore[2] = {kScoreNone, kScoreNone}, lcScore[2] = {kScoreNone, kScoreNone}, lcRow[2] = {-1, -1};
            constexpr bool kRange = FLAVOR == kFlavorGlobal && LANES == 2;  // range tracking (see search_kernel)
            reg hiTrack = TR::splat(TR::NEG), loTrack = TR::splat(32767);
            const reg* bH = reinterpret_cast<const reg*>(p.bndH) + inHalf + bo;
            const reg* bF = reinterpret_cast<const reg*>(p.bndF) + inHalf + bo;
            reg* oH = reinterpret_cast<reg*>(p.bndH) + outHalf + bo;
            reg* oF = reinterpret_cast<reg*>(p.bndF) + outHalf + bo;
#pragma unroll
            for (int j = 0; j < R; j++) {
                HG[j] = TR::splat(border_h(mode, myRow0 + j, Go, Ge) - Go);
                E[j] = NEGV;
            }
            diag = TR::splat(border_h(mode, myRow0 - 1, Go, Ge) - Go);
            outH = kSW ? negGo : NEGV; outF = outH;
            best = TR::splat(kSW ? 0 : TR::NEG);
            reg nextBH = synIdle, nextBF = synIdle;
            if (!firstPass && t == 0 && Tmax > 0) { nextBH = bH[0]; nextBF = bF[0]; }
            const unsigned storeLimit = (!lastPass && t == G - 1) ? (unsigned)Tmax : 0u;  // columns whose bottom row is parked
            // the one event inside a sweep: the last column of the shorter member of an unequal pair (OV scans it, NW reads
            // its result cell there); the longer member's last column is still in HG[] when the sweep ends
            int evCol = -2;
            if (FLAVOR == kFlavorGlobal && LANES == 2 && T[1] != T[0]) {
                if (mode == kModeOV) evCol = T[1] - 1;
                else if (mode == kModeNW && lastPass && t == tLast) evCol = T[1] - 1;
            }
            auto scan_last_column = [&](int l) {  // OV: best cell of the last target column among this thread's rows
#pragma unroll
                for (int j = 0; j < R; j++) {
                    const int r = myRow0 + j;
                    const int v = TR::lane(HG[j], l) + Go;
                    if (r >= 0 && r < Q && v > lcScore[l]) { lcScore[l] = v; lcRow[l] = r; }
                }
            };
            struct Letters { uint32_t lo, hi; };
            auto fetch = [&](int cc) -> Letters {
                Letters lt;
                if (LANES == 2) {
                    const uint8_t* q = reinterpret_cast<const uint8_t*>(ps + min(cc, Tmax));
                    lt.lo = ldg_u8(q); lt.hi = ldg_u8(q + 1);
                } else {
                    lt.lo = (cc >= 0 && cc < Tmax) ? (uint32_t)seq0[cc] + 1u : 0u; lt.hi = 0;
                }
                return lt;
            };

            int c = -t;
            Letters wnext = fetch(c);
            reg P[R];
            reg synRow = TR::splat(0), synStep = TR::splat(0);  // row -1 of the matrix as thread 0 sees it
            if (t == 0) {
                synRow = negGo;
                if (!kSW && mode == kModeNW) { synRow = TR::splat(-Go - Go); synStep = negGe; }
            }
            for (int s = 0; s < steps; s++, c++) {
                reg upH = __shfl_sync(0xffffffffu, outH, srcLane);
                reg upF = __shfl_sync(0xffffffffu, outF, srcLane);
                {
                    reg synH, synF;
                    if (firstPass) {
                        synH = synRow; synF = synH;
                        if (!kSW) synRow = TR::add(synRow, synStep);
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
                if (!kSW && !active) continue;  // (SW runs its idle columns: the "no residue" letter cannot raise best)

                const uint32_t plo = myLo + wcur.lo * rowBytes, phi = myHi + wcur.hi * rowBytes;
                load_chunk(P, plo, phi, 0);
                reg f = upF;
                const reg dIn = diag;
                diag = upH;
                const reg bestBefore = best;
                reg e0 = TR::addmax(E[0], negGe, HG[0]);
                E[0] = e0;
                reg X = kSW ? TR::addmax_relu(dIn, P[0], e0) : TR::addmax(dIn, P[0], e0);
#pragma unroll
                for (int j = 0; j < R; j++) {
                    reg Xn = 0;
                    if (j + 1 < R) {
                        const reg e1 = TR::addmax(E[j + 1], negGe, HG[j + 1]);
                        E[j + 1] = e1;
                        Xn = kSW ? TR::addmax_relu(HG[j], P[j + 1], e1) : TR::addmax(HG[j], P[j + 1], e1);
                        if ((j + 1) % 4 == 3 && j + 2 < R) load_chunk(P, plo, phi, (j + 1) / 4 + 1);
                    }
                    if (FLAVOR == kFlavorSWScore) best = TR::vmax(best, X);
                    else if (FLAVOR == kFlavorSWEnd) best = TR::track(best, X, rowLo, rowHi, j, p.one);
                    const reg XG = TR::add(X, negGo);
                    HG[j] = TR::addmax(f, negGo, XG);  // H - Go = max(X, F) - Go
                    f = TR::addmax(f, negGmin, XG);    // F of the next row
                    X = Xn;
                }
                const reg u = HG[R - 1];
                outH = u; outF = f;
                if constexpr (kRange) { hiTrack = TR::vmax(hiTrack, u); loTrack = TR::vmin(loTrack, u); }
                if (FLAVOR == kFlavorSWEnd) {
                    const reg ch = best ^ bestBefore;
                    if (LANES == 2) { if (ch & 0xffffu) colLo = c; if (ch >> 16) colHi = c; }
                    else if (ch) colLo = c;
                }
                if (FLAVOR == kFlavorGlobal) {
                    bool ph, pl;  // last query row (HW, OV): register R - 1 of thread G - 1 in the last pass
                    best = TR::bmax(best, u, &ph, &pl);
                    if (!pl) colLo = c;
                    if (LANES == 2 && !ph) colHi = c;
                    if (c == evCol) {
                        if (mode == kModeNW) {
                            reg v = HG[0];
#pragma unroll
                            for (int j = 1; j < R; j++) if (j == jLast) v = HG[j];
                            nwScore[1] = TR::lane(v, 1) + Go;
                        } else {
                            scan_last_column(1);
                        }
                    }
                }
                if ((unsigned)c < storeLimit) {  // last thread of a group, every pass but the last: park the bottom row
                    oH[c] = outH;
                    oF[c] = outF;
                }
            }
            if (FLAVOR == kFlavorGlobal && mode == kModeNW && lastPass && t == tLast && T[0] > 0) {
                reg v = HG[0];
#pragma unroll
                for (int j = 1; j < R; j++) if (j == jLast) v = HG[j];
                nwScore[0] = TR::lane(v, 0) + Go;
                if (LANES == 2 && T[1] == T[0]) nwScore[1] = TR::lane(v, 1) + Go;
            }
            if (FLAVOR == kFlavorGlobal && mode == kModeOV) {
                if (T[0] > 0) scan_last_column(0);
                if (LANES == 2 && T[1] == T[0] && T[1] > 0) scan_last_column(1);
            }

            // ---- reduce the group's candidates (key: score desc, target index asc, query index asc)
            bool outOfRange[2] = {false, false};
            if constexpr (kRange) {
                unsigned bad = 0;
#pragma unroll
                for (int l = 0; l < LANES; l++)
                    if (TR::lane(hiTrack, l) + Go > p.rangeHi || TR::lane(loTrack, l) + Go < p.rangeLo) bad |= 1u << l;
                for (int o = 1; o < G; o <<= 1) bad |= __shfl_xor_sync(0xffffffffu, bad, o);
                outOfRange[0] = bad & 1u; outOfRange[1] = (bad >> 1) & 1u;
            }
#pragma unroll
            for (int l = 0; l < LANES; l++) {
                int sc = kScoreNone, cc = 0x7fffffff, rr = 0x7fffffff;
                if (kSW) {
                    sc = TR::lane(best, l);
                    if (FLAVOR == kFlavorSWEnd && sc > 0) { cc = l ? colHi : colLo; rr = myRow0 + (l ? rowHi : rowLo); }
                } else if (mode == kModeNW) {
                    sc = nwScore[l]; cc = T[l] - 1; rr = Q - 1;
                } else {
                    if (lastPass && t == G - 1 && T[l] > 0) { sc = TR::lane(best, l) + Go; cc = l ? colHi : colLo; rr = Q - 1; }
                    if (mode == kModeOV && lcScore[l] != kScoreNone && better(lcScore[l], T[l] - 1, lcRow[l], sc, cc, rr)) {
                        sc = lcScore[l]; cc = T[l] - 1; rr = lcRow[l];
                    }
                }
                for (int o = 1; o < G; o <<= 1) {
                    const int s2 = __shfl_xor_sync(0xffffffffu, sc, o);
                    const int c2 = __shfl_xor_sync(0xffffffffu, cc, o);
                    const int r2 = __shfl_xor_sync(0xffffffffu, rr, o);
                    if (better(s2, c2, r2, sc, cc, rr)) { sc = s2; cc = c2; rr = r2; }
                }
                // ---- merge with the earlier passes' result (written by this same thread) and store
                const int i = slot[l];
                if (t == 0 && i >= 0) {
                    bool overflow = (kSW && sc > p.overflowLimit) || outOfRange[l];
                    if (!firstPass) {
                        const int ps0 = p.outScore[i];
                        if (ps0 == kScoreOverflow) overflow = true;
                        else if (ps0 != kScoreNone) {
                            const int pc = p.outEndT[i], pr = p.outEndQ[i];
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
        }
    }
}

}  // namespace opalb200
