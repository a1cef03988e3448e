// pairs.cu -- the kernels of the pairs path (pairs_kernel.cuh) and the per-call paired stream they read.
#include <algorithm>

#include "engine.h"
#include "pairs_kernel.cuh"

namespace opalb200 {

// The paired stream of one call in pack_pairs_kernel's format: task k occupies entries [col, col + T0 + 32), its T0
// columns (res0 + 1) | (res1 + 1) << 8 (0 past the shorter member's end) and then 32 zero entries; the stream starts
// with 32 zero entries.  One block per task, grid-stride over the tasks.
static __global__ void gather_pairs_kernel(const PairTask* tasks, int numTasks, const uint8_t* residues, const long long* offsets,
                                           uint16_t* stream) {
    if (blockIdx.x == 0 && threadIdx.x < 32) stream[threadIdx.x] = 0;
    for (int k = blockIdx.x; k < numTasks; k += gridDim.x) {
        const PairTask& tk = tasks[k];
        const uint8_t* r0 = residues + offsets[tk.tgt[0]];
        const uint8_t* r1 = tk.slot[1] >= 0 ? residues + offsets[tk.tgt[1]] : r0;
        const int T0 = tk.T[0], T1 = tk.slot[1] >= 0 ? tk.T[1] : 0;
        for (int c = threadIdx.x; c < T0 + 32; c += blockDim.x) {
            uint32_t word = 0;
            if (c < T0) {
                word = ((uint32_t)r0[c] + 1u) & 0xffu;
                if (c < T1) word |= (((uint32_t)r1[c] + 1u) & 0xffu) << 8;
            }
            stream[tk.col + c] = (uint16_t)word;
        }
    }
}

bool launch_gather_pairs(const PairTask* tasks, int numTasks, const uint8_t* residues, const long long* offsets, uint16_t* stream,
                         cudaStream_t st) {
    gather_pairs_kernel<<<(unsigned)std::max(1, std::min(numTasks, 1 << 16)), 256, 0, st>>>(tasks, numTasks, residues, offsets, stream);
    return cudaGetLastError() == cudaSuccess;
}

// [R index][type * 3 + flavor], type 0 = Packed16, 1 = Scalar32; flavor kFlavorSWScore / kFlavorSWEnd / kFlavorGlobal
#define OPAL_PAIRS_ROW(R)                                                                                                  \
    {(const void*)pairs_kernel<R, kFlavorSWScore, Packed16>, (const void*)pairs_kernel<R, kFlavorSWEnd, Packed16>,        \
     (const void*)pairs_kernel<R, kFlavorGlobal, Packed16>, (const void*)pairs_kernel<R, kFlavorSWScore, Scalar32>,       \
     (const void*)pairs_kernel<R, kFlavorSWEnd, Scalar32>, (const void*)pairs_kernel<R, kFlavorGlobal, Scalar32>}
static const void* const kPairsTable[2][6] = {OPAL_PAIRS_ROW(8), OPAL_PAIRS_ROW(16)};
static_assert(kPairsR[0] == 8 && kPairsR[1] == 16, "keep kPairsTable in step with kPairsR");

const void* pairs_kernel_fn(int rIndex, int type, int flavor) { return kPairsTable[rIndex][type * 3 + flavor]; }

}  // namespace opalb200
