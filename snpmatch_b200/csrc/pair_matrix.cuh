// All-against-all pairsnp: the per-chromosome counts of pairwiseScore (snpmatch.py:270-309) for every pair of S samples as
// one-hot int8 GEMMs on the tensor cores, with the GEMM of the shared-panel mode (gemm_onehot.cuh) run unchanged.
//
//   common[c, i, j] = sum_{k in chromosome c} [i has k] * [j has k]
//   same[c, i, j]   = sum_{k in chromosome c} [i has k] * [j has k] * [class_i(k) == class_j(k)]
//
// k = a column of the union of all samples' markers; class = the id of the marker's GT string (< 8).  Both are one product
// A_op[128 rows / 64 samples] * B_op[256 samples]^T per tile: A rows 0-63 are the one-hot of the sample's class ("same"),
// rows 64-127 ones in every class slot of a marker the sample has ("common"); B rows are one-hot classes.  A k-block is
// always 128 K-bytes: 32 markers of 4 slots (<= 4 classes) or 16 markers of 8 slots (5-8 classes).
#pragma once
#include "common.cuh"
#include "gemm_onehot.cuh"

namespace snpm {

// Writes the operands of the columns [c0, c1) straight from the samples' CSR (col strictly ascending inside a sample) into
// tiles the caller has zeroed: a_tiled [m_blocks][n_kb][OG_A_TILE], b_tiled [n_blocks][n_kb][OG_B_TILE].  One warp per
// sample: two lanes find the sample's markers of the chunk by binary search, then the warp writes them.
template <int SLOTS>
__global__ void __launch_bounds__(256) k_pair_expand(const int64_t *__restrict__ offsets, const int32_t *__restrict__ col,
                                                     const uint8_t *__restrict__ cls, int32_t S, int32_t c0, int32_t c1, int32_t n_kb,
                                                     unsigned char *__restrict__ a_tiled, unsigned char *__restrict__ b_tiled) {
    static_assert(SLOTS == 4 || SLOTS == 8, "a marker takes 4 or 8 K-bytes");
    constexpr int MK = 128 / SLOTS;                             // markers per k-block
    const int lane = threadIdx.x & 31;
    const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (s >= S) return;
    long long bound = 0;
    if (lane < 2) {                                             // lane 0: first marker >= c0, lane 1: first marker >= c1
        const int32_t key = lane == 0 ? c0 : c1;
        int64_t lo = offsets[s], hi = offsets[s + 1];
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (col[mid] < key) lo = mid + 1;
            else hi = mid;
        }
        bound = lo;
    }
    const int64_t first = __shfl_sync(0xFFFFFFFFu, bound, 0), last = __shfl_sync(0xFFFFFFFFu, bound, 1);
    const int a_row = s & 63, b_row = s & 255;
    unsigned char *a_base = a_tiled + size_t(s >> 6) * n_kb * OG_A_TILE;
    unsigned char *b_base = b_tiled + size_t(s >> 8) * n_kb * OG_B_TILE;
    for (int64_t i = first + lane; i < last; i += 32) {
        const int k = col[i] - c0;
        const int kb = k / MK, slot0 = SLOTS * (k % MK);
        const int byte = slot0 + cls[i];
        unsigned char *at = a_base + size_t(kb) * OG_A_TILE;
        at[og_tile_offset(a_row, byte >> 4, OG_BM) + (byte & 15)] = 1;
        unsigned char *cm = at + og_tile_offset(64 + a_row, slot0 >> 4, OG_BM) + (slot0 & 15);
        if (SLOTS == 4) *reinterpret_cast<uint32_t *>(cm) = 0x01010101u;
        else *reinterpret_cast<uint2 *>(cm) = make_uint2(0x01010101u, 0x01010101u);
        b_base[size_t(kb) * OG_B_TILE + og_tile_offset(b_row, byte >> 4, OG_BN) + (byte & 15)] = 1;
    }
}

// out[i, j] += the GEMM's [S, ld] int32 result, for both counts; grid (ceil(S / 256), S)
__global__ void __launch_bounds__(256) k_pair_accumulate(const int32_t *__restrict__ same_part, const int32_t *__restrict__ common_part,
                                                         int32_t ld, int32_t S, int32_t *__restrict__ same, int32_t *__restrict__ common) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= S) return;
    const int64_t src = int64_t(i) * ld + j, dst = int64_t(i) * S + j;
    same[dst] += same_part[src];
    common[dst] += common_part[src];
}

}  // namespace snpm
