// Accession against accession: pairwiseScore's statistic (snpmatch.py:270-309) for every pair of a selection of the resident
// panel's accessions, over the rows the handle holds, as one-hot int8 GEMMs on the tensor cores with the GEMM of the
// shared-panel mode (gemm_onehot.cuh) run unchanged.
//
//   common[i, j] = sum_r [db[r, sel_i] called] * [db[r, sel_j] called]
//   same[i, j]   = sum_r [db[r, sel_i] called] * [db[r, sel_j] called] * [db[r, sel_i] == db[r, sel_j]]
//
// called = code 0, 1 or 2 (2 counts as missing with skip_hets).  Both are one product A_op[128 rows / 64 accessions] *
// B_op[256 accessions]^T per tile: A rows 0-63 are the one-hot of the accession's call ("same"), rows 64-127 ones in every
// class slot of a row the accession has called ("common"); B rows are the one-hot calls.  K slot = 4 * row + code, slot 3
// stays zero, so a k-block is 32 panel rows.
#pragma once
#include "common.cuh"
#include "gemm_onehot.cuh"

namespace snpm {

// Both operands of the panel rows [r0, r1) for the selection sel[0 .. n) from ONE read of the packed words: thread t of CTA
// (kb, nb) is selection entry nb * 256 + t; it reads its 32 rows of k-block kb, then writes its row of the B tile (nb, kb) and
// its two rows of the A tile (4 nb + t / 64, kb).  Every byte of both tile arrays is written (rows past r1 and entries past n
// are zero), so nothing is cleared first.  a_tiled [m_blocks][n_kb][OG_A_TILE], b_tiled [ceil(n / 256)][n_kb][OG_B_TILE].
__global__ void __launch_bounds__(256) k_acc_expand(const uint64_t *__restrict__ packed, int32_t stride, const int32_t *__restrict__ sel, int32_t n,
                                                    int64_t r0, int64_t r1, int32_t n_kb, int32_t m_blocks, int32_t skip_hets,
                                                    unsigned char *__restrict__ a_tiled, unsigned char *__restrict__ b_tiled) {
    const int kb = blockIdx.x, nb = blockIdx.y, t = threadIdx.x;
    const int i = nb * OG_BN + t;
    const int32_t acc = i < n ? sel[i] : -1;
    const uint64_t *pcol = packed + (acc >= 0 ? (acc >> 5) : 0);
    const int bit = acc & 31;
    const int64_t row0 = r0 + int64_t(kb) * OG_ROWS;
    uint32_t lo = 0u, hi = 0u;                                   // bit q: the two bits of row row0 + q (both set = missing)
#pragma unroll
    for (int q = 0; q < OG_ROWS; ++q) {
        const uint64_t x = acc >= 0 && row0 + q < r1 ? __ldg(pcol + (row0 + q) * stride) : ~uint64_t(0);
        lo |= ((uint32_t(x) >> bit) & 1u) << q;
        hi |= ((uint32_t(x >> 32) >> bit) & 1u) << q;
    }
    uint32_t called = ~(lo & hi);                                // codes 0 (00), 1 (lo), 2 (hi)
    if (skip_hets) called &= lo | ~hi;
    const int m = nb * 4 + (t >> 6);
    unsigned char *b_tile = b_tiled + (size_t(nb) * n_kb + kb) * OG_B_TILE;
    unsigned char *a_tile = m < m_blocks ? a_tiled + (size_t(m) * n_kb + kb) * OG_A_TILE : nullptr;
#pragma unroll
    for (int c = 0; c < 8; ++c) {                                // K chunk c = rows 4c .. 4c+3
        uint4 hot, has;
        uint32_t *ph = reinterpret_cast<uint32_t *>(&hot), *pa = reinterpret_cast<uint32_t *>(&has);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int row = 4 * c + q;
            const bool ok = (called >> row) & 1u;
            const uint32_t code = ((lo >> row) & 1u) | (((hi >> row) & 1u) << 1);
            ph[q] = ok ? 1u << (8 * code) : 0u;
            pa[q] = ok ? 0x00010101u : 0u;
        }
        *reinterpret_cast<uint4 *>(b_tile + og_tile_offset(t, c, OG_BN)) = hot;
        if (a_tile) {
            *reinterpret_cast<uint4 *>(a_tile + og_tile_offset(t & 63, c, OG_BM)) = hot;
            *reinterpret_cast<uint4 *>(a_tile + og_tile_offset(64 + (t & 63), c, OG_BM)) = has;
        }
    }
}

// dst[i * ld_dst + j] += part[i * ld_part + j] for both counts, i < rows, j < cols; grid (ceil(cols / 256), min(rows, 65535))
__global__ void __launch_bounds__(256) k_acc_accumulate(const int32_t *__restrict__ same_part, const int32_t *__restrict__ common_part,
                                                        int32_t ld_part, int32_t rows, int32_t cols, int64_t ld_dst,
                                                        int32_t *__restrict__ same, int32_t *__restrict__ common) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= cols) return;
    for (int i = blockIdx.y; i < rows; i += gridDim.y) {
        const int64_t src = int64_t(i) * ld_part + j, dst = int64_t(i) * ld_dst + j;
        same[dst] += same_part[src];
        common[dst] += common_part[src];
    }
}

// The block below the diagonal from the one above it: [c0 + j, r0 + i] = [r0 + i, c0 + j] for i < rows, j < cols, both counts,
// through a 32 x 32 tile in shared memory; grid (ceil(cols / 32), ceil(rows / 32)), block (32, 8)
__global__ void __launch_bounds__(256) k_acc_mirror(int32_t *__restrict__ same, int32_t *__restrict__ common, int64_t ld, int64_t r0, int64_t c0,
                                                    int32_t rows, int32_t cols) {
    __shared__ int32_t ts[32][33], tc[32][33];
    const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32, tx = threadIdx.x;
    for (int k = threadIdx.y; k < 32; k += 8) {
        const int i = i0 + k, j = j0 + tx;
        if (i < rows && j < cols) {
            const int64_t src = (r0 + i) * ld + c0 + j;
            ts[k][tx] = same[src];
            tc[k][tx] = common[src];
        }
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += 8) {
        const int j = j0 + k, i = i0 + tx;
        if (i < rows && j < cols) {
            const int64_t dst = (c0 + j) * ld + r0 + i;
            same[dst] = ts[tx][k];
            common[dst] = tc[tx][k];
        }
    }
}

}  // namespace snpm
