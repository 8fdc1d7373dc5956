// A7 — simulated F1 pass.  Replaces the loop body of CrossIdentifier.match_insilico_f1s
// (csmatch.py:115-126): for every pair (i, j) of the given accession columns, over the whole-genome
// matched rows: both hom-alt -> wei[:,2]; both hom-ref -> wei[:,0]; both called and different ->
// wei[:,1]; numinfo counts those three cases.
#pragma once
#include "common.cuh"

namespace snpm {

constexpr int F1_THREADS = 256;
constexpr int F1_ROWS_PER_BLOCK = 4096;

__device__ __forceinline__ uint32_t code_at(const uint64_t *__restrict__ rowp, int32_t acc) {
    const uint64_t w = __ldg(rowp + (acc >> 5));
    const uint32_t lo = uint32_t(w) >> (acc & 31) & 1u;
    const uint32_t hi = uint32_t(w >> 32) >> (acc & 31) & 1u;
    return lo | (hi << 1);
}

// grid (pairs, row blocks, samples); partial[sample][pair][block] = (sum_alt, sum_ref, sum_het, count).  Sample s owns the
// matched pairs [mstart[s], mstart[s+1]) and the accession list acc_idx[s * n_top ...]; its row blocks start at its first pair,
// so a sample's sums do not depend on the other samples of the batch.  Blocks past a sample's pairs write zeros (the grid is
// sized for the largest sample).  The pairs sit on grid x (up to 2^31 - 1) because n_top = 4096 gives 8 386 560 of them; the
// row blocks sit on grid y, so a sample may have at most 65 535 * F1_ROWS_PER_BLOCK matched pairs.
__global__ void __launch_bounds__(F1_THREADS) k_f1_partial(const uint64_t *__restrict__ packed, int32_t stride,
                                                           const int32_t *__restrict__ pair_db, const double *__restrict__ pair_w,
                                                           const int32_t *__restrict__ mstart, const int32_t *__restrict__ acc_idx,
                                                           int32_t n_top, double *__restrict__ partial) {
    __shared__ double s_sum[3][F1_THREADS / 32];
    __shared__ long long s_cnt[F1_THREADS / 32];
    // pair index -> (i, j), i < j, itertools.combinations order
    int pi = blockIdx.x, i = 0;
    while (pi >= n_top - 1 - i) { pi -= n_top - 1 - i; ++i; }
    const int j = i + 1 + pi;
    const int s = blockIdx.z;
    const int32_t a1 = acc_idx[int64_t(s) * n_top + i], a2 = acc_idx[int64_t(s) * n_top + j];
    const int64_t m = mstart[s + 1];
    const int64_t r0 = mstart[s] + int64_t(blockIdx.y) * F1_ROWS_PER_BLOCK;
    const int64_t r1 = min(m, r0 + F1_ROWS_PER_BLOCK);
    double alt = 0.0, ref = 0.0, het = 0.0;
    long long cnt = 0;
    for (int64_t r = r0 + threadIdx.x; r < r1; r += F1_THREADS) {
        const uint64_t *rowp = packed + int64_t(pair_db[r]) * stride;
        const uint32_t g1 = code_at(rowp, a1), g2 = code_at(rowp, a2);
        const double *w = pair_w + 4 * r;
        // pair_w rows are (w_ref, w_alt, w_het, 0)
        if (g1 == 1u && g2 == 1u) { alt += w[1]; ++cnt; }
        else if (g1 == 0u && g2 == 0u) { ref += w[0]; ++cnt; }
        else if (g1 != 3u && g2 != 3u && g1 != g2) { het += w[2]; ++cnt; }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        alt += __shfl_xor_sync(0xffffffffu, alt, d);
        ref += __shfl_xor_sync(0xffffffffu, ref, d);
        het += __shfl_xor_sync(0xffffffffu, het, d);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s_sum[0][warp] = alt; s_sum[1][warp] = ref; s_sum[2][warp] = het; s_cnt[warp] = cnt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double A = 0.0, R = 0.0, H = 0.0;
        long long C = 0;
        for (int k = 0; k < F1_THREADS / 32; ++k) { A += s_sum[0][k]; R += s_sum[1][k]; H += s_sum[2][k]; C += s_cnt[k]; }
        double *o = partial + ((int64_t(s) * gridDim.x + blockIdx.x) * gridDim.y + blockIdx.y) * 4;
        o[0] = A; o[1] = R; o[2] = H; o[3] = double(C);
    }
}

// one thread per (sample, pair) sums the block partials in order: out[sample][pair] = (score, count); n_pairs here counts the
// pairs of all samples
__global__ void k_f1_final(const double *__restrict__ partial, int n_blocks, int n_pairs, double *__restrict__ out) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    double A = 0.0, R = 0.0, H = 0.0, C = 0.0;
    for (int b = 0; b < n_blocks; ++b) {
        const double *o = partial + (int64_t(p) * n_blocks + b) * 4;
        A += o[0]; R += o[1]; H += o[2]; C += o[3];
    }
    out[2 * p] = (A + R) + H;        // np.sum(alt) + np.sum(ref) + np.sum(het), csmatch.py:122
    out[2 * p + 1] = C;
}

}  // namespace snpm
