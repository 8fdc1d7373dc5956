// A5/A6 — window segmentation of the matched pairs and the per-window epilogue of `cross`.
// Replaces genomes.get_bins_echr / get_bins_genome / get_bins_arrays (genomes.py:73-127), the window
// loop of CrossIdentifier.window_genotyper (csmatch.py:80-95) and get_window_data (csmatch.py:44-61).
#pragma once
#include "common.cuh"
#include "score.cuh"

namespace snpm {

// window number of a matched pair: win_off[c] + (pos-1)/bin_len when 1 <= pos and (pos-1)/bin_len <
// win_count[c] (window k covers [1+k*b, (k+1)*b], genomes.py:113-116), else -1 (in no window)
__device__ __forceinline__ int32_t window_of_pair(const int32_t *__restrict__ pair_s, const int32_t *__restrict__ chrom,
                                                  const int32_t *__restrict__ pos, const int32_t *__restrict__ win_count,
                                                  const int32_t *__restrict__ win_off, int64_t bin_len, int64_t r) {
    const int32_t i = pair_s[r];
    const int32_t c = chrom[i];
    const int64_t p = pos[i];
    if (c < 0 || p < 1) return -1;
    const int64_t k = (p - 1) / bin_len;
    if (k >= win_count[c]) return -1;
    return win_off[c] + int32_t(k);
}

// matched pairs of sample s are [mstart[s], mstart[s+1]), ordered by (panel chromosome, position), so the pairs of one window
// of one sample are contiguous: record [begin, end) in slot s*W + w (zero-initialised -> empty windows stay [0,0)).  A pair
// opening a sample never continues the previous pair's window: the previous sample closes its own last window.
__global__ void __launch_bounds__(256) k_window_bounds(const int32_t *__restrict__ pair_s, const int32_t *__restrict__ mstart, int32_t S,
                                                       int32_t W, const int32_t *__restrict__ chrom, const int32_t *__restrict__ pos,
                                                       const int32_t *__restrict__ win_count, const int32_t *__restrict__ win_off,
                                                       int64_t bin_len, int32_t *__restrict__ win_begin, int32_t *__restrict__ win_end) {
    const int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= mstart[S]) return;
    int lo = 0, hi = S;                                   // the sample: last s with mstart[s] <= r (empty samples are skipped)
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (mstart[mid] <= r) lo = mid; else hi = mid;
    }
    const int64_t first = mstart[lo], last = int64_t(mstart[lo + 1]) - 1;
    const int64_t slot0 = int64_t(lo) * W;
    const int32_t w = window_of_pair(pair_s, chrom, pos, win_count, win_off, bin_len, r);
    const int32_t wp = r > first ? window_of_pair(pair_s, chrom, pos, win_count, win_off, bin_len, r - 1) : -2;
    if (w != wp) {
        if (w >= 0) win_begin[slot0 + w] = int32_t(r);
        if (wp >= 0) win_end[slot0 + wp] = int32_t(r);
    }
    if (r == last && w >= 0) win_end[slot0 + w] = int32_t(r + 1);
}

// rows of every window on this device, and the packing of the per-window partials into ONE f64 buffer for a cross-GPU sum
// (SURVEY 8e: a window's rows lie in one SNP-row shard except at the <= G-1 shard boundaries; summing the [W, A] partials of all
// ranks handles both): red = score [W * a_pad] | ninfo as f64 [W * a_pad] | rows as f64 [W]  (integers are exact in f64)
__global__ void __launch_bounds__(256) k_window_nrows(const int32_t *__restrict__ win_begin, const int32_t *__restrict__ win_end, int32_t W,
                                                      int32_t *__restrict__ nrows) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w < W) nrows[w] = win_end[w] - win_begin[w];
}
__global__ void __launch_bounds__(256) k_window_pack(const double *__restrict__ part_score, const int32_t *__restrict__ part_ninfo,
                                                     const int32_t *__restrict__ nrows, int64_t cells, int32_t W, double *__restrict__ red) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < cells) {
        red[i] = part_score[i];
        red[cells + i] = double(part_ninfo[i]);
    }
    if (i < W) red[2 * cells + i] = double(nrows[i]);
}
__global__ void __launch_bounds__(256) k_window_unpack(const double *__restrict__ red, int64_t cells, int32_t W, double *__restrict__ part_score,
                                                       int32_t *__restrict__ part_ninfo, int32_t *__restrict__ nrows) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < cells) {
        part_score[i] = red[i];
        part_ninfo[i] = int32_t(red[cells + i]);
    }
    if (i < W) nrows[i] = int32_t(red[2 * cells + i]);
}

// One CTA per window: likelihoods from the FLOAT window scores, per-window nanmin, LR, the number of
// accessions with LR < lr_thres, and the identity call identical <=> floor(n - x - 1) + 1 <= kmax[n]
// (np_test_identity = binom.sf(n-x-1, n, e) >= 0.05, snpmatch.py:57-72; the table is built by the host
// with the same SciPy call).
__global__ void __launch_bounds__(256) k_window_epilogue(const double *__restrict__ part_score, const int32_t *__restrict__ part_ninfo,
                                                         int32_t a_pad, int32_t n_acc, const int32_t *__restrict__ win_begin,
                                                         const int32_t *__restrict__ win_end, const int32_t *__restrict__ kmax,
                                                         int64_t kmax_len, double lr_thres, double *__restrict__ win_L,
                                                         double *__restrict__ win_LR, uint8_t *__restrict__ win_ident,
                                                         int32_t *__restrict__ win_amb, int *status) {
    __shared__ double s_red[32];
    __shared__ int s_cnt;
    const int w = blockIdx.x;
    const int64_t base = int64_t(w) * n_acc;
    if (threadIdx.x == 0) s_cnt = 0;
    if (win_end[w] - win_begin[w] <= 0) {                 // the reference emits nothing for an empty window
        for (int acc = threadIdx.x; acc < n_acc; acc += blockDim.x) {
            win_L[base + acc] = nan("");
            win_LR[base + acc] = nan("");
            win_ident[base + acc] = 0;
        }
        if (threadIdx.x == 0) win_amb[w] = 0;
        return;
    }
    __syncthreads();
    double lmin = nan("");
    int viol = 0, kviol = 0;
    for (int acc = threadIdx.x; acc < n_acc; acc += blockDim.x) {
        const double y = part_score[int64_t(w) * a_pad + acc];
        const int32_t ni = part_ninfo[int64_t(w) * a_pad + acc];
        const double n = double(ni);
        if (y > n) ++viol;
        const double l = likeli_test(n, y);
        win_L[base + acc] = l;
        if (l == l) lmin = (lmin == lmin) ? fmin(lmin, l) : l;
        uint8_t ident = 0;
        if (ni < kmax_len) ident = (floor(n - y - 1.0) + 1.0 <= double(kmax[ni])) ? 1 : 0;
        else ++kviol;
        win_ident[base + acc] = ident;
    }
    if (viol) atomicAdd(status + 1, viol);
    if (kviol) atomicAdd(status + 2, kviol);
    double top = block_nanmin(lmin, s_red);
    if (isinf(top)) top = nan("");
    int amb = 0;
    for (int acc = threadIdx.x; acc < n_acc; acc += blockDim.x) {
        const double lr = (top <= 0.0) ? nan("") : win_L[base + acc] / top;
        win_LR[base + acc] = lr;
        if (lr < lr_thres) ++amb;
    }
    if (amb) atomicAdd(&s_cnt, amb);
    __syncthreads();
    if (threadIdx.x == 0) win_amb[w] = s_cnt;
}

// ---- compaction of the rows the reference keeps (csmatch.py:57-60) -------------------------------------------------
// A window contributes its accessions with LR < lr_thres, and only when at least one but not all pass.  win_row_off =
// exclusive scan of those counts over the S*W window slots (single CTA); k_window_compact then writes the surviving rows of
// every window in accession order: accession index, float score, informative sites, likelihood, identity call.
__global__ void __launch_bounds__(1024) k_window_row_offsets(const int32_t *__restrict__ win_amb, int32_t n_windows, int32_t n_acc,
                                                             int32_t *__restrict__ win_row_off) {
    __shared__ int s_warp[33];
    int carry = 0;
    for (int base = 0; base < n_windows; base += blockDim.x) {
        const int w = base + threadIdx.x;
        int v = 0;
        if (w < n_windows) {
            const int amb = win_amb[w];
            v = (amb >= 1 && amb < n_acc) ? amb : 0;
        }
        int total;
        const int ex = block_excl_scan(v, &total, s_warp);
        if (w < n_windows) win_row_off[w] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) win_row_off[n_windows] = carry;
}

__global__ void __launch_bounds__(256) k_window_compact(const double *__restrict__ part_score, const int32_t *__restrict__ part_ninfo,
                                                        int32_t a_pad, int32_t n_acc, const double *__restrict__ win_L,
                                                        const double *__restrict__ win_LR, const uint8_t *__restrict__ win_ident,
                                                        const int32_t *__restrict__ win_row_off, double lr_thres,
                                                        int32_t *__restrict__ row_acc, double *__restrict__ row_score,
                                                        int32_t *__restrict__ row_ninfo, double *__restrict__ row_L,
                                                        uint8_t *__restrict__ row_ident) {
    __shared__ int s_warp[33];
    const int w = blockIdx.x;
    const int out0 = win_row_off[w];
    if (win_row_off[w + 1] == out0) return;               // nothing survives in this window (whole CTA leaves)
    const int64_t base = int64_t(w) * n_acc;
    int carry = 0;
    for (int a0 = 0; a0 < n_acc; a0 += blockDim.x) {
        const int acc = a0 + threadIdx.x;
        const int keep = acc < n_acc && win_LR[base + acc] < lr_thres;
        int total;
        const int ex = block_excl_scan(keep, &total, s_warp);
        if (keep) {
            const int o = out0 + carry + ex;
            row_acc[o] = acc;
            row_score[o] = part_score[int64_t(w) * a_pad + acc];
            row_ninfo[o] = part_ninfo[int64_t(w) * a_pad + acc];
            row_L[o] = win_L[base + acc];
            row_ident[o] = win_ident[base + acc];
        }
        carry += total;
    }
}

}  // namespace snpm
