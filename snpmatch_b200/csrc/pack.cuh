// A0 — packed panel in HBM: int8 -> 2-bit bit-plane words, read-back, synthetic generator.
// Layout (see include/snpmatch_b200.h): per row and per 32 accessions one u64,
// low half = bit 0 of the codes (code & 3), high half = bit 1; padding = missing (3).
#pragma once
#include "common.cuh"

namespace snpm {

// One warp packs one (row, word): lane j reads the code of accession word*32+j.
// Values below 0 are missing calls (the reference masks every value < 0, snpmatch.py:84-86); values above 2 have no meaning in
// the reference's data (makedb.py:59) and are counted in *bad (the load is refused).
__global__ void __launch_bounds__(256) k_pack_int8(const int8_t *__restrict__ snps, int64_t n_rows, int32_t n_acc,
                                                   int32_t stride, uint64_t *__restrict__ packed, int *__restrict__ bad) {
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = (int64_t(gridDim.x) * blockDim.x) >> 5;
    const int64_t items = n_rows * stride;
    for (int64_t it = warp_global; it < items; it += n_warps) {
        const int64_t row = it / stride;
        const int32_t w = int32_t(it - row * stride);
        const int32_t acc = w * 32 + lane;
        uint32_t code = 3u;
        if (acc < n_acc) {
            const int v = snps[row * int64_t(n_acc) + acc];
            if (v > 2) atomicAdd(bad, 1);
            code = v < 0 || v > 2 ? 3u : uint32_t(v);
        }
        const uint32_t lo = __ballot_sync(0xffffffffu, code & 1u);
        const uint32_t hi = __ballot_sync(0xffffffffu, code & 2u);
        if (lane == 0) packed[it] = uint64_t(lo) | (uint64_t(hi) << 32);
    }
}

// Inverse of k_pack_int8 for a list of rows: out[k, n_acc] int8 (3 -> -1).
__global__ void __launch_bounds__(256) k_unpack_rows(const uint64_t *__restrict__ packed, int32_t stride, int32_t n_acc,
                                                     const int64_t *__restrict__ rows, int64_t k, int8_t *__restrict__ out) {
    const int64_t total = k * int64_t(n_acc);
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
        const int64_t r = i / n_acc;
        const int32_t a = int32_t(i - r * n_acc);
        const uint64_t w = packed[rows[r] * stride + (a >> 5)];
        const uint32_t lo = uint32_t(w) >> (a & 31) & 1u;
        const uint32_t hi = uint32_t(w >> 32) >> (a & 31) & 1u;
        const uint32_t code = lo | (hi << 1);
        out[i] = code == 3u ? int8_t(-1) : int8_t(code);
    }
}

// Rows on which the selected accessions carry at least two different called genotypes — the segregating SNPs of
// Genotype.identify_segregating_snps (snp_genotype.py:188-211 with segregting_snps :378-383: after masking missing
// calls, t_sum / t_r_sum < 1  <=>  more than one distinct called value).  One warp per row: lanes sweep the row's words,
// AND them with the accession-selection mask, and OR-reduce the three class planes.
__global__ void __launch_bounds__(256) k_segregating_rows(const uint64_t *__restrict__ packed, int64_t n_rows, int32_t stride,
                                                          const uint32_t *__restrict__ sel, uint8_t *__restrict__ flags) {
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = (int64_t(gridDim.x) * blockDim.x) >> 5;
    for (int64_t row = warp_global; row < n_rows; row += n_warps) {
        uint32_t has_ref = 0u, has_alt = 0u, has_het = 0u;
        for (int w = lane; w < stride; w += 32) {
            const uint64_t v = __ldg(packed + row * stride + w);
            const uint32_t lo = uint32_t(v), hi = uint32_t(v >> 32), m = sel[w];
            has_ref |= ~(lo | hi) & m;
            has_alt |= lo & ~hi & m;
            has_het |= hi & ~lo & m;
        }
        const int classes = (__any_sync(0xffffffffu, has_ref != 0u) ? 1 : 0) + (__any_sync(0xffffffffu, has_alt != 0u) ? 1 : 0) +
                            (__any_sync(0xffffffffu, has_het != 0u) ? 1 : 0);
        if (lane == 0) flags[row] = classes > 1;
    }
}

// Sample of marker i of a batch: the last s in [0, S) with off[s] <= i (empty samples share their offset with the next one).
__device__ __forceinline__ int64_t sample_of_marker(const int64_t *__restrict__ off, int64_t S, int64_t i) {
    int64_t lo = 0, hi = S;
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(off + mid) <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// Per-sample segregation filter of a batch (snpm_batch_set_segregation_filter), between the join and the compaction: a marker of
// sample s that the join matched to row r keeps it only when r segregates among s's selected accessions, with the predicate of
// k_segregating_rows.  The host compacts every selection to the words it touches (sel[sel_off[s] .. sel_off[s+1]) = (word,
// mask)), so a marker reads one 8-byte word (one 32-byte sector) per touched word, not its whole row.  Selections of more than
// SEGP_NARROW words are taken by the marker's whole warp after the per-thread pass, lanes sweeping the words.  CTAs are the
// join's tiles (JOIN_TILE markers): the tile's kept count replaces its tile_cnt, so scan, scatter and the sample ranges run as
// they do after a plain join.
constexpr int SEGP_THREADS = 1024;     // = JOIN_TILE
constexpr int SEGP_NARROW = 8;

__device__ __forceinline__ void seg_classes(uint64_t v, uint32_t m, uint32_t &has_ref, uint32_t &has_alt, uint32_t &has_het) {
    const uint32_t lo = uint32_t(v), hi = uint32_t(v >> 32);
    has_ref |= ~(lo | hi) & m;
    has_alt |= lo & ~hi & m;
    has_het |= hi & ~lo & m;
}

__global__ void __launch_bounds__(SEGP_THREADS) k_segregating_pairs(const uint64_t *__restrict__ packed, int32_t stride, const int64_t *__restrict__ off,
                                                                    int64_t S, int64_t n, const uint2 *__restrict__ sel,
                                                                    const int32_t *__restrict__ sel_off, int32_t *__restrict__ match_row,
                                                                    int32_t *__restrict__ tile_cnt) {
    const int lane = threadIdx.x & 31;
    const int64_t i = int64_t(blockIdx.x) * SEGP_THREADS + threadIdx.x;
    const int32_t matched = i < n ? match_row[i] : -1;
    int32_t row = matched, w0 = 0, w1 = 0;
    if (row >= 0) {
        const int64_t s = sample_of_marker(off, S, i);
        w0 = __ldg(sel_off + s);
        w1 = __ldg(sel_off + s + 1);
    }
    const bool wide = row >= 0 && w1 - w0 > SEGP_NARROW;
    if (row >= 0 && !wide) {
        uint32_t r = 0u, a = 0u, h = 0u;
        const uint64_t *p = packed + int64_t(row) * stride;
        for (int32_t k = w0; k < w1; ++k) {
            const uint2 wm = __ldg(sel + k);
            seg_classes(__ldg(p + wm.x), wm.y, r, a, h);
        }
        if ((r != 0u) + (a != 0u) + (h != 0u) < 2) row = -1;
    }
    for (unsigned pend = __ballot_sync(0xffffffffu, wide); pend; pend &= pend - 1u) {
        const int src = __ffs(pend) - 1;
        const int32_t r_src = __shfl_sync(0xffffffffu, row, src);
        const int32_t a0 = __shfl_sync(0xffffffffu, w0, src), a1 = __shfl_sync(0xffffffffu, w1, src);
        const uint64_t *p = packed + int64_t(r_src) * stride;
        uint32_t r = 0u, a = 0u, h = 0u;
        for (int32_t k = a0 + lane; k < a1; k += 32) {
            const uint2 wm = __ldg(sel + k);
            seg_classes(__ldg(p + wm.x), wm.y, r, a, h);
        }
        const int classes = (__any_sync(0xffffffffu, r != 0u) ? 1 : 0) + (__any_sync(0xffffffffu, a != 0u) ? 1 : 0) +
                            (__any_sync(0xffffffffu, h != 0u) ? 1 : 0);
        if (lane == src && classes < 2) row = -1;
    }
    if (row != matched) match_row[i] = -1;
    const int cnt = __syncthreads_count(row >= 0);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = cnt;
}

// counts[s] += matched markers of sample s whose flag is set (snpm_batch_count_flagged_pairs); lanes of one sample add once
__global__ void __launch_bounds__(256) k_count_flagged_pairs(const int32_t *__restrict__ match_row, const uint8_t *__restrict__ flags, int64_t n,
                                                             const int64_t *__restrict__ off, int64_t S, unsigned long long *__restrict__ counts) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const bool hit = i < n && match_row[i] >= 0 && flags[i] != 0;
    const int64_t s = hit ? sample_of_marker(off, S, i) : -1;
    const unsigned peers = __match_any_sync(0xffffffffu, s);
    if (hit && __ffs(peers) - 1 == int(threadIdx.x & 31)) atomicAdd(counts + s, (unsigned long long)__popc(peers));
}

// ---- synthetic panel: the integer hash of snpmatch_b200/synth.py --------------------------------
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t key, uint64_t seed) {
    uint64_t z = key + (seed + 1ull) * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__host__ __device__ __forceinline__ uint64_t row_alt_threshold(uint64_t seed, uint64_t row) {
    const uint64_t z = mix64((row << 20) | 0xFFFFFull, seed ^ 0x5A5Aull);
    const uint64_t u = z >> 32;
    return (((u * u) >> 32) * u) >> 32;
}

__host__ __device__ __forceinline__ uint32_t synth_code(uint64_t seed, uint64_t row, uint64_t col, uint64_t thr) {
    const uint64_t z = mix64((row << 20) | col, seed);
    const uint64_t u = z >> 32;
    uint32_t code = u < thr ? 1u : 0u;
    if (((z >> 16) & 0xFFFFull) < 131ull) code = 2u;     // synth.HET_THRESH
    if ((z & 0xFFFFull) < 3277ull) code = 3u;            // synth.MISS_THRESH
    return code;
}

// One thread produces one (row, word).
__global__ void __launch_bounds__(256) k_fill_synthetic(uint64_t *__restrict__ packed, int64_t n_rows, int32_t n_acc,
                                                        int32_t stride, uint64_t seed, int64_t row0_global) {
    const int64_t items = n_rows * stride;
    for (int64_t it = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; it < items; it += int64_t(gridDim.x) * blockDim.x) {
        const int64_t row = it / stride;
        const int32_t w = int32_t(it - row * stride);
        const uint64_t grow = uint64_t(row + row0_global);
        const uint64_t thr = row_alt_threshold(seed, grow);
        uint32_t lo = 0u, hi = 0u;
#pragma unroll 4
        for (int j = 0; j < 32; ++j) {
            const int32_t acc = w * 32 + j;
            const uint32_t code = acc < n_acc ? synth_code(seed, grow, uint64_t(acc), thr) : 3u;
            lo |= (code & 1u) << j;
            hi |= (code >> 1) << j;
        }
        packed[it] = uint64_t(lo) | (uint64_t(hi) << 32);
    }
}

}  // namespace snpm
