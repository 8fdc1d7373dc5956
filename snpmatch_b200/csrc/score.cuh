// A2/A3/A4 — per-accession scoring of matched rows, chunk combine, likelihood epilogue.
//
// k_score_segments is the hot kernel.  It restates matchGTsAccs (snpmatch.py:74-89) for a list of
// row segments — the 1000-pair chunks of Genotyper.genotyper (snpmatch.py:218-225) or the windows of
// CrossIdentifier.window_genotyper (csmatch.py:80-95) — in the reference's floating-point order:
// per accession and class a plain left-to-right sum over the segment's rows, classes combined as
// ((0 + ref) + het) + alt (SURVEY A.2), so fp64 scores are bit-identical to NumPy's.
//
// Data movement: a CTA owns a contiguous word slice of every row of ONE segment.  A dedicated producer
// warp gathers the segment's rows of the 2-bit panel (one 1-D TMA bulk copy per row, cp.async.bulk +
// mbarrier complete_tx) and the matched weights (one bulk copy per tile) into an SC_STAGES-deep shared
// memory ring; consumer warps release a stage through an "empty" mbarrier, so no block-wide barrier sits
// in the loop.
//
// Arithmetic: a consumer warp owns SC_WPW words (32 accessions each); lane = accession.  Rows are taken
// 32 at a time: lane l loads row l's word, a 5-stage shuffle butterfly transposes the two bit planes so
// that every lane holds the 32 row-bits of ITS accession, class masks cost one LOP3 per 32 rows, ninfo is
// a popcount, and the unrolled row loop tests immediate bit positions — which ptxas turns into R2P (seven
// predicates per instruction) feeding predicated DADDs.  The FP64 pipe (two DADDs per comparison: ref and
// alt; het only for rows that have one) is what bounds the kernel, not HBM.
#pragma once
#include "common.cuh"
#include <cooperative_groups.h>

namespace snpm {

constexpr int SC_TILE_ROWS = 64;   // multiple of 32
constexpr int SC_STAGES = 4;
constexpr int SC_WPW = 4;          // words (of 32 accessions) per consumer warp
constexpr int SC_MAX_WARPS = 12;   // consumer warps per CTA (+1 producer warp)

// ---- PTX helpers (sm_100a) ----------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return uint32_t(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// named barriers 1..SC_STAGES signal "stage free": consumer warps arrive (non-blocking), the producer warp syncs and
// therefore sleeps in hardware instead of spinning on an mbarrier and stealing issue slots from the consumers
__device__ __forceinline__ void named_bar_arrive(int id, int n_threads) {
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n_threads) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int n_threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n_threads) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
// 1-D TMA bulk copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst_smem, const void *src_gmem, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
                 "l"(src_gmem), "r"(bytes), "r"(bar)
                 : "memory");
}

// 16-byte Ampere-style async copy global -> shared (LDGSTS) and its mbarrier hook
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void *src_gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint32_t bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}

#ifndef SC_GATHER_LDGSTS
#define SC_GATHER_LDGSTS 1      // 1: rows gathered with 16-byte cp.async by the producer warp; 0: one TMA bulk copy per row
#endif

struct ScoreArgs {
    const uint64_t *packed;     // [n_rows, stride]
    int32_t stride;
    const int32_t *pair_db;     // matched local rows
    const double *pair_w;       // [m, 4] = (w_ref, w_alt, w_het, 0) per matched pair, 32-byte rows
    // chunk mode (table == 0): segment j belongs to sample s with seg_off[s] <= j < seg_off[s+1]
    const int32_t *seg_off;     // [S+1]
    const int32_t *mstart;      // [S+1]
    int32_t S;
    int32_t chunk;
    // table mode (table == 1): explicit [begin, end) per segment
    const int32_t *seg_begin;
    const int32_t *seg_end;
    int32_t table;
    int32_t nseg;               // table mode: number of segments; chunk mode: unused (seg_off[S])
    double *part_score;         // [nseg, a_pad]
    int32_t *part_ninfo;        // [nseg, a_pad]
    int32_t a_pad;              // stride * 32
};

// shared-memory pitch of one staged row slice: a multiple of 16 bytes (TMA) whose 16-byte count is odd, so
// that the 64-bit row-per-lane loads of the transpose are at worst 2-way bank conflicted
__host__ __device__ __forceinline__ uint32_t score_row_pitch(int slice_words) {
    const uint32_t b = uint32_t(slice_words) * 8u;
    return ((b >> 4) & 1u) ? b : b + 16u;
}

// 32x32 bit transpose across the warp: on return bit r of lane l = bit l of the value lane r passed in
__device__ __forceinline__ uint32_t warp_transpose32(uint32_t x, const uint32_t (&sel)[5], const uint32_t (&rot)[5]) {
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        uint32_t y = __shfl_xor_sync(0xffffffffu, x, 16 >> s);
        y = __funnelshift_l(y, y, rot[s]);
        x = (x & ~sel[s]) | (y & sel[s]);
    }
    return x;
}

template <bool SKIP_HETS, int NWARPS, int MIN_BLOCKS>
__global__ void __launch_bounds__(32 * NWARPS, MIN_BLOCKS) k_score_segments(const ScoreArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x, warp = threadIdx.y, ncons = blockDim.y - 1;
    const bool producer = warp == ncons;
    const int seg = blockIdx.x;

    int32_t begin, end;
    if (a.table) {
        if (seg >= a.nseg) return;
        begin = a.seg_begin[seg];
        end = a.seg_end[seg];
    } else {
        if (seg >= a.seg_off[a.S]) return;
        int lo = 0, hi = a.S;                 // last s with seg_off[s] <= seg
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (a.seg_off[mid] <= seg) lo = mid; else hi = mid - 1;
        }
        begin = a.mstart[lo] + (seg - a.seg_off[lo]) * a.chunk;
        end = min(a.mstart[lo + 1], begin + a.chunk);
    }

    const int w_start = blockIdx.y * (SC_WPW * ncons);
    const int slice_words = min(SC_WPW * ncons, a.stride - w_start);
    const uint32_t slice_bytes = uint32_t(slice_words) * 8u;
    const uint32_t pitch = score_row_pitch(SC_WPW * ncons);
    const int vw = max(0, min(SC_WPW, slice_words - warp * SC_WPW));   // valid words of this warp: 0, 2 or 4

    // shared memory: full[STAGES], empty[STAGES] mbarriers | STAGES x (row tile | weight tile)
    uint64_t *full = reinterpret_cast<uint64_t *>(smem);
    const uint32_t tile_bytes = uint32_t(SC_TILE_ROWS) * pitch;
    const uint32_t wtile_bytes = SC_TILE_ROWS * 32u;
    unsigned char *stage0 = smem + 128;
    const uint32_t stage_bytes = tile_bytes + wtile_bytes;

    const int n_rows = end - begin;
    const int n_tiles = (n_rows + SC_TILE_ROWS - 1) / SC_TILE_ROWS;

    if (n_tiles > 0) {
        if (warp == 0 && lane == 0) {
            for (int s = 0; s < SC_STAGES; ++s) {
                mbar_init(smem_u32(full + s), SC_GATHER_LDGSTS ? 33u : 1u);
            }
            mbar_fence_init();
        }
        __syncthreads();
    }

    if (producer) {
        // ---- producer warp: gather rows + weights of tile t into stage t % STAGES ----------------------
        for (int t = 0; t < n_tiles; ++t) {
            const int st = t % SC_STAGES;
            if (t >= SC_STAGES) named_bar_sync(1 + st, 32 * (ncons + 1));
            const int r0 = begin + t * SC_TILE_ROWS;
            const int rows = min(SC_TILE_ROWS, end - r0);
            const uint32_t bar = smem_u32(full + st);
            unsigned char *dst = stage0 + size_t(st) * stage_bytes;
#if SC_GATHER_LDGSTS
            // row indices of the tile: lane l keeps rows l and l+32, handed out by shuffle below
            const int64_t idx0 = lane < rows ? int64_t(a.pair_db[r0 + lane]) : 0;
            const int64_t idx1 = lane + 32 < rows ? int64_t(a.pair_db[r0 + 32 + lane]) : 0;
            if (lane == 0) {
                mbar_arrive_expect_tx(bar, uint32_t(rows) * 32u);
                tma_bulk_g2s(smem_u32(dst + tile_bytes), a.pair_w + 4 * int64_t(r0), uint32_t(rows) * 32u, bar);
            }
            const uint32_t cpr = slice_bytes >> 4;                         // 16-byte chunks per row slice
            const uint32_t total = uint32_t(rows) * cpr;
            const uint32_t magic = cpr > 1u ? 0xFFFFFFFFu / cpr + 1u : 0u; // floor(i / cpr) = umulhi(i, magic) for i < 2^16, cpr > 1
            const uint64_t *src0 = a.packed + w_start;
#pragma unroll 6
            for (uint32_t i = lane; i < ((total + 31u) & ~31u); i += 32) {
                const uint32_t r = cpr > 1u ? __umulhi(i, magic) : i, c = i - r * cpr;
                const int64_t lo_i = __shfl_sync(0xffffffffu, idx0, r & 31), hi_i = __shfl_sync(0xffffffffu, idx1, r & 31);
                const int64_t row = r < 32 ? lo_i : hi_i;
                if (i < total) cp_async16(smem_u32(dst + size_t(r) * pitch + c * 16u), src0 + row * a.stride + c * 2u);
            }
            cp_async_mbar_arrive_noinc(bar);
#else
            if (lane == 0) mbar_arrive_expect_tx(bar, uint32_t(rows) * (slice_bytes + 32u));
            __syncwarp();
            for (int r = lane; r < rows; r += 32) {
                const int64_t row = a.pair_db[r0 + r];
                tma_bulk_g2s(smem_u32(dst + size_t(r) * pitch), a.packed + row * a.stride + w_start, slice_bytes, bar);
            }
            if (lane == 0) tma_bulk_g2s(smem_u32(dst + tile_bytes), a.pair_w + 4 * int64_t(r0), uint32_t(rows) * 32u, bar);
#endif
        }
        return;
    }

    // ---- consumer warps --------------------------------------------------------------------------------
    double s_ref[SC_WPW], s_het[SC_WPW], s_alt[SC_WPW];
    int32_t ninfo[SC_WPW];
#pragma unroll
    for (int j = 0; j < SC_WPW; ++j) { s_ref[j] = 0.0; s_het[j] = 0.0; s_alt[j] = 0.0; ninfo[j] = 0; }
    const uint32_t lanebit = 1u << lane;
    // per-stage constants of the transpose butterfly (j = 16, 8, 4, 2, 1)
    uint32_t t_sel[5], t_rot[5];
    {
        const uint32_t m[5] = {0x0000FFFFu, 0x00FF00FFu, 0x0F0F0F0Fu, 0x33333333u, 0x55555555u};
#pragma unroll
        for (int s = 0; s < 5; ++s) {
            const int j = 16 >> s;
            t_sel[s] = (lane & j) ? m[s] : ~m[s];
            t_rot[s] = (lane & j) ? uint32_t(32 - j) : uint32_t(j);
        }
    }

    // PRMT selectors of the two byte-exchange stages: [send, merge even, merge odd] for accession bit 4, then bit 3
    uint32_t b_sel[6];
    b_sel[0] = (lane & 16) ? 0x5410u : 0x7632u;
    b_sel[1] = (lane & 16) ? 0x3254u : 0x5410u;
    b_sel[2] = (lane & 16) ? 0x3276u : 0x7610u;
    b_sel[3] = (lane & 8) ? 0x6420u : 0x7531u;
    b_sel[4] = (lane & 8) ? 0x3514u : 0x5240u;
    b_sel[5] = (lane & 8) ? 0x3716u : 0x7260u;

    for (int t = 0; t < n_tiles; ++t) {
        const int st = t % SC_STAGES;
        mbar_wait(smem_u32(full + st), uint32_t(t / SC_STAGES) & 1u);
        const int rows = min(SC_TILE_ROWS, n_rows - t * SC_TILE_ROWS);
        const unsigned char *tile = stage0 + size_t(st) * stage_bytes;
        const unsigned char *wt = tile + tile_bytes;
        {
            for (int g0 = 0; g0 < rows; g0 += 32) {
                // lane l holds row g0+l: load its SC_WPW words, transpose both bit planes
                const bool have = g0 + lane < rows;
                const unsigned char *mine = tile + size_t(g0 + lane) * pitch + warp * (SC_WPW * 8);
                // class planes of row g0+lane: x[j] = hom-ref plane of word j, x[4+j] = hom-alt plane (bit = accession);
                // the het plane stays row-major and is consulted only for rows that hold a het
                uint32_t x[2 * SC_WPW], het[SC_WPW], het_rows[SC_WPW];
#pragma unroll
                for (int j = 0; j < SC_WPW; ++j) {
                    uint64_t v = ~0ull;
                    if (have && j < vw) v = *reinterpret_cast<const uint64_t *>(mine + j * 8);
                    const uint32_t lo = uint32_t(v), hi = uint32_t(v >> 32);
                    het[j] = hi & ~lo;
                    het_rows[j] = SKIP_HETS ? 0u : __ballot_sync(0xffffffffu, het[j] != 0u);
                    x[j] = ~(lo | hi);
                    x[SC_WPW + j] = lo & ~hi;
                    // informative sites of this lane's accession (snpmatch.py:78-79,88): transpose the plane of called
                    // genotypes (hets count unless they are skipped) and count its rows
                    ninfo[j] += __popc(warp_transpose32(SKIP_HETS ? (x[j] | x[SC_WPW + j]) : ~(lo & hi), t_sel, t_rot));
                }
                // (1) inside the lane: 8x8 bit transpose of the eight planes per byte column, after which byte b of
                //     x[i] holds the eight class flags (ref word 0-3, alt word 0-3) of accession 8b+i in this row
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    const int jj = 4 >> s;
                    const uint32_t m = s == 0 ? 0x0F0F0F0Fu : (s == 1 ? 0x33333333u : 0x55555555u);
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        if (k & jj) continue;
                        const uint32_t t = ((x[k] >> jj) ^ x[k + jj]) & m;
                        x[k + jj] ^= t;
                        x[k] ^= t << jj;
                    }
                }
                // (2) across the warp: 32x32 transpose of those bytes (lane <-> accession, slot <-> row); afterwards
                //     byte b of x[i] in lane a holds the flags of (row 8b+i, accession a)
#pragma unroll
                for (int k = 0; k < 4; ++k) {          // accession bit 4: byte positions {2,3} <-> {0,1}
                    const uint32_t recv = __shfl_xor_sync(0xffffffffu, __byte_perm(x[2 * k], x[2 * k + 1], b_sel[0]), 16);
                    x[2 * k] = __byte_perm(x[2 * k], recv, b_sel[1]);
                    x[2 * k + 1] = __byte_perm(x[2 * k + 1], recv, b_sel[2]);
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {          // accession bit 3: byte positions {1,3} <-> {0,2}
                    const uint32_t recv = __shfl_xor_sync(0xffffffffu, __byte_perm(x[2 * k], x[2 * k + 1], b_sel[3]), 8);
                    x[2 * k] = __byte_perm(x[2 * k], recv, b_sel[4]);
                    x[2 * k + 1] = __byte_perm(x[2 * k + 1], recv, b_sel[5]);
                }
#pragma unroll
                for (int q = 2; q >= 0; --q) {         // accession bits 2..0: whole registers
                    const bool up = (lane >> q) & 1;
#pragma unroll
                    for (int i0 = 0; i0 < 8; ++i0) {
                        if (i0 & (1 << q)) continue;
                        const int i1 = i0 | (1 << q);
                        const uint32_t recv = __shfl_xor_sync(0xffffffffu, up ? x[i0] : x[i1], 1 << q);
                        x[i0] = up ? recv : x[i0];
                        x[i1] = up ? x[i1] : recv;
                    }
                }
                const unsigned char *wg = wt + g0 * 32;
                // Row loop: the eight flags of a row sit in one register byte, so ptxas extracts them with one R2P (7
                // predicates) + one LOP3 and they feed eight INDEPENDENT predicated DADDs (four words x ref/alt).  Each
                // accumulator still sees its rows in ascending order.  The add is a volatile asm so that neither nvvm
                // nor ptxas rewrites it as add + select.
#pragma unroll
                for (int r = 0; r < 32; ++r) {
                    const uint32_t z = x[r & 7];
                    const int sh = (r >> 3) * 8;
                    const double2 w_ra = *reinterpret_cast<const double2 *>(wg + r * 32);     // (w_ref, w_alt)
                    const double w_ref = w_ra.x, w_alt = w_ra.y;
#pragma unroll
                    for (int j = 0; j < SC_WPW; ++j)
                        if (z & (1u << (sh + j))) asm volatile("add.f64 %0, %0, %1;" : "+d"(s_ref[j]) : "d"(w_ref));
#pragma unroll
                    for (int j = 0; j < SC_WPW; ++j)
                        if (z & (1u << (sh + SC_WPW + j))) asm volatile("add.f64 %0, %0, %1;" : "+d"(s_alt[j]) : "d"(w_alt));
                }
                if (!SKIP_HETS) {
                    // hets are rare (makedb.py:59 code 2; ~0.2 % of calls): visit only the rows of a word that hold
                    // one, in ascending row order (het_rows is warp-uniform, so the loop does not diverge)
#pragma unroll
                    for (int j = 0; j < SC_WPW; ++j) {
                        uint32_t m = het_rows[j];
                        while (m) {
                            const int r = __ffs(m) - 1;
                            m &= m - 1;
                            const double w_het = *reinterpret_cast<const double *>(wg + r * 32 + 16);
                            const uint32_t hw = __shfl_sync(0xffffffffu, het[j], r);       // het plane of row r
                            if (hw & lanebit) asm volatile("add.f64 %0, %0, %1;" : "+d"(s_het[j]) : "d"(w_het));
                        }
                    }
                }
            }
        }
        if (t + SC_STAGES < n_tiles) named_bar_arrive(1 + st, 32 * (ncons + 1));   // this warp is done with stage st
    }

#pragma unroll
    for (int j = 0; j < SC_WPW; ++j) {
        if (j < vw) {
            const int64_t acc = int64_t(w_start + warp * SC_WPW + j) * 32 + lane;
            const int64_t o = int64_t(seg) * a.a_pad + acc;
            a.part_score[o] = ((0.0 + s_ref[j]) + s_het[j]) + s_alt[j];     // snpmatch.py:84-87
            a.part_ninfo[o] = ninfo[j];
        }
    }
}

static inline void score_launch_shape(int32_t stride, int *nwarps, int *yblocks, size_t *smem_bytes) {
    int nw = (stride + SC_WPW - 1) / SC_WPW;       // consumer warps
    if (nw > SC_MAX_WARPS) nw = 8;
    *nwarps = nw;
    *yblocks = (stride + SC_WPW * nw - 1) / (SC_WPW * nw);
    *smem_bytes = 128 + size_t(SC_STAGES) * (size_t(SC_TILE_ROWS) * score_row_pitch(SC_WPW * nw) + SC_TILE_ROWS * 32);
}

// ---- combine: sequential sum of the segment partials of one sample, in segment order ----------------
// (ScoreList = ScoreList + t_s, snpmatch.py:224-225; TotScoreList, csmatch.py:88-89)
// red row layout [2*n_acc + 2]: score[n_acc] | ninfo[n_acc] as f64 | matched pairs | y>n violations
__global__ void __launch_bounds__(256) k_combine(const double *__restrict__ part_score, const int32_t *__restrict__ part_ninfo,
                                                 int32_t a_pad, int32_t n_acc, const int32_t *__restrict__ seg_off,
                                                 const int32_t *__restrict__ mstart, int32_t nseg_table,
                                                 const int32_t *__restrict__ seg_begin, const int32_t *__restrict__ seg_end,
                                                 double *__restrict__ red) {
    const int s = blockIdx.y;
    const int acc = blockIdx.x * blockDim.x + threadIdx.x;
    // without seg_off the segments are windows: sample s owns the slots [s * nseg_table, (s+1) * nseg_table)
    int j0, j1;
    if (seg_off) { j0 = seg_off[s]; j1 = seg_off[s + 1]; } else { j0 = s * nseg_table; j1 = j0 + nseg_table; }
    double *row = red + int64_t(s) * (2 * int64_t(n_acc) + 2);
    if (acc < n_acc) {
        double tot = 0.0;
        long long ni = 0;
        // the adds are sequential (reference order); the loads are not: fetch 16 segments ahead, then add in order
        constexpr int CB = 16;
        int j = j0;
        for (; j + CB <= j1; j += CB) {
            double v[CB];
            int32_t c[CB];
#pragma unroll
            for (int k = 0; k < CB; ++k) {
                v[k] = __ldg(part_score + int64_t(j + k) * a_pad + acc);
                c[k] = __ldg(part_ninfo + int64_t(j + k) * a_pad + acc);
            }
#pragma unroll
            for (int k = 0; k < CB; ++k) {
                tot = tot + v[k];
                ni += c[k];
            }
        }
        for (; j < j1; ++j) {
            tot = tot + part_score[int64_t(j) * a_pad + acc];
            ni += part_ninfo[int64_t(j) * a_pad + acc];
        }
        row[acc] = tot;
        row[n_acc + acc] = double(ni);
    }
    if (acc == 0) {
        long long m = 0;
        if (seg_off) m = mstart[s + 1] - mstart[s];
        else for (int j = j0; j < j1; ++j) m += seg_end[j] - seg_begin[j];
        row[2 * n_acc] = double(m);
        row[2 * n_acc + 1] = 0.0;
    }
}

// ---- likelihood epilogue ------------------------------------------------------------------------
// likeliTest (snpmatch.py:40-55)
__device__ __forceinline__ double likeli_test(double n, double y) {
    const double p = 0.99999999;
    if (n == 0.0) return nan("");
    if (y == n) return 1.0;
    if (y > 0.0) {
        const double ps = y / n;
        return y * log(ps / p) + (n - y) * log((1.0 - ps) / (1.0 - p));
    }
    return nan("");
}

__device__ __forceinline__ double block_nanmin(double v, double *s_red /*[32]*/) {
    // nan-ignoring minimum over the block; +inf when every value is nan
    double x = (v == v) ? v : __longlong_as_double(0x7ff0000000000000ll);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) x = fmin(x, __shfl_xor_sync(0xffffffffu, x, d));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) s_red[warp] = x;
    __syncthreads();
    x = lane < nwarp ? s_red[lane] : __longlong_as_double(0x7ff0000000000000ll);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) x = fmin(x, __shfl_xor_sync(0xffffffffu, x, d));
    return x;
}

// One thread-block CLUSTER per sample row of `red` (E CTAs, each takes every E-th stretch of blockDim accessions): the
// per-accession work — truncation, probability, the two fp64 logarithms of likeliTest — spreads over E SMs, the sample's
// minimum likelihood is combined through distributed shared memory (every CTA reads the E block minima after one
// cluster barrier) and the ratios follow in the same launch.  With one 1024-thread CTA per sample the epilogue of a rank
// that finishes 8 samples of a 20 000-accession panel ran on 8 SMs (0.049 ms).
// truncate != 0: y = int(score) first (GenotyperOutput.__init__, snpmatch.py:96).  amin_mode 0: TopHit = nanmin(L); 1: TopHit = amin.
// `pitch` = doubles per sample row of `red` (2*n_acc + 2, or 3*n_acc + 2 for grouped batches; the first 2*n_acc + 2 are used).
__global__ void __launch_bounds__(1024) k_epilogue(double *__restrict__ red, int64_t pitch, int32_t n_acc, int truncate, int amin_mode, double amin,
                                                   int64_t *__restrict__ matches, int64_t *__restrict__ ninfo64,
                                                   double *__restrict__ prob, double *__restrict__ L, double *__restrict__ LR) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned E = cluster.num_blocks(), rank = cluster.block_rank();
    __shared__ double s_red[32];
    __shared__ double s_top;
    __shared__ int s_viol;
    const int s = blockIdx.x / E;
    double *row = red + int64_t(s) * pitch;
    if (threadIdx.x == 0) s_viol = 0;
    __syncthreads();
    double lmin = nan("");
    int viol = 0;
    const int first = int(rank * blockDim.x + threadIdx.x), step = int(E * blockDim.x);
    for (int acc = first; acc < n_acc; acc += step) {
        double y = row[acc];
        const double n = row[n_acc + acc];
        if (truncate) y = double((long long)y);
        const int64_t o = int64_t(s) * n_acc + acc;
        if (matches) matches[o] = (long long)y;
        if (ninfo64) ninfo64[o] = (long long)n;
        prob[o] = n > 0.0 ? y / n : nan("");                  // get_fraction, snpmatch.py:25-28
        if (y > n) ++viol;
        const double l = likeli_test(n, y);
        L[o] = l;
        if (l == l) lmin = (lmin == lmin) ? fmin(lmin, l) : l;
    }
    if (viol) atomicAdd(&s_viol, viol);
    const double mine = block_nanmin(lmin, s_red);           // +inf when every value of this CTA is nan
    if (threadIdx.x == 0) s_top = mine;
    cluster.sync();                                          // every CTA's minimum and violation count are in its shared memory
    double top = __longlong_as_double(0x7ff0000000000000ll);
    for (unsigned e = 0; e < E; ++e) top = fmin(top, *cluster.map_shared_rank(&s_top, e));
    if (isinf(top)) top = nan("");                           // all nan (np.nanmin -> nan)
    if (amin_mode) top = amin;
    for (int acc = first; acc < n_acc; acc += step) {
        const int64_t o = int64_t(s) * n_acc + acc;
        LR[o] = (top <= 0.0) ? nan("") : L[o] / top;         // get_fraction(L, TopHit)
    }
    if (rank == 0 && threadIdx.x == 0) {
        int v = 0;
        for (unsigned e = 0; e < E; ++e) v += *cluster.map_shared_rank(&s_viol, e);
        row[2 * n_acc + 1] = double(v);
    }
    cluster.sync();                                          // nobody leaves while its shared memory may still be read
}

// launch: clusters of 1, 2, 4 or 8 CTAs of 256 threads per sample, about two accessions per thread at most until the cluster is full
inline cudaError_t launch_epilogue(cudaStream_t st, int64_t n_samples, double *red, int64_t pitch, int32_t n_acc, int truncate, int amin_mode, double amin,
                                   int64_t *matches, int64_t *ninfo64, double *prob, double *L, double *LR) {
    if (n_samples <= 0) return cudaSuccess;
    unsigned E = 1;
    while (E < 8 && int64_t(E) * 512 < n_acc) E *= 2;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(unsigned(n_samples) * E, 1, 1);
    cfg.blockDim = dim3(256, 1, 1);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = E;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, k_epilogue, red, pitch, n_acc, truncate, amin_mode, amin, matches, ninfo64, prob, L, LR);
}

}  // namespace snpm
