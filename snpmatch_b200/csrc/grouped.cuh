// A2/A3 in "grouped" order — the throughput path of likelihood-weighted scoring (matchGTsAccs, snpmatch.py:74-89, inside the
// chunk loop of Genotyper.genotyper, snpmatch.py:207-233).
//
// The reference adds, per accession, one fp64 weight per matched row: two DADDs per SNP x accession comparison once the
// summation order is fixed, which caps an order-exact kernel at 38 % of the HBM roofline (k_score_segments, score.cuh).
// This kernel does integer work per comparison instead.  exp(-PL/10) takes few distinct values, so the markers of a
// sample are ordered (by the host, once, at parse time: snpm_group_markers) by their weight triple (w_ref, w_het, w_alt).
// Inside a group every row carries the same three weights, hence
//     score[a] = sum over groups g of  w_ref(g)*#{rows of g: d=ref} + w_alt(g)*#{d=alt} + w_het(g)*#{d=het}
// and the per-row work is counting: a thread owns one 32-accession word column, forms the three class planes of a row
// with one LOP3 each and adds them into bit-sliced vertical counters (Harley-Seal carry-save tree, 16 rows per step,
// ~2.6 LOP3 per row and counter).  At a group boundary the counters are read out (8x8 bit transposes -> one byte per
// accession) and folded into the thread's 32 fp64 accumulators with ONE fma per accession and class; classes whose weight
// is exactly 1.0 (the called genotype of a normalised PL triple, and every one-hot weight) never touch fp64: their counts
// go into an integer counter by a bit-sliced add.  The result is split as  score = I + F,  I an exact integer and F a sum
// of non-negative fractional terms, which is what makes the truncated `matches = int(score)` of the reference
// (snpmatch.py:96) reproducible without its summation order: the reference's sum is >= I and < I + F + eps, so
// matches = I + floor(F) unless F lies within the rounding-error bound of an integer k >= 1 — those (sample, accession)
// cells are flagged (k_grouped_finalize) and the sample is re-scored by the order-exact kernel.  fp64 scores agree with the
// reference to a few ulp (tests: rtol 1e-12), integers bit for bit.
//
// Data movement: every thread fetches its own 8-byte column of the rows with cp.async (LDGSTS) into a private slot of a
// 64-row shared-memory ring, 4 blocks of 16 rows in flight, so no barrier or mbarrier sits in the loop and ~150 KB of
// gathers are outstanding per SM.  Measured gather ceiling for this access pattern (scripts/microbench_gather.cu):
// 4.7-4.9 TB/s for rows in panel order, 4.3 TB/s for the weight-grouped order.
#pragma once
#include "common.cuh"
#include "hardcall.cuh"

namespace snpm {

constexpr int GR_THREADS = 128;                       // 3 teams of 36 threads; two CTAs per SM at ~240 registers per thread, no spills
constexpr int GR_MAX_WX = 36;                         // words per team (one 1135-accession row)
constexpr int GR_MAX_TEAMS = 3;
constexpr int GR_BLOCK = 16;                          // rows per step
constexpr int GR_RING = 64;                           // rows of the per-team ring
constexpr int GR_INFLIGHT = GR_RING / GR_BLOCK;
constexpr int GR_LP = 10;                             // planes of a counter (chunk <= 1023 rows)
constexpr int GR_MAX_CHUNK = 1008;

struct GroupArgs {
    const uint64_t *packed;
    int32_t stride;
    const int32_t *pair_db;       // [m] matched local rows, grouped order
    const uint16_t *pair_gid;     // [m] weight-triple id of every matched pair
    const double *table;          // [T, 4] = (w_ref, w_alt, w_het, 0)
    const int32_t *seg_off;       // [S+1]
    const int32_t *mstart;        // [S+1]
    int32_t S;
    int32_t chunk;
    double *part_score;           // [nseg, 32, stride]  fractional part F of the segment; accession 32 w + b at [b][w]
    int32_t *part_int;            // [nseg, 32, stride]  low half: integer part I (matches of weight-1.0 classes); high half: ninfo
    int32_t a_pad;
    int32_t wx;                   // words per team slice
    int32_t spc;                  // teams (segments) per CTA
    int32_t jmax;                 // upper bound of the segments of one sample
};

__device__ __forceinline__ void cp_async8(uint32_t dst_smem, const void *src_gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst_smem), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// bit-sliced counter of 32 lanes, P planes
template <int P>
struct BitCounter {
    uint32_t p[P];
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int k = 0; k < P; ++k) p[k] = 0u;
    }
    __device__ __forceinline__ uint32_t any() const {
        uint32_t o = 0u;
#pragma unroll
        for (int k = 0; k < P; ++k) o |= p[k];
        return o;
    }
    // add sixteen 1-bit planes: 15 carry-save adders arranged as a tree (depth 8 instead of 15, for instruction-level
    // parallelism), then the sixteens ripple upwards
    __device__ __forceinline__ void add16(const uint32_t (&m)[16]) {
        uint32_t c0, c1, c2, c3, c4, c5, c6, c7, s0, s1, s2, s3, s4, t0, t1;
        SNPM_CSA(c0, s0, m[0], m[1], m[2]);
        SNPM_CSA(c1, s1, m[3], m[4], m[5]);
        SNPM_CSA(c2, s2, m[6], m[7], m[8]);
        SNPM_CSA(c3, s3, m[9], m[10], m[11]);
        SNPM_CSA(c4, s4, m[12], m[13], m[14]);
        SNPM_CSA(c5, t0, s0, s1, s2);
        SNPM_CSA(c6, t1, s3, s4, m[15]);
        SNPM_CSA(c7, p[0], t0, t1, p[0]);
        uint32_t d0, d1, d2, d3, u0, u1, u2;
        SNPM_CSA(d0, u0, c0, c1, c2);
        SNPM_CSA(d1, u1, c3, c4, c5);
        SNPM_CSA(d2, u2, c6, c7, p[1]);
        SNPM_CSA(d3, p[1], u0, u1, u2);
        uint32_t e0, e1, v0, s;
        SNPM_CSA(e0, v0, d0, d1, d2);
        SNPM_CSA(e1, p[2], v0, d3, p[2]);
        SNPM_CSA(s, p[3], e0, e1, p[3]);
#pragma unroll
        for (int k = 4; k < P; ++k) {
            const uint32_t c = p[k] & s;
            p[k] ^= s;
            s = c;
        }
    }
    // add a shorter counter (bit-sliced ripple-carry adder)
    template <int Q>
    __device__ __forceinline__ void add_counter(const BitCounter<Q> &o) {
        uint32_t carry = 0u;
#pragma unroll
        for (int k = 0; k < P; ++k) {
            if (k < Q) {
                uint32_t h, l;
                SNPM_CSA(h, l, p[k], o.p[k], carry);
                p[k] = l;
                carry = h;
            } else {
                const uint32_t c = p[k] & carry;
                p[k] ^= carry;
                carry = c;
            }
        }
    }
};

// 8x8 bit transposes of the four byte columns of eight planes: afterwards byte j of r[i] holds, for lane 8j+i, the eight
// plane bits as one number (bit k = plane k)
__device__ __forceinline__ void transpose_planes8(uint32_t (&r)[8]) {
#define SNPM_SWAP(a, b, s, m)                            \
    do {                                                 \
        const uint32_t t__ = (((a) >> (s)) ^ (b)) & (m); \
        (b) ^= t__;                                      \
        (a) ^= t__ << (s);                               \
    } while (0)
    SNPM_SWAP(r[0], r[1], 1, 0x55555555u);
    SNPM_SWAP(r[2], r[3], 1, 0x55555555u);
    SNPM_SWAP(r[4], r[5], 1, 0x55555555u);
    SNPM_SWAP(r[6], r[7], 1, 0x55555555u);
    SNPM_SWAP(r[0], r[2], 2, 0x33333333u);
    SNPM_SWAP(r[1], r[3], 2, 0x33333333u);
    SNPM_SWAP(r[4], r[6], 2, 0x33333333u);
    SNPM_SWAP(r[5], r[7], 2, 0x33333333u);
    SNPM_SWAP(r[0], r[4], 4, 0x0F0F0F0Fu);
    SNPM_SWAP(r[1], r[5], 4, 0x0F0F0F0Fu);
    SNPM_SWAP(r[2], r[6], 4, 0x0F0F0F0Fu);
    SNPM_SWAP(r[3], r[7], 4, 0x0F0F0F0Fu);
#undef SNPM_SWAP
}

// F[lane] += w * count[lane] for the 32 lanes of a class counter
__device__ __forceinline__ void fold_counts(const BitCounter<GR_LP> &c, double w, double (&F)[32]) {
    uint32_t t[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) t[k] = c.p[k];
    transpose_planes8(t);
    if ((c.p[8] | c.p[9]) == 0u) {                // fewer than 256 rows since the last read-out: the common case
#pragma unroll
        for (int i = 0; i < 8; ++i) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int cnt = int((t[i] >> (8 * j)) & 0xffu);
                F[8 * j + i] = fma(w, double(cnt), F[8 * j + i]);
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int b = 8 * j + i;
                const int cnt = int((t[i] >> (8 * j)) & 0xffu) | int(((c.p[8] >> b) & 1u) << 8) | int(((c.p[9] >> b) & 1u) << 9);
                F[b] = fma(w, double(cnt), F[b]);
            }
        }
    }
}

// values of a 10-plane counter for the 32 lanes
__device__ __forceinline__ void counter_values(const BitCounter<GR_LP> &c, int32_t (&v)[32]) {
    uint32_t t[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) t[k] = c.p[k];
    transpose_planes8(t);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int b = 8 * j + i;
            v[b] = int32_t((t[i] >> (8 * j)) & 0xffu) | int32_t(((c.p[8] >> b) & 1u) << 8) | int32_t(((c.p[9] >> b) & 1u) << 9);
        }
    }
}

// shared memory of one team: ring | row numbers | triple ids | per-block weight-change masks
__host__ __device__ __forceinline__ size_t grouped_team_smem(int wx, int chunk) {
    const size_t n_blocks = size_t(chunk + GR_BLOCK - 1) / GR_BLOCK;
    return size_t(GR_RING) * wx * 8 + size_t(chunk) * 4 + ((size_t(chunk) * 2 + 15) & ~size_t(15)) + ((n_blocks * 8 + 15) & ~size_t(15));
}

// grid.x = ceil(S * jmax / teams per CTA), grid.y = word slices.  thread -> (team q, word w); a team scores one segment.
// WX > 0: words per team known at compile time (ring addresses fold into the instructions); WX == 0: a.wx.
template <bool SKIP_HETS, int WX>
__global__ void __launch_bounds__(GR_THREADS, 2) k_score_grouped(const GroupArgs a) {
    extern __shared__ __align__(16) unsigned char gr_smem[];
    const int wx = WX ? WX : a.wx;
    const int spc = a.spc;
    const int q = threadIdx.x / wx, w = threadIdx.x - q * wx;
    // Team slot -> segment, longest first: the tail of every sample's group order holds the rare weight triples (many small
    // groups, i.e. many counter read-outs), so the LAST segments of the samples are the slow ones.  Slots walk the segments
    // by position inside the sample, descending, over all samples: the slow segments start first and the cheap ones fill
    // the end of the grid, instead of one sample's slow tail running alone when everything else has finished.
    const int slot = blockIdx.x * spc + q;
    const int word = blockIdx.y * wx + w;
    int seg = 0, begin = 0, end = 0;
    bool team_ok = false;
    if (q < spc) {
        const int j = a.jmax - 1 - slot / a.S, smp = slot % a.S;
        if (j >= 0 && j < a.seg_off[smp + 1] - a.seg_off[smp]) {
            team_ok = true;
            seg = a.seg_off[smp] + j;
            begin = a.mstart[smp] + j * a.chunk;
            end = min(a.mstart[smp + 1], begin + a.chunk);
        }
    }
    const int n_rows = end - begin;
    const int n_blocks = (n_rows + GR_BLOCK - 1) / GR_BLOCK;
    unsigned char *team = gr_smem + size_t(q < spc ? q : 0) * grouped_team_smem(wx, a.chunk);
    uint64_t *ring = reinterpret_cast<uint64_t *>(team);
    int32_t *s_row = reinterpret_cast<int32_t *>(team + size_t(GR_RING) * wx * 8);
    uint16_t *s_gid = reinterpret_cast<uint16_t *>(team + size_t(GR_RING) * wx * 8 + size_t(a.chunk) * 4);
    // s_chg[b] = three 16-bit masks (ref | alt << 16 | het << 32): bit k set <=> the weight of that class at row 16b+k differs
    // from the row before it (never set for the first row of the segment)
    unsigned long long *s_chg = reinterpret_cast<unsigned long long *>(team + size_t(GR_RING) * wx * 8 + size_t(a.chunk) * 4 +
                                                                       ((size_t(a.chunk) * 2 + 15) & ~size_t(15)));
    if (team_ok) {
        for (int b = w; b < n_blocks; b += wx) s_chg[b] = 0ull;
#pragma unroll 4
        for (int r = w; r < n_rows; r += wx) {
            s_row[r] = __ldg(a.pair_db + begin + r);
            s_gid[r] = __ldg(a.pair_gid + begin + r);
        }
    }
    __syncthreads();
    if (team_ok) {
        for (int r = w + 1; r < n_rows; r += wx) {
            const int g1 = s_gid[r], g0 = s_gid[r - 1];
            if (g1 != g0) {
                const double4 t1 = reinterpret_cast<const double4 *>(a.table)[g1];
                const double4 t0 = reinterpret_cast<const double4 *>(a.table)[g0];
                unsigned long long f = 0ull;
                if (t1.x != t0.x) f |= 1ull << (r & 15);
                if (t1.y != t0.y) f |= 1ull << (16 + (r & 15));
                if (t1.z != t0.z) f |= 1ull << (32 + (r & 15));
                if (f) atomicOr(s_chg + (r >> 4), f);
            }
        }
    }
    __syncthreads();                              // the last CTA-wide barrier: threads may leave from here on
    if (!team_ok || word >= a.stride) return;

    const uint32_t my_ring = smem_u32(ring + w);
    const uint32_t ring_pitch = uint32_t(wx) * 8u;
    const int64_t stride = a.stride;
    const int n_full = n_rows / GR_BLOCK;         // blocks without a ragged end
    // Queue the gathers of block b.  Two neighbouring threads (words 2i, 2i+1: always lanes of one warp) share the work: each
    // copies the 16 bytes that hold BOTH their columns, the even one for rows 0..7 of the block, the odd one for rows 8..15 —
    // 8 LDGSTS.128 per thread instead of 16 LDGSTS.64, which halves the load on the LSU instruction queue.  Full blocks carry
    // no predicates.
    const int odd = w & 1;
    const uint32_t pair_ring = smem_u32(ring + (w & ~1));
    // byte address of a row's pair of columns = base + row * stride_b: one IMAD.WIDE.U32 (32 x 32 -> 64 bit, plus the 64-bit base)
    const unsigned char *pair_col = reinterpret_cast<const unsigned char *>(a.packed + (word & ~1));
    const uint32_t stride_b = uint32_t(a.stride) * 8u;
    // The two partners must see each other's copies: a barrier between them.  __syncwarp with a per-pair mask compiles to
    // MATCH.ANY + REDUX + a divergent branch (11 % of the kernel's stall samples); the whole-warp form is one WARPSYNC.  It is
    // safe here: every live thread of a warp passes the same barriers per block, threads that have left do not count, and the
    // extra coupling (a warp may hold lanes of two teams) only makes one team wait for the other's block.
    constexpr unsigned pair_mask = 0xffffffffu;
    auto issue = [&](int b) {
        const int r0 = b * GR_BLOCK + 8 * odd;
        const uint32_t slot0 = pair_ring + uint32_t(r0 % GR_RING) * ring_pitch;
        if (b < n_full) {
#pragma unroll
            for (int k4 = 0; k4 < GR_BLOCK / 2; k4 += 4) {
                const int4 rr = *reinterpret_cast<const int4 *>(s_row + r0 + k4);
                cp_async16(slot0 + uint32_t(k4 + 0) * ring_pitch, pair_col + (unsigned long long)(uint32_t(rr.x)) * stride_b);
                cp_async16(slot0 + uint32_t(k4 + 1) * ring_pitch, pair_col + (unsigned long long)(uint32_t(rr.y)) * stride_b);
                cp_async16(slot0 + uint32_t(k4 + 2) * ring_pitch, pair_col + (unsigned long long)(uint32_t(rr.z)) * stride_b);
                cp_async16(slot0 + uint32_t(k4 + 3) * ring_pitch, pair_col + (unsigned long long)(uint32_t(rr.w)) * stride_b);
            }
        } else if (b < n_blocks) {
            for (int k = 0; k < GR_BLOCK / 2 && r0 + k < n_rows; ++k) cp_async16(slot0 + uint32_t(k) * ring_pitch, pair_col + (unsigned long long)(uint32_t(s_row[r0 + k])) * stride_b);
        }
        cp_async_commit();                        // always: the wait below counts groups
    };
#pragma unroll
    for (int b = 0; b < GR_INFLIGHT; ++b) issue(b);

    double F[32];
#pragma unroll
    for (int b = 0; b < 32; ++b) F[b] = 0.0;
    BitCounter<GR_LP> c_int, c_ninfo, c_ref, c_alt, c_het;
    c_int.clear();
    c_ninfo.clear();
    c_ref.clear();
    c_alt.clear();
    c_het.clear();
    double w_ref, w_alt, w_het;
    {
        const double4 t = *reinterpret_cast<const double4 *>(a.table + 4 * size_t(s_gid[0]));
        w_ref = t.x;
        w_alt = t.y;
        w_het = t.z;
    }
    // read a class counter out: its counts are informative sites, and matches weighted by `wt`
    auto flush_class = [&](BitCounter<GR_LP> &c, double wt) {
        if (c.any()) {
            c_ninfo.add_counter(c);
            if (wt == 1.0) c_int.add_counter(c);
            else if (wt != 0.0) fold_counts(c, wt, F);
            c.clear();
        }
    };
    // one class: add the block's planes; where the class weight changes inside the block (bit k of `mask`: row k starts a
    // new weight), add the rows piece by piece and read the counter out in between
    auto add_class = [&](BitCounter<GR_LP> &c, double &wt, const uint32_t (&pl)[GR_BLOCK], uint32_t mask, int which, int r0) {
        if (mask == 0u) {
            c.add16(pl);
            return;
        }
        int k0 = 0;
        while (true) {
            const int k1 = mask ? __ffs(mask) - 1 : GR_BLOCK;
            if (k1 > k0) {
                const uint32_t rm = ((1u << k1) - 1u) & ~((1u << k0) - 1u);
                uint32_t m[GR_BLOCK];
#pragma unroll
                for (int k = 0; k < GR_BLOCK; ++k) m[k] = pl[k] & uint32_t(int32_t(rm << (31 - k)) >> 31);
                c.add16(m);
            }
            if (k1 >= GR_BLOCK) break;
            flush_class(c, wt);
            wt = a.table[4 * size_t(s_gid[r0 + k1]) + which];
            mask &= mask - 1u;
            k0 = k1;
        }
    };
    auto score_block = [&](const uint32_t (&lo)[GR_BLOCK], const uint32_t (&hi)[GR_BLOCK], int b) {
        const unsigned long long chg = s_chg[b];
        uint32_t pl[GR_BLOCK];
#pragma unroll
        for (int k = 0; k < GR_BLOCK; ++k) pl[k] = ~(lo[k] | hi[k]);
        add_class(c_ref, w_ref, pl, uint32_t(chg) & 0xffffu, 0, b * GR_BLOCK);
#pragma unroll
        for (int k = 0; k < GR_BLOCK; ++k) pl[k] = lo[k] & ~hi[k];
        add_class(c_alt, w_alt, pl, uint32_t(chg >> 16) & 0xffffu, 1, b * GR_BLOCK);
        if (!SKIP_HETS) {                         // snpmatch.py:78-79: masked hets match nothing and are not informative
#pragma unroll
            for (int k = 0; k < GR_BLOCK; ++k) pl[k] = hi[k] & ~lo[k];
            add_class(c_het, w_het, pl, uint32_t(chg >> 32) & 0xffffu, 2, b * GR_BLOCK);
        }
    };

    for (int b = 0; b < n_full; ++b) {
        cp_async_wait<GR_INFLIGHT - 1>();         // block b has landed: this thread's copies ...
        __syncwarp(pair_mask);                    // ... and its neighbour's
        const uint64_t *slot = ring + size_t((b * GR_BLOCK) % GR_RING) * wx + w;
        uint32_t lo[GR_BLOCK], hi[GR_BLOCK];
#pragma unroll
        for (int k = 0; k < GR_BLOCK; ++k) {
            const uint64_t v = slot[size_t(k) * wx];
            lo[k] = uint32_t(v);
            hi[k] = uint32_t(v >> 32);
        }
        score_block(lo, hi, b);
        __syncwarp(pair_mask);                    // the neighbour has read its half of the block too
        issue(b + GR_INFLIGHT);                   // refill the slots of this block
    }
    if (n_full < n_blocks) {                      // ragged last block: rows past the end read as missing everywhere
        cp_async_wait<0>();
        __syncwarp(pair_mask);
        const int r0 = n_full * GR_BLOCK;
        const uint64_t *slot = ring + size_t(r0 % GR_RING) * wx + w;
        uint32_t lo[GR_BLOCK], hi[GR_BLOCK];
#pragma unroll
        for (int k = 0; k < GR_BLOCK; ++k) {
            uint64_t v = ~0ull;
            if (r0 + k < n_rows) v = slot[size_t(k) * wx];
            lo[k] = uint32_t(v);
            hi[k] = uint32_t(v >> 32);
        }
        score_block(lo, hi, n_full);
    }
    flush_class(c_ref, w_ref);
    flush_class(c_alt, w_alt);
    if (!SKIP_HETS) flush_class(c_het, w_het);

    int32_t vi[32], vn[32];
    counter_values(c_int, vi);
    counter_values(c_ninfo, vn);
    // segment partials are stored lane-major ([seg][lane 0..31][word]): consecutive threads write consecutive addresses
    const int64_t o = int64_t(seg) * a.a_pad + word;
    const int64_t lane_pitch = a.stride;
#pragma unroll
    for (int b = 0; b < 32; ++b) {
        a.part_score[o + b * lane_pitch] = F[b];
        a.part_int[o + b * lane_pitch] = vi[b] | (vn[b] << 16);      // both counts are <= 1008 rows: one word carries them
    }
}

// ---- compaction for the grouped order -------------------------------------------------------------
// as k_scatter_pairs (join.cuh) but the payload of a pair is its weight-triple id
__global__ void __launch_bounds__(JOIN_TILE) k_scatter_pairs_grouped(
        const int32_t *__restrict__ match_row, int64_t n, const int32_t *__restrict__ tile_off, const uint16_t *__restrict__ gid,
        int32_t n_table, int32_t *__restrict__ prefix, int32_t *__restrict__ pair_db, int32_t *__restrict__ pair_s,
        uint16_t *__restrict__ pair_gid, int *status) {
    __shared__ int s_warp[33];
    const int64_t i = int64_t(blockIdx.x) * JOIN_TILE + threadIdx.x;
    const int32_t row = i < n ? match_row[i] : -1;
    const int flag = row >= 0;
    int total;
    const int ex = block_excl_scan(flag, &total, s_warp);
    if (i < n) {
        const int32_t p = tile_off[blockIdx.x] + ex;
        prefix[i] = p;
        if (flag) {
            pair_db[p] = row;
            pair_s[p] = int32_t(i);
            uint16_t g = gid[i];
            if (int32_t(g) >= n_table) {            // an id outside the weight table: reported at wait / fetch (status[4])
                atomicAdd(status + 4, 1);
                g = 0;
            }
            pair_gid[p] = g;
        }
    }
}

// chromosome ids travel as one byte (255 = not in the panel)
__global__ void __launch_bounds__(256) k_expand_chrom(const uint8_t *__restrict__ c8, int64_t n, int32_t *__restrict__ c32) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) c32[i] = c8[i] == 255 ? -1 : int32_t(c8[i]);
}

// chromosome id and position in one word: id << 27 | position (ids 0..30, 31 = not in the panel; positions below 2^27)
__global__ void __launch_bounds__(256) k_expand_packed(const uint32_t *__restrict__ cp, int64_t n, int32_t *__restrict__ c32, int32_t *__restrict__ pos) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) {
        const uint32_t v = cp[i];
        const uint32_t c = v >> 27;
        c32[i] = c == 31u ? -1 : int32_t(c);
        pos[i] = int32_t(v & 0x7ffffffu);
    }
}

// weight-triple ids travel run-length coded (markers are ordered by id inside a sample: ~70 markers per run): run r covers
// markers [run_end[r-1], run_end[r]) and carries run_gid[r].  One warp per run, lanes stride over its markers (coalesced
// 2-byte stores).  Ends that do not ascend or leave [0, n] are counted in status_bad (reported by the upload).
__global__ void __launch_bounds__(256) k_expand_runs(const uint32_t *__restrict__ run_end, const uint16_t *__restrict__ run_gid, int32_t n_runs,
                                                     int64_t n, uint16_t *__restrict__ gid, int *__restrict__ status_bad) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (r >= n_runs) return;
    const int64_t begin = r ? int64_t(__ldg(run_end + r - 1)) : 0, end = int64_t(__ldg(run_end + r));
    if (end <= begin || end > n) {
        if (lane == 0) atomicAdd(status_bad, 1);
        return;
    }
    const uint16_t g = __ldg(run_gid + r);
    for (int64_t i = begin + lane; i < end; i += 32) gid[i] = g;
}

// ---- combine: totals of the segment partials of one sample ----------------------------------------------
// red row layout in grouped mode [3*n_acc + 2]: F[n_acc] | ninfo[n_acc] | matched pairs | overflow, then y>n violations | I[n_acc]
// (the first 2*n_acc + 2 entries are laid out as in k_combine; k_grouped_finalize turns F into the score in place).  Slot
// 2*n_acc + 1 carries the grouping's overflow flag of this shard (coded batches; 0 otherwise) until k_grouped_finalize has read
// it; k_epilogue then stores the y>n count there.  The flag travels through the cross-GPU sum with the totals, so the rank that
// finishes a sample sees an overflow of any rank.
constexpr int CG_PARTS = 8;           // warps of a CTA = contiguous parts of a sample's segments, summed in part order at the end
__global__ void __launch_bounds__(32 * CG_PARTS) k_combine_grouped(const double *__restrict__ part_score, const int32_t *__restrict__ part_int,
                                                                   int32_t a_pad, int32_t stride, int32_t n_acc,
                                                                   const int32_t *__restrict__ seg_off, const int32_t *__restrict__ mstart,
                                                                   const int *__restrict__ overflow, double *__restrict__ red) {
    // thread (x, y) -> position p = 32 * blockIdx.x + x of the lane-major segment partials ([lane b][word w], p = b * stride + w:
    // coalesced reads), part y of the segments.  The order of the fp64 adds is fixed (segments in order inside a part, parts in
    // order), so results are reproducible run to run.
    __shared__ double s_f[CG_PARTS][32];
    __shared__ long long s_i[CG_PARTS][32], s_n[CG_PARTS][32];
    const int s = blockIdx.y;
    const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
    const int p = blockIdx.x * 32 + x;
    const int j0 = seg_off[s], j1 = seg_off[s + 1];
    const int per = (j1 - j0 + CG_PARTS - 1) / CG_PARTS;
    const int ja = min(j1, j0 + y * per), jb = min(j1, ja + per);
    double f = 0.0;
    long long ii = 0, ni = 0;
    if (p < a_pad) {
        constexpr int CB = 8;
        int j = ja;
        for (; j + CB <= jb; j += CB) {
            double v[CB];
            int32_t ci[CB];
#pragma unroll
            for (int k = 0; k < CB; ++k) {
                v[k] = __ldg(part_score + int64_t(j + k) * a_pad + p);
                ci[k] = __ldg(part_int + int64_t(j + k) * a_pad + p);
            }
#pragma unroll
            for (int k = 0; k < CB; ++k) {
                f += v[k];
                ii += ci[k] & 0xffff;
                ni += ci[k] >> 16;
            }
        }
        for (; j < jb; ++j) {
            f += part_score[int64_t(j) * a_pad + p];
            const int32_t c = part_int[int64_t(j) * a_pad + p];
            ii += c & 0xffff;
            ni += c >> 16;
        }
    }
    s_f[y][x] = f;
    s_i[y][x] = ii;
    s_n[y][x] = ni;
    __syncthreads();
    double *row = red + int64_t(s) * (3 * int64_t(n_acc) + 2);
    if (y == 0) {
        const int b = p / stride, w = p - b * stride;
        const int acc = 32 * w + b;
        if (p < a_pad && acc < n_acc) {
#pragma unroll
            for (int k = 1; k < CG_PARTS; ++k) {
                f += s_f[k][x];
                ii += s_i[k][x];
                ni += s_n[k][x];
            }
            row[acc] = f;
            row[n_acc + acc] = double(ni);
            row[2 * n_acc + 2 + acc] = double(ii);
        }
        if (p == 0) {
            row[2 * n_acc] = double(mstart[s + 1] - mstart[s]);
            row[2 * n_acc + 1] = (overflow != nullptr && overflow[s]) ? 1.0 : 0.0;
        }
    }
}

// ---- one-shot reduce over peer memory (SURVEY 8e) --------------------------------------------------------
// The cross-GPU sum of the per-sample totals with no collective library on the path: every rank's reduce buffer is mapped
// into every other rank (CUDA IPC over NVLink / NVSwitch).  k_reduce_peers is barrier + reduce-scatter in one kernel:
//   arrive  block 0 publishes "my totals of step t are complete" into every peer's flag block (st.release.sys; the totals were
//           written by the kernels before this one on the stream),
//   wait    every block spins (ld.acquire.sys) until all ranks have arrived at step t,
//   reduce  the rows of THIS rank's share of the samples are pulled from all ranks with 16-byte loads and summed in rank
//           order (every rank would compute the same bits) into the own buffer; nothing is pushed, and the rows a rank
//           writes are never read by a peer,
//   done    the last block publishes "I have pulled my rows of step t": k_wait_peers_done at the head of the next run keeps
//           the next totals from overwriting rows a peer is still reading.
// Flags are step counters (monotonic, compared with wrap-around), so a rank that is one step ahead disturbs nobody.  A spin
// gives up after thirty seconds and raises status[5] instead of hanging the GPU.  Works for both row layouts (2A+2, 3A+2).
constexpr int PR_MAX_WORLD = 16;
constexpr int PR_FLAG_BYTES = 4096;      // tail of the exported allocation: arrive[16] at u32 0.., done[16] at u32 64..
constexpr int PR_DONE_OFF = 64;
struct PeerPtrs {
    const double *p[PR_MAX_WORLD];
    uint32_t *flags[PR_MAX_WORLD];
};
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// true when *f has reached `want` (step counters: signed distance); false after ~30 s (a rank that died, not one that is late)
__device__ __forceinline__ bool spin_until(const uint32_t *f, uint32_t want) {
    const unsigned long long t0 = global_timer_ns();
    while (int32_t(ld_acquire_sys_u32(f) - want) < 0) {
        __nanosleep(40);
        if (global_timer_ns() - t0 > 30000000000ull) return false;
    }
    return true;
}
template <typename V>
__device__ __forceinline__ V ld_peer(const double *p);
template <>
__device__ __forceinline__ double ld_peer<double>(const double *p) {
    double v;
    asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
template <>
__device__ __forceinline__ double2 ld_peer<double2>(const double *p) {
    double2 v;
    asm volatile("ld.volatile.global.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p) : "memory");
    return v;
}

template <typename V>
__global__ void __launch_bounds__(256) k_reduce_peers(const PeerPtrs peers, int32_t world, int32_t rank, uint32_t step, int64_t first, int64_t count,
                                                      double *__restrict__ own, int *status) {
    // V = double2 when `first` and `count` (in doubles) are even: 16-byte peer loads; else double
    constexpr int W = int(sizeof(V) / sizeof(double));
    __shared__ int s_last;
    if (blockIdx.x == 0 && threadIdx.x < world) {
        __threadfence_system();
        st_release_sys_u32(peers.flags[threadIdx.x] + rank, step);                     // arrive
    }
    const unsigned long long t_wait = global_timer_ns();
    if (threadIdx.x < world && !spin_until(peers.flags[rank] + threadIdx.x, step)) atomicExch(status + 5, 1);   // wait
    __syncthreads();
    if (blockIdx.x == 0 && threadIdx.x == 0) status[7] = int(global_timer_ns() - t_wait);       // ns spent waiting for the slowest rank
    const int64_t nv = count / W;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < nv; i += int64_t(gridDim.x) * blockDim.x) {
        const int64_t o = first + W * i;
        double acc[W];
#pragma unroll
        for (int k = 0; k < W; ++k) acc[k] = 0.0;
#pragma unroll 4
        for (int r = 0; r < world; ++r) {
            const V v = ld_peer<V>(peers.p[r] + o);
            const double *e = reinterpret_cast<const double *>(&v);
#pragma unroll
            for (int k = 0; k < W; ++k) acc[k] += e[k];
        }
#pragma unroll
        for (int k = 0; k < W; ++k) own[o + k] = acc[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const int prev = atomicAdd(status + 6, 1);                                     // blocks that have pulled their part
        s_last = prev == int(gridDim.x) - 1;
        if (s_last) status[6] = 0;
    }
    __syncthreads();
    if (s_last && threadIdx.x < world) st_release_sys_u32(peers.flags[threadIdx.x] + PR_DONE_OFF + rank, step);   // done
}

// head of the next run: every peer has pulled its rows of step `want`
__global__ void __launch_bounds__(32) k_wait_peers_done(const uint32_t *own_flags, int32_t world, uint32_t want, int *status) {
    if (threadIdx.x < world && !spin_until(own_flags + PR_DONE_OFF + threadIdx.x, want)) atomicExch(status + 5, 1);
}

// score = I + F with the reference's truncation made explicit: matches = I + floor(F) (see the header).  The score is
// stored so that the epilogue's int(score) gives exactly that, and cells whose F lies within the summation-error bound of
// an integer k >= 1 are counted in guard[s]: for them the reference's own rounding decides, so the caller re-scores the
// sample in reference order.  Runs after the cross-GPU reduce, on totals.
__global__ void __launch_bounds__(256) k_grouped_finalize(double *__restrict__ red, int32_t n_acc, int32_t *__restrict__ guard) {
    const int s = blockIdx.y;
    const int acc = blockIdx.x * blockDim.x + threadIdx.x;
    if (acc >= n_acc) return;
    double *row = red + int64_t(s) * (3 * int64_t(n_acc) + 2);
    // a sample whose weight triples did not fit the dense ids of the device grouping (group_sort.cuh) on some shard was scored
    // with ids folded together: flag it like a guard hit, the caller re-scores it in reference order.  The flag is the sum
    // over the shards of slot 2*n_acc + 1 (k_combine_grouped), not this rank's own.
    if (acc == 0 && row[2 * n_acc + 1] > 0.0) atomicAdd(guard + s, 1);
    const double f = row[acc], ii = row[2 * n_acc + 2 + acc], m = row[2 * n_acc];
    // |reference - exact| <= (1000 + 2 + m/1000) u (I+F) for its chunked sequential sums (SURVEY A.2), the same bound holds
    // for the sums above; u = 2^-53.  Factor 4 covers both plus slack.
    const double depth = 1010.0 + m * (1.0 / 500.0);
    const double g = 4.0 * depth * 1.1102230246251565e-16 * (ii + f + 1.0);
    const double k = rint(f);
    if (k >= 1.0 && fabs(f - k) <= g) atomicAdd(guard + s, 1);
    const double want = ii + floor(f);
    double v = ii + f;
    if (floor(v) != want) v = __longlong_as_double(__double_as_longlong(want + 1.0) - 1);   // largest double below want + 1
    row[acc] = v;
}

}  // namespace snpm
