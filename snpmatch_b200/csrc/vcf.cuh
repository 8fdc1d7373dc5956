// Multi-sample VCF text -> every sample's called genotypes (`inbred --samples_vcf`, `cross --samples_vcf`).
//
// The host streams the text after the #CHROM line in chunks of whole lines; per chunk (snpm_vcf_parse):
//   1. line index: k_vcf_line_count + scan + k_vcf_line_starts find the line starts with Python's universal-newline rule
//      (\n, \r\n and a lone \r end a line: the host parsers read in text mode), flag a non-ASCII byte anywhere in the chunk and
//      count `##INFO=<ID=DP,` lines;
//   2. k_vcf_records, one warp per line: tab positions from ballots, POS, INFO DP with read_vcf_minimal's regex semantics
//      (first (?:^|;)DP= with a non-empty value), the GT / PL indices of FORMAT, the number of sample fields;
//   3. k_vcf_cells, one warp per record, lanes over its cells: the GT and PL subfields of every cell of samples 0..S-1, the
//      GT rendered as two allele codes, the first three PLs; and whether CHROM equals the previous record's;
//   4. a record whose result the device cannot vouch for is flagged VCF_FALLBACK (the host re-parses it with the Python code):
//      POS / DP that are not 1-9 plain digits, a PL value that is not '.', empty or 1-9 digits, an allele that is not '.',
//      empty or 1-2 digits, GT or PL twice in FORMAT, a non-ASCII byte in the fixed fields;
//   5. k_vcf_count_called + scan + k_vcf_write_called: per sample, the called cells (rendered GT != ./.) of the records that
//      did not fall back, in record order (sample-major CSR).  The dense [cells] arrays stay on the device.
//
// `makedb --no_csv` (snpm_vcf_parse_gt_packed) reuses the line index and takes makedb's rules instead of steps 2-5:
//   2'. k_vcf_records<true>: tab positions, POS, the index of the FIRST GT in FORMAT (vcf_to_csv's keys.index), the number of
//       sample fields; only a POS that is not 1-9 plain digits flags a record (the host converts that POS text);
//   3'. scan of the records whose sample-field count equals the header's: each one's row in the chunk's packed panel;
//   4'. k_vcf_gt_packed, one warp per record: lane j classifies cell 32 w + j by the exact GT text of vcf_to_csv's _GT_CODE and
//       two ballots write packed word w in k_pack_int8's layout (padding lanes and words missing); calls that are no _GT_CODE
//       string are counted with one atomic per warp.  No per-cell array exists.
//
// `genotype_cross --gpu_parse` (snpm_vcf_parse_gt_codes) reuses the line index and 2' with a row for every record:
//   2''. k_vcf_records_all: k_vcf_records<true>'s fields, ncell = 1 for every record whatever its number of sample fields;
//   3''. scan of the records: each one's row of the chunk's [rows, n_samples] int8 codes;
//   4''. k_vcf_gt_codes, one warp per record: lane j writes the code read_vcf_samples + parseGT give cell 32 w + j (1 for 1/1, 2
//        for 0/1 and 1/0, -1 for ./., a missing GT and a cell past the record's sample fields, 0 otherwise).  The rule is total:
//        no cell falls back to the host.
#pragma once
#include "common.cuh"

namespace snpm {

constexpr int VCF_TILE = 4096;          // bytes per CTA of the line index: 256 threads x 16 bytes
constexpr int VCF_SCAN_ITEMS = 4096;    // elements per CTA of vcf_scan: 1024 threads x 4
constexpr int VCF_CTILE = 128;          // lines per tile of the per-sample compaction
constexpr int VCF_NCODE = 111;          // allele codes: 0 '.', 1 + d for the digit d, 11 + 10 x + y for the two digits xy

// line flags
enum { VCF_REC = 1, VCF_FALLBACK = 2, VCF_HAS_PL = 4, VCF_NEW_CHROM = 8 };

template <int NT>
__device__ __forceinline__ int vcf_block_excl_scan(int v, int *sm, int &total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) sm[w] = x;
    __syncthreads();
    if (w == 0) {
        int t = lane < NT / 32 ? sm[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, t, o);
            if (lane >= o) t += y;
        }
        if (lane < NT / 32) sm[lane] = t;
    }
    __syncthreads();
    total = sm[NT / 32 - 1];
    const int base = w ? sm[w - 1] : 0;
    __syncthreads();
    return base + x - v;
}

// ---- exclusive scan of int32 counts: out[0..n] with out[n] = total ------------------------------------------------------
__global__ void __launch_bounds__(1024) k_vcf_scan_reduce(const int *__restrict__ in, int64_t n, int *__restrict__ bsum) {
    __shared__ int sm[32];
    const int64_t base = int64_t(blockIdx.x) * VCF_SCAN_ITEMS + threadIdx.x * 4;
    int v = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (base + k < n) v += in[base + k];
    int total;
    vcf_block_excl_scan<1024>(v, sm, total);
    if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024) k_vcf_scan_top(int *bsum, int nb) {
    __shared__ int sm[32];
    int carry = 0;
    for (int b0 = 0; b0 < nb; b0 += 1024) {
        const int i = b0 + threadIdx.x;
        int total;
        const int ex = vcf_block_excl_scan<1024>(i < nb ? bsum[i] : 0, sm, total);
        if (i < nb) bsum[i] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) bsum[nb] = carry;
}

__global__ void __launch_bounds__(1024) k_vcf_scan_apply(const int *__restrict__ in, int64_t n, const int *__restrict__ bsum,
                                                         int *__restrict__ out) {
    __shared__ int sm[32];
    const int64_t base = int64_t(blockIdx.x) * VCF_SCAN_ITEMS + threadIdx.x * 4;
    int v[4], s = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        v[k] = base + k < n ? in[base + k] : 0;
        s += v[k];
    }
    int total;
    int ex = vcf_block_excl_scan<1024>(s, sm, total) + bsum[blockIdx.x];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (base + k < n) out[base + k] = ex;
        ex += v[k];
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) out[n] = bsum[gridDim.x];
}

// ---- 1. line index ---------------------------------------------------------------------------------------------------------
// byte p ends a line: '\n', or '\r' not followed by '\n' (the chunk's last byte always ends one)
__device__ __forceinline__ bool vcf_ends_line(uint8_t c, uint8_t next, bool last) {
    return c == '\n' || (c == '\r' && (last || next != '\n'));
}

// the 16 bytes of thread `threadIdx.x` of the tile, and the byte after them
__device__ __forceinline__ void vcf_load16(const uint8_t *__restrict__ t, int64_t n, int64_t p0, uint8_t (&b)[17]) {
    if (p0 + 16 <= n) {
        const uint4 v = *reinterpret_cast<const uint4 *>(t + p0);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 16; ++k) b[k] = uint8_t(w[k >> 2] >> (8 * (k & 3)));
    } else {
#pragma unroll
        for (int k = 0; k < 16; ++k) b[k] = p0 + k < n ? t[p0 + k] : 0;
    }
    b[16] = p0 + 16 < n ? t[p0 + 16] : 0;
}

__global__ void __launch_bounds__(256) k_vcf_line_count(const uint8_t *__restrict__ t, int64_t n, int *__restrict__ tile_cnt,
                                                        int *__restrict__ chunk_flags) {
    __shared__ int sm[8];
    const int64_t p0 = int64_t(blockIdx.x) * VCF_TILE + threadIdx.x * 16;
    uint8_t b[17];
    vcf_load16(t, n, p0, b);
    int c = 0;
    bool high = false;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        if (p0 + k >= n) continue;
        c += vcf_ends_line(b[k], b[k + 1], p0 + k + 1 >= n);
        high |= b[k] >= 0x80;
    }
    int total;
    vcf_block_excl_scan<256>(c, sm, total);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = total;
    if (__syncthreads_or(high) && threadIdx.x == 0) atomicOr(chunk_flags, 1);
}

__device__ __forceinline__ bool vcf_info_dp_line(const uint8_t *__restrict__ t, int64_t n, int64_t q) {
    const char *key = "##INFO=<ID=DP,";
    if (q + 14 > n) return false;
    for (int i = 0; i < 14; ++i)
        if (t[q + i] != uint8_t(key[i])) return false;
    return true;
}

// starts[0] = 0, starts[1 + k] = one past the k-th line end; chunk_flags[1] counts `##INFO=<ID=DP,` lines
__global__ void __launch_bounds__(256) k_vcf_line_starts(const uint8_t *__restrict__ t, int64_t n, const int *__restrict__ tile_off,
                                                         int *__restrict__ starts, int *__restrict__ chunk_flags) {
    __shared__ int sm[8];
    const int64_t p0 = int64_t(blockIdx.x) * VCF_TILE + threadIdx.x * 16;
    uint8_t b[17];
    vcf_load16(t, n, p0, b);
    int c = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k)
        if (p0 + k < n) c += vcf_ends_line(b[k], b[k + 1], p0 + k + 1 >= n);
    int total;
    int o = tile_off[blockIdx.x] + vcf_block_excl_scan<256>(c, sm, total);
    int info = 0;
    if (p0 == 0) {
        starts[0] = 0;
        info += vcf_info_dp_line(t, n, 0);
    }
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        if (p0 + k < n && vcf_ends_line(b[k], b[k + 1], p0 + k + 1 >= n)) {
            starts[1 + o++] = int(p0 + k + 1);
            info += vcf_info_dp_line(t, n, p0 + k + 1);
        }
    }
    if (info) atomicAdd(chunk_flags + 1, info);
}

// ---- 2. fixed fields, one warp per line -----------------------------------------------------------------------------------
__device__ __forceinline__ int vcf_line_end(const uint8_t *__restrict__ t, int s, int e) {
    if (e > s && t[e - 1] == '\n') {
        --e;
        if (e > s && t[e - 1] == '\r') --e;
    } else if (e > s && t[e - 1] == '\r') {
        --e;
    }
    return e;
}

// [a, b) as 1-9 plain decimal digits
__device__ __forceinline__ bool vcf_uint9(const uint8_t *__restrict__ t, int a, int b, int &v) {
    if (b - a < 1 || b - a > 9) return false;
    int x = 0;
    for (int i = a; i < b; ++i) {
        const int d = int(t[i]) - '0';
        if (d < 0 || d > 9) return false;
        x = x * 10 + d;
    }
    v = x;
    return true;
}

struct VcfLines {
    int *flags, *nsf, *pos, *dp, *chrom_len, *samp0, *fmt, *ncell;
};

// MAKEDB: vcf_to_csv's rules (first GT of FORMAT, only POS flags a record, ncell = 1 for a record of exactly n_samples sample
// fields: the rows of the packed panel); otherwise read_vcf_minimal's (see the top of the file).  ALL_ROWS (with MAKEDB): ncell = 1
// for every record, whatever its number of sample fields (the rows of k_vcf_gt_codes).
template <bool MAKEDB, bool ALL_ROWS>
__device__ __forceinline__ void vcf_records(const uint8_t *__restrict__ t, const int *__restrict__ starts, int n_lines, int n_samples,
                                            VcfLines o) {
    const int lane = threadIdx.x & 31;
    const int n_warps = int(gridDim.x) * (blockDim.x >> 5);
    for (int L = int(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); L < n_lines; L += n_warps) {
        const int s = starts[L], e = vcf_line_end(t, s, starts[L + 1]);
        int flags = 0, nsf = 0, pos = 0, dp = -1, clen = 0, samp0 = 0, fmt = 0;
        if (e > s && t[s] != '#') {
            int ntab = 0, tab = -1, first_high = e;
            for (int base = s; base < e; base += 32) {
                const int p = base + lane;
                const uint8_t c = p < e ? t[p] : 0;
                const unsigned m = __ballot_sync(0xffffffffu, c == '\t');
                if constexpr (!MAKEDB) {
                    const unsigned hm = __ballot_sync(0xffffffffu, c >= 0x80);
                    if (hm && first_high == e) first_high = base + __ffs(hm) - 1;
                }
                const int j = lane - ntab;                    // lane k < 9 keeps the position of tab k
                if (lane < 9 && j >= 0 && j < __popc(m)) tab = base + int(__fns(m, 0, j + 1));
                ntab += __popc(m);
            }
            if (ntab >= 9) {
                int tb[9];
#pragma unroll
                for (int k = 0; k < 9; ++k) tb[k] = __shfl_sync(0xffffffffu, tab, k);
                flags = VCF_REC;
                nsf = ntab - 8;
                clen = tb[0] - s;
                samp0 = tb[8] + 1;
                if constexpr (MAKEDB) {
                    if (lane == 0) {
                        if (!vcf_uint9(t, tb[0] + 1, tb[1], pos)) flags |= VCF_FALLBACK;
                        // FORMAT: the index of the first GT (1-based, 0 = absent)
                        int k = 0, ks = tb[7] + 1, gi = 0;
                        for (int p = tb[7] + 1; p <= tb[8] && !gi; ++p) {
                            if (p < tb[8] && t[p] != ':') continue;
                            if (p - ks == 2 && t[ks] == 'G' && t[ks + 1] == 'T') gi = k + 1;
                            ++k;
                            ks = p + 1;
                        }
                        fmt = gi;
                    }
                } else {
                    bool fb = first_high < tb[8];
                    // INFO: the first (?:^|;)DP= followed by a non-empty value
                    const int i0 = tb[6] + 1, i1 = tb[7];
                    int found = -1;
                    for (int base = i0; base < i1 && found < 0; base += 32) {
                        const int p = base + lane;
                        const bool cand = p + 3 < i1 && (p == i0 || t[p - 1] == ';') && t[p] == 'D' && t[p + 1] == 'P' && t[p + 2] == '=' &&
                                          t[p + 3] != ';';
                        const unsigned m = __ballot_sync(0xffffffffu, cand);
                        if (m) found = base + __ffs(m) - 1;
                    }
                    if (lane == 0) {
                        fb |= !vcf_uint9(t, tb[0] + 1, tb[1], pos);
                        if (found >= 0) {
                            int v = found + 3;
                            while (v < i1 && t[v] != ';' && v - found < 13) ++v;      // 10 characters are already too many
                            fb |= !vcf_uint9(t, found + 3, v, dp);
                        }
                        // FORMAT: indices of GT and PL (1-based, 0 = absent), either one twice falls back (dict(zip()) keeps the last)
                        int k = 0, ks = tb[7] + 1, gi = 0, pi = 0;
                        for (int p = tb[7] + 1; p <= tb[8]; ++p) {
                            if (p < tb[8] && t[p] != ':') continue;
                            if (p - ks == 2 && t[ks] == 'G' && t[ks + 1] == 'T') {
                                fb |= gi != 0;
                                gi = k + 1;
                            } else if (p - ks == 2 && t[ks] == 'P' && t[ks + 1] == 'L') {
                                fb |= pi != 0;
                                pi = k + 1;
                            }
                            ++k;
                            ks = p + 1;
                        }
                        fb |= k >= 0xffff;
                        fmt = (gi & 0xffff) | (pi << 16);
                        if (pi) flags |= VCF_HAS_PL;
                        if (fb) flags |= VCF_FALLBACK;
                    }
                }
                flags = __shfl_sync(0xffffffffu, flags, 0);
            }
        }
        if (lane == 0) {
            o.flags[L] = flags;
            o.nsf[L] = nsf;
            o.pos[L] = pos;
            o.dp[L] = dp;
            o.chrom_len[L] = clen;
            o.samp0[L] = samp0;
            o.fmt[L] = fmt;
            if constexpr (ALL_ROWS)
                o.ncell[L] = flags & VCF_REC;
            else if constexpr (MAKEDB)
                o.ncell[L] = (flags & VCF_REC) && nsf == n_samples;
            else
                o.ncell[L] = (flags & (VCF_REC | VCF_FALLBACK)) == VCF_REC ? min(nsf, n_samples) : 0;
        }
    }
}

template <bool MAKEDB>
__global__ void __launch_bounds__(256) k_vcf_records(const uint8_t *__restrict__ t, const int *__restrict__ starts, int n_lines,
                                                     int n_samples, VcfLines o) {
    vcf_records<MAKEDB, false>(t, starts, n_lines, n_samples, o);
}

// makedb's rules, a row for every record
__global__ void __launch_bounds__(256) k_vcf_records_all(const uint8_t *__restrict__ t, const int *__restrict__ starts, int n_lines,
                                                         VcfLines o) {
    vcf_records<true, true>(t, starts, n_lines, 0, o);
}

// ---- 3. cells, one warp per record, lanes over its cells --------------------------------------------------------------------
// allele [a, b): '.' or empty -> 0, one digit d -> 1 + d, two digits xy -> 11 + 10x + y; anything else is not representable
__device__ __forceinline__ bool vcf_allele(const uint8_t *__restrict__ t, int a, int b, int &code) {
    const int len = b - a;
    if (len == 0) { code = 0; return true; }
    const int d0 = int(t[a]) - '0';
    if (len == 1) {
        if (t[a] == '.') { code = 0; return true; }
        if (d0 < 0 || d0 > 9) return false;
        code = 1 + d0;
        return true;
    }
    if (len != 2) return false;
    const int d1 = int(t[a + 1]) - '0';
    if (d0 < 0 || d0 > 9 || d1 < 0 || d1 > 9) return false;
    code = 11 + 10 * d0 + d1;
    return true;
}

// one cell [a, b) with GT subfield gi and PL subfield pi (0-based, -1 absent): rendered GT class a1 * 111 + a2, PLs (-1 missing).
// Returns false when the device cannot reproduce read_vcf_minimal on it.
__device__ bool vcf_cell(const uint8_t *__restrict__ t, int a, int b, int gi, int pi, uint16_t &cls, int (&pl)[3]) {
    int g0 = -1, g1 = -1, q0 = -1, q1 = -1;
    const int last = max(gi, pi);
    for (int p = a, k = 0, fs = a; p <= b && k <= last; ++p) {
        if (p < b && t[p] != ':') continue;
        if (k == gi) { g0 = fs; g1 = p; }
        if (k == pi) { q0 = fs; q1 = p; }
        ++k;
        fs = p + 1;
    }
    bool ok = true;
    int al[2] = {0, 0};
    if (g0 >= 0) {
        for (int p = g0, n = 0, st = g0; p <= g1 && n < 2; ++p) {
            if (p < g1 && t[p] != '/' && t[p] != '|') continue;
            ok &= vcf_allele(t, st, p, al[n]);
            ++n;
            st = p + 1;
        }
    }
    cls = uint16_t(al[0] * VCF_NCODE + al[1]);
    pl[0] = pl[1] = pl[2] = -1;
    if (q0 >= 0) {
        for (int p = q0, n = 0, st = q0; p <= q1 && n < 3; ++p) {
            if (p < q1 && t[p] != ',') continue;
            if (!(p == st || (p == st + 1 && t[st] == '.'))) ok &= vcf_uint9(t, st, p, pl[n]);
            ++n;
            st = p + 1;
        }
    }
    return ok;
}

__global__ void __launch_bounds__(256) k_vcf_cells(const uint8_t *__restrict__ t, const int *__restrict__ starts, int n_lines,
                                                   VcfLines o, const int *__restrict__ cell_off, uint16_t *__restrict__ cls,
                                                   int *__restrict__ pl) {
    const int lane = threadIdx.x & 31;
    const int n_warps = int(gridDim.x) * (blockDim.x >> 5);
    for (int L = int(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); L < n_lines; L += n_warps) {
        const int fl = o.flags[L];
        if (!(fl & VCF_REC)) continue;
        const int s = starts[L];
        // CHROM equal to the previous line's, which is a record: the host re-uses that record's name
        const int clen = o.chrom_len[L];
        bool same = L > 0 && (o.flags[L - 1] & VCF_REC) && o.chrom_len[L - 1] == clen;
        if (same) {
            const int ps = starts[L - 1];
            for (int b0 = 0; b0 < clen && same; b0 += 32) {
                const int i = b0 + lane;
                same = __all_sync(0xffffffffu, i >= clen || t[ps + i] == t[s + i]);
            }
        }
        int add = same ? 0 : VCF_NEW_CHROM;
        const int nc = o.ncell[L];
        if (nc > 0) {
            const int e = vcf_line_end(t, s, starts[L + 1]);
            const int gi = (o.fmt[L] & 0xffff) - 1, pi = (o.fmt[L] >> 16) - 1;
            const int off = cell_off[L];
            int cell = 0, cur = o.samp0[L], my_a = 0, my_b = 0;
            bool ok = true;
            for (int base = cur; base < e && cell < nc; base += 32) {
                const int p = base + lane;
                unsigned m = __ballot_sync(0xffffffffu, p < e && t[p] == '\t');
                while (m && cell < nc) {
                    const int tp = base + __ffs(m) - 1;
                    m &= m - 1;
                    if (lane == (cell & 31)) { my_a = cur; my_b = tp; }
                    cur = tp + 1;
                    if ((++cell & 31) == 0) {
                        uint16_t c;
                        int v[3];
                        ok &= vcf_cell(t, my_a, my_b, gi, pi, c, v);
                        const int64_t q = off + cell - 32 + lane;
                        cls[q] = c;
                        pl[3 * q] = v[0]; pl[3 * q + 1] = v[1]; pl[3 * q + 2] = v[2];
                    }
                }
            }
            bool closed_by_end = false;
            if (cell < nc) {                                   // the line end closes the last sample field
                if (lane == (cell & 31)) { my_a = cur; my_b = e; }
                ++cell;
                closed_by_end = true;
            }
            // the cells not parsed yet: the last partial batch, or a full one completed by the line end
            const int pending = (cell & 31) ? (cell & 31) : (closed_by_end ? 32 : 0);
            if (lane < pending) {
                uint16_t c;
                int v[3];
                ok &= vcf_cell(t, my_a, my_b, gi, pi, c, v);
                const int64_t q = off + cell - pending + lane;
                cls[q] = c;
                pl[3 * q] = v[0]; pl[3 * q + 1] = v[1]; pl[3 * q + 2] = v[2];
            }
            if (!__all_sync(0xffffffffu, ok)) add |= VCF_FALLBACK;
        }
        if (lane == 0 && add) atomicOr(o.flags + L, add);
    }
}

// ---- 5. per-sample compaction of the called cells ---------------------------------------------------------------------------
__device__ __forceinline__ bool vcf_called(const VcfLines &o, const int *__restrict__ cell_off, const uint16_t *__restrict__ cls,
                                           int L, int smp) {
    return (o.flags[L] & (VCF_REC | VCF_FALLBACK)) == VCF_REC && smp < o.ncell[L] && cls[cell_off[L] + smp] != 0;
}

// cnt[s * n_ctiles + tile] = called cells of sample s in the tile's lines
__global__ void __launch_bounds__(128) k_vcf_count_called(int n_lines, int n_samples, VcfLines o, const int *__restrict__ cell_off,
                                                          const uint16_t *__restrict__ cls, int *__restrict__ cnt) {
    const int smp = int(blockIdx.y) * 128 + threadIdx.x;
    if (smp >= n_samples) return;
    const int L0 = int(blockIdx.x) * VCF_CTILE, L1 = min(L0 + VCF_CTILE, n_lines);
    int c = 0;
    for (int L = L0; L < L1; ++L) c += vcf_called(o, cell_off, cls, L, smp);
    cnt[int64_t(smp) * gridDim.x + blockIdx.x] = c;
}

__global__ void __launch_bounds__(128) k_vcf_write_called(int n_lines, int n_samples, VcfLines o, const int *__restrict__ cell_off,
                                                          const uint16_t *__restrict__ cls, const int *__restrict__ pl,
                                                          const int *__restrict__ coff, int *__restrict__ out_line,
                                                          uint16_t *__restrict__ out_cls, int *__restrict__ out_pl) {
    const int smp = int(blockIdx.y) * 128 + threadIdx.x;
    if (smp >= n_samples) return;
    const int L0 = int(blockIdx.x) * VCF_CTILE, L1 = min(L0 + VCF_CTILE, n_lines);
    int w = coff[int64_t(smp) * gridDim.x + blockIdx.x];
    for (int L = L0; L < L1; ++L) {
        if (!vcf_called(o, cell_off, cls, L, smp)) continue;
        const int64_t q = cell_off[L] + smp;
        out_line[w] = L;
        out_cls[w] = cls[q];
        out_pl[3 * int64_t(w)] = pl[3 * q];
        out_pl[3 * int64_t(w) + 1] = pl[3 * q + 1];
        out_pl[3 * int64_t(w) + 2] = pl[3 * q + 2];
        ++w;
    }
}

// sample_off[s] = coff[s * n_ctiles], s = 0..S
__global__ void k_vcf_sample_off(const int *__restrict__ coff, int n_samples, int n_ctiles, int *__restrict__ sample_off) {
    const int s = int(blockIdx.x) * blockDim.x + threadIdx.x;
    if (s <= n_samples) sample_off[s] = coff[int64_t(s) * n_ctiles];
}

// ---- makedb: records -> packed panel rows ------------------------------------------------------------------------------------
// the code of vcf_to_csv's _GT_CODE for the cell [a, b) whose GT is subfield gi (0-based, -1 absent): 0 for 0/0 0|0, 1 for 1/1
// 1|1, 2 for 0/1 0|1 1/0 1|0, 3 (missing) for ./. .|. . and for a cell without that subfield; any other text is missing and
// sets `other`.
__device__ __forceinline__ uint32_t vcf_gt_code(const uint8_t *__restrict__ t, int a, int b, int gi, bool &other) {
    if (gi < 0) return 3u;
    int k = 0, g0 = a;
    for (int p = a; p < b && k < gi; ++p)
        if (t[p] == ':') { ++k; g0 = p + 1; }
    if (k < gi) return 3u;
    int g1 = g0;
    while (g1 < b && t[g1] != ':') ++g1;
    if (g1 - g0 == 1 && t[g0] == '.') return 3u;
    if (g1 - g0 == 3 && (t[g0 + 1] == '/' || t[g0 + 1] == '|')) {
        const uint8_t x = t[g0], y = t[g0 + 2];
        if (x == '.' && y == '.') return 3u;
        if ((x == '0' || x == '1') && (y == '0' || y == '1')) return x == y ? uint32_t(x - '0') : 2u;
    }
    other = true;
    return 3u;
}

// one packed word from the warp's 32 cells (lanes without a cell are missing); returns the other calls among them on lane 0
__device__ __forceinline__ int vcf_pack_word(const uint8_t *__restrict__ t, bool have, int a, int b, int gi, uint64_t *__restrict__ dst) {
    bool other = false;
    const uint32_t code = have ? vcf_gt_code(t, a, b, gi, other) : 3u;
    const uint32_t lo = __ballot_sync(0xffffffffu, code & 1u);
    const uint32_t hi = __ballot_sync(0xffffffffu, code & 2u);
    const int n_other = __popc(__ballot_sync(0xffffffffu, other));
    if ((threadIdx.x & 31) == 0) {
        *dst = uint64_t(lo) | (uint64_t(hi) << 32);
        return n_other;
    }
    return 0;
}

// One warp per record of exactly n_samples sample fields (ncell == 1): its row row_off[L] of packed [rows, stride], the cells
// walked as in k_vcf_cells; VCF_NEW_CHROM as there.  chunk_flags[2] += the calls that are no _GT_CODE string.
__global__ void __launch_bounds__(256) k_vcf_gt_packed(const uint8_t *__restrict__ t, const int *__restrict__ starts, int n_lines,
                                                       VcfLines o, const int *__restrict__ row_off, int n_samples, int stride,
                                                       uint64_t *__restrict__ packed, int *__restrict__ chunk_flags) {
    const int lane = threadIdx.x & 31;
    const int n_warps = int(gridDim.x) * (blockDim.x >> 5);
    int other = 0;
    for (int L = int(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); L < n_lines; L += n_warps) {
        if (!o.ncell[L]) continue;
        const int s = starts[L];
        const int clen = o.chrom_len[L];
        bool same = L > 0 && (o.flags[L - 1] & VCF_REC) && o.chrom_len[L - 1] == clen;
        if (same) {
            const int ps = starts[L - 1];
            for (int b0 = 0; b0 < clen && same; b0 += 32) {
                const int i = b0 + lane;
                same = __all_sync(0xffffffffu, i >= clen || t[ps + i] == t[s + i]);
            }
        }
        uint64_t *row = packed + int64_t(row_off[L]) * stride;
        const int gi = o.fmt[L] - 1;
        const int nc = gi >= 0 ? n_samples : 0;          // without GT every call is missing: nothing to read
        const int e = vcf_line_end(t, s, starts[L + 1]);
        int cell = 0, w = 0, cur = o.samp0[L], my_a = 0, my_b = 0;
        for (int base = cur; base < e && cell < nc; base += 32) {
            const int p = base + lane;
            unsigned m = __ballot_sync(0xffffffffu, p < e && t[p] == '\t');
            while (m && cell < nc) {
                const int tp = base + __ffs(m) - 1;
                m &= m - 1;
                if (lane == (cell & 31)) { my_a = cur; my_b = tp; }
                cur = tp + 1;
                if ((++cell & 31) == 0) other += vcf_pack_word(t, true, my_a, my_b, gi, row + w++);
            }
        }
        bool closed_by_end = false;
        if (cell < nc) {                                   // the line end closes the last sample field
            if (lane == (cell & 31)) { my_a = cur; my_b = e; }
            ++cell;
            closed_by_end = true;
        }
        const int pending = (cell & 31) ? (cell & 31) : (closed_by_end ? 32 : 0);
        if (pending) other += vcf_pack_word(t, lane < pending, my_a, my_b, gi, row + w++);
        for (int k = w + lane; k < stride; k += 32) row[k] = ~0ull;     // padding words, or every word without GT
        if (lane == 0 && !same) atomicOr(o.flags + L, VCF_NEW_CHROM);
    }
    if (lane == 0 && other) atomicAdd(chunk_flags + 2, other);
}

// ---- genotype_cross: records -> rows of int8 window-call codes ---------------------------------------------------------------
// class of the GT token [a, b): 0 '.' or empty, 1 "0", 2 "1", 3 anything else
__device__ __forceinline__ int vcf_token_class(const uint8_t *__restrict__ t, int a, int b) {
    if (b == a) return 0;
    if (b - a > 1) return 3;
    return t[a] == '.' ? 0 : t[a] == '0' ? 1 : t[a] == '1' ? 2 : 3;
}

// The code read_vcf_samples + parseGT give the cell [a, b) whose GT is subfield gi (0-based, -1 absent): the GT text split at '/'
// and '|', the first two tokens kept, a missing or empty one read as '.'; 1 for (1,1), 2 for (0,1) and (1,0), -1 for (.,.), 0 for
// any other pair; -1 for a cell without that subfield.
__device__ __forceinline__ int8_t vcf_cross_code(const uint8_t *__restrict__ t, int a, int b, int gi) {
    if (gi < 0) return -1;
    int k = 0, g0 = a;
    for (int p = a; p < b && k < gi; ++p)
        if (t[p] == ':') { ++k; g0 = p + 1; }
    if (k < gi) return -1;
    int c[2] = {0, 0}, n = 0;
    for (int p = g0, st = g0; n < 2; ++p) {
        const bool end = p >= b || t[p] == ':';
        if (!end && t[p] != '/' && t[p] != '|') continue;
        c[n++] = vcf_token_class(t, st, p);
        st = p + 1;
        if (end) break;
    }
    if (c[0] == 2 && c[1] == 2) return 1;
    if (c[0] + c[1] == 3 && c[0] != 3 && c[1] != 3) return 2;
    return c[0] == 0 && c[1] == 0 ? -1 : 0;
}

// One warp per record (ncell == 1): row row_off[L] of codes [rows, n_samples], lane j writing the code of cell 32 w + j, so a
// warp stores 32 consecutive bytes per step; the cells walked as in k_vcf_cells, VCF_NEW_CHROM as there.  Cells past
// min(nsf, n_samples), and every cell of a record without GT in FORMAT, are -1.
__global__ void __launch_bounds__(256) k_vcf_gt_codes(const uint8_t *__restrict__ t, const int *__restrict__ starts, int n_lines,
                                                      VcfLines o, const int *__restrict__ row_off, int n_samples,
                                                      int8_t *__restrict__ codes) {
    const int lane = threadIdx.x & 31;
    const int n_warps = int(gridDim.x) * (blockDim.x >> 5);
    for (int L = int(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); L < n_lines; L += n_warps) {
        if (!o.ncell[L]) continue;
        const int s = starts[L];
        const int clen = o.chrom_len[L];
        bool same = L > 0 && (o.flags[L - 1] & VCF_REC) && o.chrom_len[L - 1] == clen;
        if (same) {
            const int ps = starts[L - 1];
            for (int b0 = 0; b0 < clen && same; b0 += 32) {
                const int i = b0 + lane;
                same = __all_sync(0xffffffffu, i >= clen || t[ps + i] == t[s + i]);
            }
        }
        int8_t *row = codes + int64_t(row_off[L]) * n_samples;
        const int gi = o.fmt[L] - 1;
        const int nc = gi >= 0 ? min(o.nsf[L], n_samples) : 0;    // without GT every call is missing: nothing to read
        const int e = vcf_line_end(t, s, starts[L + 1]);
        int cell = 0, cur = o.samp0[L], my_a = 0, my_b = 0;
        for (int base = cur; base < e && cell < nc; base += 32) {
            const int p = base + lane;
            unsigned m = __ballot_sync(0xffffffffu, p < e && t[p] == '\t');
            while (m && cell < nc) {
                const int tp = base + __ffs(m) - 1;
                m &= m - 1;
                if (lane == (cell & 31)) { my_a = cur; my_b = tp; }
                cur = tp + 1;
                if ((++cell & 31) == 0) row[cell - 32 + lane] = vcf_cross_code(t, my_a, my_b, gi);
            }
        }
        bool closed_by_end = false;
        if (cell < nc) {                                   // the line end closes the last sample field
            if (lane == (cell & 31)) { my_a = cur; my_b = e; }
            ++cell;
            closed_by_end = true;
        }
        const int pending = (cell & 31) ? (cell & 31) : (closed_by_end ? 32 : 0);
        if (lane < pending) row[cell - pending + lane] = vcf_cross_code(t, my_a, my_b, gi);
        for (int k = cell + lane; k < n_samples; k += 32) row[k] = -1;
        if (lane == 0 && !same) atomicOr(o.flags + L, VCF_NEW_CHROM);
    }
}

}  // namespace snpm
