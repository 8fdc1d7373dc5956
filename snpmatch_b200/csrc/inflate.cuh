// BGZF members inflated on the device (`.vcf.gz` input of the device VCF readers).
//
// BGZF (the gzip flavour of bgzip / `bcftools -Oz`) is a series of independent gzip members of at most 64 KiB of text, each
// naming its compressed size in a `BC` extra subfield and its text size in the trailer.  k_bgzf_inflate gives each member one
// warp: the warp decodes the member's raw DEFLATE stream (RFC 1951) into its slot of the output, then checks ISIZE and CRC-32.
//
// The bit reader, table build and symbol decode are __host__ __device__ and take (lane, n_lanes): on the device every lane of
// the warp runs the same serial decode on the same bits (shared-memory and input loads broadcast, so no shuffles are needed),
// lane 0 writes literals and the lanes copy a match together; compiled for the host with n_lanes = 1 the same code is the
// decoder the CPU tests check against zlib.  Every input is untrusted: each bit read is checked against the payload length,
// each write against the member's ISIZE, each back-reference against the bytes the member has produced, and code-length sets
// follow zlib's inftrees rules (over-subscribed and incomplete sets are refused, except a single code of length 1; an all-zero
// distance set is accepted and fails only when a distance is used).
#pragma once
#include <stdint.h>

#if defined(__CUDA_ARCH__)
#define BGZF_SYNC() __syncwarp()
#else
#define BGZF_SYNC() ((void)0)
#endif

enum { BGZF_OK = 0, BGZF_BAD_STREAM = 1, BGZF_BAD_LENGTH = 2, BGZF_BAD_CRC = 3 };

#define BGZF_LIT_BITS 10                 // primary lookup of literal/length codes; longer codes take the canonical walk
#define BGZF_DIST_BITS 8                 // primary lookup of distance codes
#define BGZF_CL_BITS 7                   // code-length codes are at most 7 bits
#define BGZF_WARPS 8                     // decoders (warps) per block of k_bgzf_inflate

// per-decoder tables (shared memory on the device): 3.6 KB
struct BgzfTables {
    uint16_t lit[1 << BGZF_LIT_BITS];    // (symbol << 4) | length for codes of <= 10 bits, 0 otherwise
    uint16_t dist[1 << BGZF_DIST_BITS];
    uint16_t lcount[16], dcount[16];     // codes per length
    uint16_t lsym[288], dsym[32];        // symbols ordered by (length, value)
    uint16_t offs[16];                   // scratch of the table build
    uint8_t lens[288 + 32];              // code lengths of the block being set up
};

struct BgzfBits {
    const uint8_t *p;
    uint32_t n, pos;                     // payload bytes, bytes moved into buf
    uint64_t buf;
    int cnt;                             // bits in buf
};

__host__ __device__ inline uint8_t bgzf_load(const uint8_t *p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}

__host__ __device__ inline void bgzf_refill(BgzfBits &b) {
    while (b.cnt <= 56 && b.pos < b.n) {
        b.buf |= uint64_t(bgzf_load(b.p + b.pos)) << b.cnt;
        ++b.pos;
        b.cnt += 8;
    }
}

// k (<= 32) bits, or -1 when the payload ends first
__host__ __device__ inline int64_t bgzf_bits(BgzfBits &b, int k) {
    if (b.cnt < k) {
        bgzf_refill(b);
        if (b.cnt < k) return -1;
    }
    const uint32_t v = uint32_t(b.buf & ((uint64_t(1) << k) - 1));
    b.buf >>= k;
    b.cnt -= k;
    return v;
}

__host__ __device__ inline uint32_t bgzf_rev(uint32_t code, int len) {
#if defined(__CUDA_ARCH__)
    return __brev(code) >> (32 - len);
#else
    uint32_t r = 0;
    for (int i = 0; i < len; ++i) r |= ((code >> i) & 1u) << (len - 1 - i);
    return r;
#endif
}

// Canonical code of lens[0..n) into table (tbits primary bits), count and sym.  codes: the code-length code, which must be
// complete; otherwise a literal/length or distance code, which may be incomplete only as a single code of length 1, and may
// be empty (no table entry then decodes).  Returns false on a refused set.  lens and the outputs are shared by the lanes.
__host__ __device__ inline bool bgzf_build(BgzfTables &T, const uint8_t *lens, int n, uint16_t *table, int tbits, uint16_t *count,
                                           uint16_t *sym, bool codes, int lane, int n_lanes) {
    if (lane == 0) {
        for (int l = 0; l < 16; ++l) count[l] = 0;
        for (int s = 0; s < n; ++s) ++count[lens[s]];
        count[0] = 0;
        T.offs[1] = 0;
        for (int l = 1; l < 15; ++l) T.offs[l + 1] = T.offs[l] + count[l];
        for (int s = 0; s < n; ++s)
            if (lens[s]) sym[T.offs[lens[s]]++] = uint16_t(s);
    }
    for (int i = lane; i < (1 << tbits); i += n_lanes) table[i] = 0;
    BGZF_SYNC();
    int left = 1, max_len = 0, total = 0;
    for (int l = 1; l < 16; ++l) {
        left = (left << 1) - count[l];
        if (left < 0) return false;                       // over-subscribed
        if (count[l]) max_len = l;
        total += count[l];
    }
    if (max_len == 0) return !codes;
    if (left > 0 && (codes || max_len != 1)) return false;  // incomplete
    // the codes of at most tbits bits, lane-parallel over the sorted symbols
    for (int i = lane; i < total; i += n_lanes) {
        int start = 0, first = 0, len = 1;
        for (;; ++len) {                                  // canonical: first code and first sorted index of each length
            if (i < start + count[len]) break;
            start += count[len];
            first = (first + count[len]) << 1;
        }
        if (len > tbits) continue;
        const uint16_t s = sym[i];
        const uint16_t e = uint16_t((s << 4) | len);
        for (uint32_t r = bgzf_rev(uint32_t(first + i - start), len); r < (1u << tbits); r += 1u << len) table[r] = e;
    }
    BGZF_SYNC();
    return true;
}

// one symbol, or -1 on a code not in the set or a code running past the payload
__host__ __device__ inline int bgzf_decode(BgzfBits &b, const uint16_t *table, int tbits, const uint16_t *count, const uint16_t *sym) {
    if (b.cnt < 15) bgzf_refill(b);
    const uint32_t e = table[b.buf & ((1u << tbits) - 1)];
    if (e) {
        const int len = int(e & 15);
        if (len > b.cnt) return -1;
        b.buf >>= len;
        b.cnt -= len;
        return int(e >> 4);
    }
    int code = 0, first = 0, index = 0;
    uint64_t bits = b.buf;
    for (int len = 1; len < 16; ++len) {
        code |= int(bits & 1);
        bits >>= 1;
        const int c = count[len];
        if (code - c < first) {
            if (len > b.cnt) return -1;
            b.buf >>= len;
            b.cnt -= len;
            return sym[index + (code - first)];
        }
        index += c;
        first = (first + c) << 1;
        code <<= 1;
    }
    return -1;
}

// length and distance bases (RFC 1951 3.2.5) in closed form: no per-call table in local memory
__host__ __device__ inline uint32_t bgzf_len_base(int s) {
    return s < 8 ? uint32_t(s + 3) : s == 28 ? 258u : ((4u + (s & 3)) << ((s >> 2) - 1)) + 3;
}
__host__ __device__ inline int bgzf_len_extra(int s) { return s < 8 || s == 28 ? 0 : (s - 4) >> 2; }
__host__ __device__ inline uint32_t bgzf_dist_base(int s) {
    return s < 4 ? uint32_t(s + 1) : ((2u + (s & 1)) << ((s >> 1) - 1)) + 1;
}
__host__ __device__ inline int bgzf_dist_extra(int s) { return s < 4 ? 0 : (s >> 1) - 1; }

// Inflate one raw DEFLATE stream in[0..in_len) into out[0..cap).  Returns BGZF_OK with *produced set, BGZF_BAD_STREAM (an
// invalid stream, one that reads past in_len or one whose final block ends before the last payload byte) or BGZF_BAD_LENGTH
// (more than cap bytes of output).  Every lane must call it with the same arguments.
__host__ __device__ inline int bgzf_inflate_raw(const uint8_t *in, uint32_t in_len, uint8_t *out, uint32_t cap, uint32_t *produced,
                                                BgzfTables &T, int lane, int n_lanes) {
    BgzfBits b{in, in_len, 0, 0, 0};
    uint32_t o = 0;
    int64_t last;
    do {
        last = bgzf_bits(b, 1);
        const int64_t type = bgzf_bits(b, 2);
        if (last < 0 || type < 0 || type == 3) return BGZF_BAD_STREAM;
        if (type == 0) {                                  // stored
            const int skip = b.cnt & 7;
            b.buf >>= skip;
            b.cnt -= skip;
            const int64_t len = bgzf_bits(b, 16), nlen = bgzf_bits(b, 16);
            if (len < 0 || nlen < 0 || len != (~nlen & 0xffff)) return BGZF_BAD_STREAM;
            if (uint64_t(o) + uint64_t(len) > cap) return BGZF_BAD_LENGTH;
            uint32_t k = 0;
            for (; k < uint32_t(len) && b.cnt >= 8; ++k) {        // whole bytes still in the bit buffer
                if (lane == 0) out[o + k] = uint8_t(b.buf);
                b.buf >>= 8;
                b.cnt -= 8;
            }
            const uint32_t rest = uint32_t(len) - k;
            if (b.pos + uint64_t(rest) > b.n) return BGZF_BAD_STREAM;
            for (uint32_t i = lane; i < rest; i += n_lanes) out[o + k + i] = bgzf_load(b.p + b.pos + i);
            b.pos += rest;
            o += uint32_t(len);
            continue;
        }
        int hlit = 288, hdist = 32;
        if (type == 1) {                                  // fixed codes
            for (int i = lane; i < 320; i += n_lanes) T.lens[i] = uint8_t(i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : 5);
            BGZF_SYNC();
        } else {                                          // dynamic codes
            const int64_t a = bgzf_bits(b, 5), d = bgzf_bits(b, 5), c = bgzf_bits(b, 4);
            if (a < 0 || d < 0 || c < 0) return BGZF_BAD_STREAM;
            hlit = int(a) + 257;
            hdist = int(d) + 1;
            if (hlit > 286 || hdist > 30) return BGZF_BAD_STREAM;
            // code-length code lengths in the order of RFC 1951 3.2.7
            const char *order = "\x10\x11\x12\x00\x08\x07\x09\x06\x0a\x05\x0b\x04\x0c\x03\x0d\x02\x0e\x01\x0f";
            if (lane == 0)
                for (int i = 0; i < 19; ++i) T.lens[i] = 0;
            for (int i = 0; i < int(c) + 4; ++i) {
                const int64_t v = bgzf_bits(b, 3);
                if (v < 0) return BGZF_BAD_STREAM;
                if (lane == 0) T.lens[int(order[i])] = uint8_t(v);
            }
            BGZF_SYNC();
            if (!bgzf_build(T, T.lens, 19, T.lit, BGZF_CL_BITS, T.lcount, T.lsym, true, lane, n_lanes)) return BGZF_BAD_STREAM;
            // the literal/length lengths go to lens[0..hlit), the distance lengths to lens[288..288 + hdist)
            int n = 0, prev = 0;
            const int want = hlit + hdist;
            while (n < want) {
                const int s = bgzf_decode(b, T.lit, BGZF_CL_BITS, T.lcount, T.lsym);
                if (s < 0) return BGZF_BAD_STREAM;
                if (s < 16) {
                    if (lane == 0) T.lens[n < hlit ? n : n - hlit + 288] = uint8_t(s);
                    prev = s;
                    ++n;
                    continue;
                }
                int val = 0;
                int64_t rep;
                if (s == 16) {
                    if (n == 0) return BGZF_BAD_STREAM;
                    val = prev;
                    rep = bgzf_bits(b, 2);
                    rep = rep < 0 ? -1 : rep + 3;
                } else if (s == 17) {
                    rep = bgzf_bits(b, 3);
                    rep = rep < 0 ? -1 : rep + 3;
                } else {
                    rep = bgzf_bits(b, 7);
                    rep = rep < 0 ? -1 : rep + 11;
                }
                if (rep < 0 || n + rep > want) return BGZF_BAD_STREAM;
                for (int i = n + lane; i < n + int(rep); i += n_lanes) T.lens[i < hlit ? i : i - hlit + 288] = uint8_t(val);
                n += int(rep);
                prev = val;
            }
            BGZF_SYNC();
            if (T.lens[256] == 0) return BGZF_BAD_STREAM;  // no end-of-block code
        }
        if (!bgzf_build(T, T.lens, hlit, T.lit, BGZF_LIT_BITS, T.lcount, T.lsym, false, lane, n_lanes)) return BGZF_BAD_STREAM;
        if (!bgzf_build(T, T.lens + 288, hdist, T.dist, BGZF_DIST_BITS, T.dcount, T.dsym, false, lane, n_lanes)) return BGZF_BAD_STREAM;
        for (;;) {
            int s = bgzf_decode(b, T.lit, BGZF_LIT_BITS, T.lcount, T.lsym);
            if (s < 0) return BGZF_BAD_STREAM;
            if (s < 256) {
                if (o >= cap) return BGZF_BAD_LENGTH;
                if (lane == 0) out[o] = uint8_t(s);
                ++o;
                continue;
            }
            if (s == 256) break;
            s -= 257;
            if (s >= 29) return BGZF_BAD_STREAM;          // symbols 286, 287
            const int64_t le = bgzf_bits(b, bgzf_len_extra(s));
            if (le < 0) return BGZF_BAD_STREAM;
            const uint32_t len = bgzf_len_base(s) + uint32_t(le);
            const int ds = bgzf_decode(b, T.dist, BGZF_DIST_BITS, T.dcount, T.dsym);
            if (ds < 0 || ds >= 30) return BGZF_BAD_STREAM;  // no code, or symbols 30, 31
            const int64_t de = bgzf_bits(b, bgzf_dist_extra(ds));
            if (de < 0) return BGZF_BAD_STREAM;
            const uint32_t dist = bgzf_dist_base(ds) + uint32_t(de);
            if (dist > o) return BGZF_BAD_STREAM;          // before the member's first byte
            if (uint64_t(o) + len > cap) return BGZF_BAD_LENGTH;
            BGZF_SYNC();                                  // the bytes produced so far are visible to every lane
            for (uint32_t i = lane; i < len; i += n_lanes) out[o + i] = out[o - dist + (i < dist ? i : i % dist)];
            o += len;
        }
    } while (!last);
    BGZF_SYNC();
    if (b.pos - uint32_t(b.cnt >> 3) != in_len) return BGZF_BAD_STREAM;  // the final block must end in the last payload byte
    *produced = o;
    return BGZF_OK;
}

// ---- CRC-32 (gzip's, reflected 0xEDB88320) over lane slices, combined with x^(8n) mod P factors ---------------------------
__host__ __device__ inline uint32_t bgzf_multmodp(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (uint32_t m = 1u << 31; m; m >>= 1) {
        if (a & m) p ^= b;
        b = b & 1 ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}

// tab[256]: the byte table; x2n[32]: x^(2^k) mod P
__host__ __device__ inline void bgzf_crc_tables(uint32_t *tab, uint32_t *x2n, int lane, int n_lanes) {
    for (int i = lane; i < 256; i += n_lanes) {
        uint32_t c = uint32_t(i);
        for (int k = 0; k < 8; ++k) c = c & 1 ? (c >> 1) ^ 0xEDB88320u : c >> 1;
        tab[i] = c;
    }
    if (lane == 0) {
        uint32_t p = 1u << 30;                            // x^1
        x2n[0] = p;
        for (int k = 1; k < 32; ++k) x2n[k] = p = bgzf_multmodp(p, p);
    }
}

// r * x^(8n) mod P: a CRC register carried over n more bytes (zlib's crc32_combine step)
__host__ __device__ inline uint32_t bgzf_shift(uint32_t r, uint64_t n, const uint32_t *x2n) {
    uint32_t p = 1u << 31;                                // x^0
    for (int k = 3; n; n >>= 1, ++k)
        if (n & 1) p = bgzf_multmodp(x2n[k & 31], p);
    return bgzf_multmodp(p, r);
}

// slice `lane` of n_lanes of d[0..n): its term of the CRC register of the whole, from a zero register
__host__ __device__ inline uint32_t bgzf_crc_slice(const uint8_t *d, uint32_t n, const uint32_t *tab, const uint32_t *x2n, int lane,
                                                   int n_lanes) {
    const uint32_t per = (n + n_lanes - 1) / n_lanes;
    const uint32_t a = per * uint32_t(lane) < n ? per * uint32_t(lane) : n;
    const uint32_t e = a + per < n ? a + per : n;
    uint32_t r = 0;
    for (uint32_t i = a; i < e; ++i) r = tab[(r ^ d[i]) & 255] ^ (r >> 8);
    return bgzf_shift(r, n - e, x2n);
}

// gzip's CRC-32 of d[0..n) from the XOR of the n_lanes slice terms
__host__ __device__ inline uint32_t bgzf_crc_final(uint32_t terms, uint32_t n, const uint32_t *x2n) {
    return ~(terms ^ bgzf_shift(0xFFFFFFFFu, n, x2n));
}

struct BgzfMember {
    uint32_t in_off, in_len;                              // the raw DEFLATE payload in the batch's compressed bytes
    uint32_t out_off, isize;                              // the text's place in the batch's output (exclusive sum of ISIZE)
    uint32_t crc;                                         // the trailer's CRC-32
};

#if defined(__CUDACC__)
// one warp per member; status[m] = BGZF_OK or the reason the member is refused
__global__ void __launch_bounds__(BGZF_WARPS * 32) k_bgzf_inflate(const uint8_t *__restrict__ comp, const BgzfMember *__restrict__ mem,
                                                                  int n, uint8_t *__restrict__ out, int32_t *__restrict__ status) {
    __shared__ BgzfTables tabs[BGZF_WARPS];
    __shared__ uint32_t crc_tab[256], x2n[32];
    bgzf_crc_tables(crc_tab, x2n, threadIdx.x, blockDim.x);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int m = blockIdx.x * BGZF_WARPS + warp; m < n; m += gridDim.x * BGZF_WARPS) {
        const BgzfMember d = mem[m];
        uint8_t *o = out + d.out_off;
        uint32_t produced = 0;
        int st = bgzf_inflate_raw(comp + d.in_off, d.in_len, o, d.isize, &produced, tabs[warp], lane, 32);
        if (st == BGZF_OK && produced != d.isize) st = BGZF_BAD_LENGTH;
        if (st == BGZF_OK) {
            uint32_t t = bgzf_crc_slice(o, d.isize, crc_tab, x2n, lane, 32);
            for (int k = 16; k; k >>= 1) t ^= __shfl_xor_sync(0xffffffffu, t, k);
            if (bgzf_crc_final(t, d.isize, x2n) != d.crc) st = BGZF_BAD_CRC;
        }
        if (lane == 0) status[m] = st;
        __syncwarp();
    }
}
#endif
