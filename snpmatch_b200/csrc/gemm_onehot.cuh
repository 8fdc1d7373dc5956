// A9 — batched scoring of many called-genotype samples on a SHARED marker panel as a one-hot int8 GEMM on the 5th-gen
// tensor cores (tcgen05.mma kind::i8, accumulators in TMEM).  North-star item (d); no reference symbol (the reference
// runs one process per sample, README.md:9).
//
//   score[s, a] = sum_k sum_c [code_s[k] == c] * [db[k, a] == c]          c in {ref, alt, het}
//   ninfo[s, a] = sum_k [code_s[k] called] * [db[k, a] called]
//
// Both are one GEMM  C[2*64 rows, 128 accessions] += A_op[128, 4K] * B_op[128, 4K]^T  per CTA tile: every panel row k
// contributes four int8 K-slots (slot c = one-hot of the code, slot 3 unused); the first 64 rows of a tile are the score
// operands of 64 samples (one-hot of the sample's call), the last 64 their ninfo operands (1 in every class slot when the
// sample has the marker).  Two expansion kernels write the one-hot operands once, tile by tile, in the exact shared-memory
// image of the canonical no-swizzle K-major UMMA layout; the GEMM kernel is then a pure pipeline: a producer thread fills a
// 4-stage ring with two 1-D TMA bulk copies per k-block, one elected thread issues four tcgen05.mma (M=128, N=256, K=32) per
// block into a 128 x 256 int32 accumulator in TMEM, four epilogue warps read it back with tcgen05.ld.  int32 accumulation is
// exact.  (A first version expanded the operands inside the GEMM kernel; the expansion ALU work and its dependent panel
// loads ran 100x slower than the tensor pipe — profiles/r1_configs.jsonl keeps that measurement.)
#pragma once
#include "common.cuh"
#include "score.cuh"

namespace snpm {

constexpr int OG_STAGES = 4;
constexpr int OG_BM = 128, OG_BN = 256;
constexpr int OG_ROWS = 32;                     // panel rows per k-block = 128 K-bytes = 4 MMAs of K=32
constexpr int OG_A_TILE = OG_BM * 128;          // bytes of one A tile (128 operand rows x 128 K-bytes)
constexpr int OG_B_TILE = OG_BN * 128;
constexpr int OG_THREADS = 192;                 // warp 0: TMA producer, warp 1: TMEM owner + MMA issuer, warps 2-5: epilogue

// Operand tiles live in HBM already in the shared-memory image the tensor core reads: the canonical no-swizzle K-major UMMA
// layout — core matrix = 8 operand rows x 16 K-bytes, contiguous (128 B); the core matrices of one 16-byte K chunk follow each
// other (stride 128 B = SBO), the 8 K chunks of a k-block are R*16 bytes apart (LBO; R = rows of the tile).  A tile therefore
// reaches shared memory with ONE 1-D TMA bulk copy, no tensor map and no swizzle.
__host__ __device__ __forceinline__ uint32_t og_tile_offset(int row, int chunk, int tile_rows) {
    return uint32_t(chunk) * uint32_t(tile_rows) * 16u + uint32_t(row >> 3) * 128u + uint32_t(row & 7) * 16u;
}

// A operand: tile (m_blk, kb) = 64 samples x 32 markers; rows 0-63 one-hot of the sample's call (score), rows 64-127 ones in
// every class slot when the sample has the marker (ninfo).  K slot = 4 * marker + class; slot 3 stays zero.
// PACKED: codes are 2 bits per marker, four markers per byte (marker k in bits 2(k&3)..2(k&3)+1 of byte k >> 2), `pitch` bytes
// per sample; else one byte per marker.
template <bool PACKED>
__global__ void __launch_bounds__(128) k_onehot_expand_samples(const uint8_t *__restrict__ codes, int32_t S, int32_t Kpad, int64_t pitch,
                                                               unsigned char *__restrict__ a_tiled) {
    const int n_kb = Kpad / OG_ROWS;
    const int kb = blockIdx.x, m_blk = blockIdx.y, t = threadIdx.x;
    const int sample = m_blk * 64 + (t & 63);
    const bool ninfo_row = t >= 64;
    unsigned char *tile = a_tiled + (size_t(m_blk) * n_kb + kb) * OG_A_TILE;
    uint32_t pk[2] = {0xFFFFFFFFu, 0xFFFFFFFFu};              // PACKED: the 32 markers of this k-block (8 bytes)
    if (PACKED && sample < S) {
        const uint2 v = *reinterpret_cast<const uint2 *>(codes + size_t(sample) * pitch + size_t(kb) * (OG_ROWS / 4));
        pk[0] = v.x;
        pk[1] = v.y;
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        uint32_t cw;
        if (PACKED) {
            const uint32_t b = (pk[c >> 2] >> (8 * (c & 3))) & 0xFFu;
            cw = (b & 3u) | ((b >> 2 & 3u) << 8) | ((b >> 4 & 3u) << 16) | ((b >> 6) << 24);
        } else {
            cw = sample < S ? *reinterpret_cast<const uint32_t *>(codes + size_t(sample) * pitch + kb * OG_ROWS + 4 * c) : 0x03030303u;
        }
        uint4 v;
        uint32_t *pv = reinterpret_cast<uint32_t *>(&v);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint32_t code = (cw >> (8 * q)) & 0xFFu;
            pv[q] = code < 3u ? (ninfo_row ? 0x00010101u : (1u << (8 * code))) : 0u;
        }
        *reinterpret_cast<uint4 *>(tile + og_tile_offset(t, c, OG_BM)) = v;
    }
}

// B operand: tile (n_blk, kb) = 256 accessions x 32 panel rows, one-hot of the database call (missing, masked hets and padding
// rows/accessions are all-zero)
__global__ void __launch_bounds__(256) k_onehot_expand_panel(const uint64_t *__restrict__ packed, int32_t stride, const int32_t *__restrict__ rows,
                                                             int32_t Kpad, int32_t skip_hets, unsigned char *__restrict__ b_tiled) {
    const int n_kb = Kpad / OG_ROWS;
    const int kb = blockIdx.x, n_blk = blockIdx.y, t = threadIdx.x;
    const int acc = n_blk * OG_BN + t;
    const bool acc_ok = acc < stride * 32;
    const uint64_t *pcol = packed + (acc_ok ? (acc >> 5) : 0);
    const int bit = acc & 31;
    unsigned char *tile = b_tiled + (size_t(n_blk) * n_kb + kb) * OG_B_TILE;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        uint4 v;
        uint32_t *pv = reinterpret_cast<uint32_t *>(&v);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int32_t r = rows[kb * OG_ROWS + 4 * c + q];
            uint32_t w = 0u;
            if (r >= 0 && acc_ok) {
                const uint64_t x = __ldg(pcol + int64_t(r) * stride);
                const uint32_t code = (uint32_t(x) >> bit & 1u) | ((uint32_t(x >> 32) >> bit & 1u) << 1);
                if (code < 3u && !(skip_hets && code == 2u)) w = 1u << (8 * code);
            }
            pv[q] = w;
        }
        *reinterpret_cast<uint4 *>(tile + og_tile_offset(t, c, OG_BN)) = v;
    }
}

struct OneHotGemmArgs {
    const unsigned char *a_tiled;   // [m_blocks][n_kb][OG_A_TILE]
    const unsigned char *b_tiled;   // [n_blocks][n_kb][OG_B_TILE]
    int32_t n_kb, m_blocks, n_blocks;
    int32_t S;
    int32_t *out_score;             // [S, ld_out]
    int32_t *out_ninfo;             // [S, ld_out]
    int32_t ld_out;                 // accessions rounded up to a multiple of OG_BN
};

__device__ __forceinline__ uint64_t og_smem_desc(uint32_t saddr, uint32_t lbo_bytes) {
    // K-major, no swizzle.  Bits: [0,14) address>>4, [16,30) LBO>>4 (between the two 16-byte K chunks of an MMA), [32,46) SBO>>4
    // (between 8-row groups = 128 B), [46,48) descriptor version 1 (Blackwell), layout type 0.
    return uint64_t((saddr & 0x3FFFFu) >> 4) | (uint64_t(lbo_bytes >> 4) << 16) | (uint64_t(128u >> 4) << 32) | (uint64_t(1) << 46);
}

// Persistent: grid = min(tiles, SMs); a CTA walks tiles blockIdx.x, +gridDim.x, ... (m fastest, so CTAs running at the same
// time share the B operand in L2).  Two 256-column accumulators in TMEM alternate, so the epilogue of tile i overlaps the
// MMAs of tile i+1.
__global__ void __launch_bounds__(OG_THREADS, 1) k_onehot_gemm(const OneHotGemmArgs a) {
    extern __shared__ __align__(1024) unsigned char og_smem[];
    __shared__ uint64_t full[OG_STAGES], empty[OG_STAGES], acc_ready[2], acc_free[2];
    __shared__ uint32_t tmem_base_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_kb = a.n_kb;
    const int n_tiles = a.m_blocks * a.n_blocks;
    constexpr uint32_t STAGE_BYTES = OG_A_TILE + OG_B_TILE;

    if (threadIdx.x == 0) {
        for (int s = 0; s < OG_STAGES; ++s) {
            mbar_init(smem_u32(&full[s]), 1u);          // producer's arrive.expect_tx + the bytes of two bulk copies
            mbar_init(smem_u32(&empty[s]), 1u);         // tcgen05.commit
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(smem_u32(&acc_ready[s]), 1u);     // tcgen05.commit after a tile's last MMA
            mbar_init(smem_u32(&acc_free[s]), 4u);      // one arrive per epilogue warp
        }
        mbar_fence_init();
    }
    if (warp == 1) {                                    // all of TMEM: two 128-lane x 256-column int32 accumulators
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&tmem_base_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_slot;

    if (warp == 0) {
        // ---- producer: two 1-D TMA bulk copies per k-block (the tiles are stored in their shared-memory image) ----------
        if (lane == 0) {
            uint32_t it = 0;                             // k-blocks issued so far, over all tiles
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const int m_blk = tile % a.m_blocks, n_blk = tile / a.m_blocks;
                const unsigned char *ga = a.a_tiled + size_t(m_blk) * n_kb * OG_A_TILE;
                const unsigned char *gb = a.b_tiled + size_t(n_blk) * n_kb * OG_B_TILE;
                for (int kb = 0; kb < n_kb; ++kb, ++it) {
                    const uint32_t st = it % OG_STAGES;
                    mbar_wait(smem_u32(&empty[st]), ((it / OG_STAGES) & 1u) ^ 1u);
                    const uint32_t bar = smem_u32(&full[st]);
                    unsigned char *sa = og_smem + size_t(st) * STAGE_BYTES;
                    mbar_arrive_expect_tx(bar, STAGE_BYTES);
                    tma_bulk_g2s(smem_u32(sa), ga + size_t(kb) * OG_A_TILE, OG_A_TILE, bar);
                    tma_bulk_g2s(smem_u32(sa + OG_A_TILE), gb + size_t(kb) * OG_B_TILE, OG_B_TILE, bar);
                }
            }
        }
    } else if (warp == 1) {
        // ---- MMA issuer: one elected thread ---------------------------------------------------------------------------------
        // instruction descriptor (kind::i8): D = S32 (bits 4-5 = 2), A/B = unsigned 8-bit, both K-major, N>>3 at bit 17, M>>4 at bit 24
        const uint32_t idesc = (2u << 4) | (uint32_t(OG_BN >> 3) << 17) | (uint32_t(OG_BM >> 4) << 24);
        uint32_t it = 0, ti = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
            const uint32_t buf = ti & 1u;
            mbar_wait(smem_u32(&acc_free[buf]), ((ti >> 1) & 1u) ^ 1u);      // the epilogue has drained this accumulator
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t tmem_acc = tmem_base + buf * uint32_t(OG_BN);
            for (int kb = 0; kb < n_kb; ++kb, ++it) {
                const uint32_t st = it % OG_STAGES;
                mbar_wait(smem_u32(&full[st]), (it / OG_STAGES) & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (lane == 0) {
                    const uint32_t sa = smem_u32(og_smem + size_t(st) * STAGE_BYTES), sb = sa + OG_A_TILE;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {     // K = 32 bytes = K chunks 2kk, 2kk+1
                        const uint64_t da = og_smem_desc(sa + kk * 2 * (OG_BM * 16), OG_BM * 16);
                        const uint64_t db = og_smem_desc(sb + kk * 2 * (OG_BN * 16), OG_BN * 16);
                        const uint32_t accumulate = (kb | kk) ? 1u : 0u;
                        asm volatile(
                            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                            "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                            ::"r"(tmem_acc), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
                    }
                    // the stage is free once these MMAs have read it; the accumulator is complete after the last block
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&empty[st])) : "memory");
                    if (kb == n_kb - 1)
                        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&acc_ready[buf])) : "memory");
                }
                __syncwarp();
            }
        }
    } else {
        // ---- epilogue: TMEM -> registers -> global; a warp may touch TMEM lanes 32*(warp%4) .. +31 = tile rows ----------------
        const int lg = warp & 3;
        const int row = lg * 32 + lane;                  // tile row: < 64 score of a sample, >= 64 its ninfo
        uint32_t ti = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
            const int m_blk = tile % a.m_blocks, n_blk = tile / a.m_blocks;
            const uint32_t buf = ti & 1u;
            mbar_wait(smem_u32(&acc_ready[buf]), (ti >> 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int s_out = m_blk * 64 + (row & 63);
            int32_t *dst = (row < 64 ? a.out_score : a.out_ninfo) + int64_t(s_out) * a.ld_out + n_blk * OG_BN;
#pragma unroll 1
            for (int col = 0; col < OG_BN; col += 32) {
                uint32_t r[32];
                const uint32_t taddr = tmem_base + buf * uint32_t(OG_BN) + (uint32_t(lg * 32) << 16) + uint32_t(col);
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                      "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
                      "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
                      "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                    : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (s_out < a.S) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4)
                        *reinterpret_cast<int4 *>(dst + col + j) = make_int4(int(r[j]), int(r[j + 1]), int(r[j + 2]), int(r[j + 3]));
                }
            }
            // this warp has read its lanes of the accumulator: hand the buffer back to the MMA warp
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&acc_free[buf]));
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

// packed codes, K not a multiple of 4: the spare bit pairs of a row's last byte read as absent (code 3)
__global__ void k_onehot_mask_tail(uint8_t *__restrict__ codes, int64_t S, int64_t pitch, int64_t K) {
    const int64_t s = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (s < S) codes[s * pitch + (K >> 2)] |= uint8_t(0xFFu << (2 * (K & 3)));
}

// int32 GEMM outputs -> the f64 reduce rows the likelihood epilogue reads (score | ninfo | markers | 0).  Sample = blockIdx.x (grid
// x takes 2^31 - 1, grid y only 65 535); the CTAs along y stride over the accessions.
__global__ void __launch_bounds__(256) k_onehot_totals(const int32_t *__restrict__ out_score, const int32_t *__restrict__ out_ninfo,
                                                       int32_t ld_out, int32_t n_acc, int32_t k_markers, double *__restrict__ red) {
    const int s = blockIdx.x;
    double *row = red + int64_t(s) * (2 * int64_t(n_acc) + 2);
    for (int acc = blockIdx.y * blockDim.x + threadIdx.x; acc < n_acc; acc += gridDim.y * blockDim.x) {
        row[acc] = double(out_score[int64_t(s) * ld_out + acc]);
        row[n_acc + acc] = double(out_ninfo[int64_t(s) * ld_out + acc]);
    }
    if (blockIdx.y == 0 && threadIdx.x == 0) {
        row[2 * n_acc] = double(k_markers);
        row[2 * n_acc + 1] = 0.0;
    }
}

}  // namespace snpm
