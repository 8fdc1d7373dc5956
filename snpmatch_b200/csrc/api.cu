// C ABI of libsnpmatch_b200 (include/snpmatch_b200.h): handle lifecycle, uploads, kernel launches.
#include "common.cuh"
#include <atomic>
#include <memory>
#include <new>
#include "pack.cuh"
#include "join.cuh"
#include "score.cuh"
#include "windows.cuh"
#include "f1.cuh"
#include "hardcall.cuh"
#include "gemm_onehot.cuh"
#include "grouped.cuh"
#include "group_sort.cuh"
#include "grouped2.cuh"
#include "pairs.cuh"
#include "pair_matrix.cuh"
#include "cross_geno.cuh"
#include <unordered_map>

namespace snpm {
thread_local std::string g_last_error;

static int grid_for(int64_t items, int threads, int n_sm, int per_sm = 16) {
    int64_t g = ceil_div64(items, threads);
    const int64_t cap = int64_t(n_sm) * per_sm;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return int(g);
}

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
};

// A kernel's dynamic shared-memory limit is an attribute of the function in the CURRENT device's context, so a kernel that asks
// for more than 48 KB needs it set on every device it runs on (a Database per GPU in one process).  Set once per (kernel,
// device): bit d of `done` = set on device d (devices past 63 set it on every call).
template <auto Kernel>
static cudaError_t smem_attr(int bytes) {
    static std::atomic<uint64_t> done{0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const uint64_t bit = dev < 64 ? uint64_t(1) << dev : 0;
    if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
    e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) done.fetch_or(bit, std::memory_order_release);
    return e;
}

template <bool SKIP, int NW, int MINB>
static int launch_score_t(cudaStream_t st, const ScoreArgs &a, dim3 grid, dim3 block, size_t smem) {
    SNPM_CUDA((smem_attr<k_score_segments<SKIP, NW, MINB>>(200 * 1024)));
    k_score_segments<SKIP, NW, MINB><<<grid, block, smem, st>>>(a);
    SNPM_KERNEL_CHECK();
    return SNPM_OK;
}

static int launch_score(cudaStream_t st, const ScoreArgs &a, int grid_x, bool skip_hets) {
    int nw, yb;
    size_t smem;
    score_launch_shape(a.stride, &nw, &yb, &smem);
    if (grid_x <= 0) return SNPM_OK;
    dim3 grid(grid_x, yb), block(32, nw + 1);      // + the producer warp
    // launch bounds match the two shapes that occur in practice: 9 consumer warps (a 1135-accession row in one CTA)
    // and 8 (32-word slices of wide panels); anything else takes the generic instantiation
    if (nw + 1 == 10) return skip_hets ? launch_score_t<true, 10, 2>(st, a, grid, block, smem) : launch_score_t<false, 10, 2>(st, a, grid, block, smem);
    if (nw + 1 == 9) return skip_hets ? launch_score_t<true, 9, 2>(st, a, grid, block, smem) : launch_score_t<false, 9, 2>(st, a, grid, block, smem);
    return skip_hets ? launch_score_t<true, SC_MAX_WARPS + 1, 1>(st, a, grid, block, smem)
                     : launch_score_t<false, SC_MAX_WARPS + 1, 1>(st, a, grid, block, smem);
}
}  // namespace snpm

using namespace snpm;

extern "C" {

int snpm_version(void) { return SNPM_VERSION; }
const char *snpm_last_error(void) { return g_last_error.c_str(); }

int snpm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int snpm_device_info(int device, char *name_buf, int name_len, int *sm, int64_t *mem_bytes, int *n_sm) {
    cudaDeviceProp p;
    SNPM_CUDA(cudaGetDeviceProperties(&p, device));
    if (name_buf && name_len > 0) { strncpy(name_buf, p.name, size_t(name_len) - 1); name_buf[name_len - 1] = 0; }
    if (sm) *sm = p.major * 10 + p.minor;
    if (mem_bytes) *mem_bytes = int64_t(p.totalGlobalMem);
    if (n_sm) *n_sm = p.multiProcessorCount;
    return SNPM_OK;
}

// ---- A0 ------------------------------------------------------------------------------------------
int snpm_db_create(int device, int64_t n_rows, int32_t n_acc, const int32_t *positions, const int64_t *chr_regions,
                   int32_t n_chr, int64_t row0_global, snpm_db **out) {
    if (!out) return fail(SNPM_E_ARG, "snpm_db_create: out is NULL");
    *out = nullptr;
    if (n_rows < 0 || n_rows >= (int64_t(1) << 31) || n_acc <= 0 || n_chr < 0 || (n_rows > 0 && !positions) || (n_chr > 0 && !chr_regions))
        return fail(SNPM_E_ARG, "snpm_db_create: bad shape (n_rows=%lld n_acc=%d n_chr=%d)", (long long)n_rows, n_acc, n_chr);
    for (int c = 0; c < n_chr; ++c) {
        const int64_t s = chr_regions[2 * c], e = chr_regions[2 * c + 1];
        if (s < 0 || e < s || e > n_rows) return fail(SNPM_E_ARG, "snpm_db_create: chr_regions[%d] = [%lld,%lld) outside the shard", c, (long long)s, (long long)e);
    }
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0)
        return fail(SNPM_E_CUDA, "snpm_db_create: no CUDA device (there is no CPU fallback)");
    if (device < 0 || device >= n_dev) return fail(SNPM_E_ARG, "snpm_db_create: device %d of %d", device, n_dev);
    SNPM_CUDA(cudaSetDevice(device));
    snpm_db *db = new snpm_db();
    db->device = device;
    db->n_rows = n_rows;
    db->n_acc = n_acc;
    db->n_words = (n_acc + 31) / 32;
    db->stride = (db->n_words + 1) & ~1;
    db->row0_global = row0_global;
    db->n_chr = n_chr;
    db->h_chr_regions.assign(chr_regions, chr_regions + 2 * size_t(n_chr));
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, device) == cudaSuccess) db->n_sm = p.multiProcessorCount;
    cudaError_t e = cudaStreamCreateWithFlags(&db->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete db; return fail(SNPM_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
    db->own_stream = true;
    const size_t pbytes = std::max<size_t>(size_t(n_rows) * db->stride * 8, 256);
    e = cudaMalloc(&db->d_packed, pbytes);
    if (e == cudaSuccess) e = cudaMalloc(&db->d_pos, std::max<size_t>(size_t(n_rows) * 4, 256));
    if (e == cudaSuccess) e = cudaMalloc(&db->d_chr_regions, std::max<size_t>(size_t(n_chr) * 16, 256));
    if (e != cudaSuccess) { snpm_db_destroy(db); return fail(SNPM_E_NOMEM, "snpm_db_create: cudaMalloc of the packed panel (%zu bytes): %s", pbytes, cudaGetErrorString(e)); }
    // every call is missing until loaded
    e = cudaMemsetAsync(db->d_packed, 0xFF, pbytes, db->stream);
    if (e == cudaSuccess && n_rows) e = cudaMemcpyAsync(db->d_pos, positions, size_t(n_rows) * 4, cudaMemcpyHostToDevice, db->stream);
    if (e == cudaSuccess && n_chr) e = cudaMemcpyAsync(db->d_chr_regions, chr_regions, size_t(n_chr) * 16, cudaMemcpyHostToDevice, db->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(db->stream);
    if (e != cudaSuccess) { snpm_db_destroy(db); return fail(SNPM_E_CUDA, "snpm_db_create: upload: %s", cudaGetErrorString(e)); }
    {   // coarse position index for the join: 2-4 rows per bucket (one table sector + one position sector per marker)
        int64_t span = 0;
        for (int c = 0; c < n_chr; ++c)
            if (chr_regions[2 * c + 1] > chr_regions[2 * c]) span += int64_t(positions[chr_regions[2 * c + 1] - 1]) + 1;
        int shift = 0;
        while (shift < 30 && (span >> shift) * 2 > std::max<int64_t>(n_rows, 1)) ++shift;           // (span >> shift) buckets <= n_rows / 2: 2-4 rows per bucket
        std::vector<int32_t> boff(size_t(n_chr) + 1, 0);
        int64_t total = 0;
        for (int c = 0; c < n_chr; ++c) {
            boff[size_t(c)] = int32_t(total);
            const int64_t last = chr_regions[2 * c + 1] > chr_regions[2 * c] ? int64_t(positions[chr_regions[2 * c + 1] - 1]) : -1;
            total += (last < 0 ? 0 : (last >> shift) + 1) + 1;                                  // + the closing entry
        }
        boff[size_t(n_chr)] = int32_t(total);
        if (total >= (int64_t(1) << 31)) { snpm_db_destroy(db); return fail(SNPM_E_ARG, "snpm_db_create: position index too large"); }
        db->bucket_shift = shift;
        e = cudaMalloc(&db->d_bucket, std::max<size_t>(size_t(total) * 4, 256));
        if (e == cudaSuccess) e = cudaMalloc(&db->d_bucket_off, (size_t(n_chr) + 1) * 4);
        if (e == cudaSuccess) e = cudaMemcpyAsync(db->d_bucket_off, boff.data(), (size_t(n_chr) + 1) * 4, cudaMemcpyHostToDevice, db->stream);
        if (e == cudaSuccess && total > 0) {
            k_build_buckets<<<int(ceil_div64(total, 256)), 256, 0, db->stream>>>(db->d_pos, db->d_chr_regions, n_chr, db->d_bucket_off, shift, db->d_bucket);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(db->stream);
        if (e != cudaSuccess) { snpm_db_destroy(db); return fail(SNPM_E_CUDA, "snpm_db_create: position index: %s", cudaGetErrorString(e)); }
    }
    {   // exact position index (bitmap + first row per word) when the genome fits 2^31 bits
        std::vector<int64_t> bm(size_t(n_chr) + 1, 0);
        int64_t bits = 0;
        for (int c = 0; c < n_chr; ++c) {
            bm[size_t(c)] = bits;
            const int64_t last = chr_regions[2 * c + 1] > chr_regions[2 * c] ? int64_t(positions[chr_regions[2 * c + 1] - 1]) : -1;
            bits += ((last + 1) + 63) / 64 * 64;
        }
        bm[size_t(n_chr)] = bits;
        static const bool no_bitmap = getenv("SNPM_JOIN_BITMAP") && !strcmp(getenv("SNPM_JOIN_BITMAP"), "0");      // measurement switch
        if (bits > 0 && bits <= (int64_t(1) << 31) && n_rows > 0 && !no_bitmap) {
            const int64_t n_words = bits / 64;
            e = cudaMalloc(&db->d_bitmap, size_t(n_words) * 8);
            if (e == cudaSuccess) e = cudaMalloc(&db->d_bm_first_row, size_t(n_words) * 4);
            if (e == cudaSuccess) e = cudaMalloc(&db->d_bm_off, (size_t(n_chr) + 1) * 8);
            if (e == cudaSuccess) e = cudaMemsetAsync(db->d_bitmap, 0, size_t(n_words) * 8, db->stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(db->d_bm_off, bm.data(), (size_t(n_chr) + 1) * 8, cudaMemcpyHostToDevice, db->stream);
            if (e == cudaSuccess) {
                k_bitmap_set<<<int(ceil_div64(n_rows, 256)), 256, 0, db->stream>>>(db->d_pos, db->d_chr_regions, n_chr, db->d_bm_off, n_rows, db->d_bitmap);
                k_bitmap_rows<<<int(ceil_div64(n_words, 256)), 256, 0, db->stream>>>(db->d_pos, db->d_chr_regions, n_chr, db->d_bm_off, n_words, db->d_bm_first_row);
                e = cudaGetLastError();
            }
            if (e == cudaSuccess) e = cudaStreamSynchronize(db->stream);
            if (e != cudaSuccess) {                            // the bitmap is an optimisation: fall back to the bucket search
                cudaGetLastError();
                if (db->d_bitmap) cudaFree(db->d_bitmap);
                if (db->d_bm_first_row) cudaFree(db->d_bm_first_row);
                if (db->d_bm_off) cudaFree(db->d_bm_off);
                db->d_bitmap = nullptr; db->d_bm_first_row = nullptr; db->d_bm_off = nullptr;
            }
        }
    }
    *out = db;
    return SNPM_OK;
}

int snpm_db_destroy(snpm_db *db) {
    if (!db) return SNPM_OK;
    cudaSetDevice(db->device);
    if (db->stream) cudaStreamSynchronize(db->stream);
    if (db->d_packed) cudaFree(db->d_packed);
    if (db->d_pos) cudaFree(db->d_pos);
    if (db->d_chr_regions) cudaFree(db->d_chr_regions);
    if (db->d_bucket) cudaFree(db->d_bucket);
    if (db->d_bucket_off) cudaFree(db->d_bucket_off);
    if (db->d_bitmap) cudaFree(db->d_bitmap);
    if (db->d_bm_first_row) cudaFree(db->d_bm_first_row);
    if (db->d_bm_off) cudaFree(db->d_bm_off);
    if (db->scratch_batch_) { snpm_batch_destroy(db->scratch_batch_); db->scratch_batch_ = nullptr; }
    if (db->own_stream && db->stream) cudaStreamDestroy(db->stream);
    delete db;
    return SNPM_OK;
}

int snpm_db_set_stream(snpm_db *db, void *cuda_stream) {
    if (!db) return fail(SNPM_E_ARG, "snpm_db_set_stream: db is NULL");
    SNPM_CUDA(cudaSetDevice(db->device));
    SNPM_CUDA(cudaStreamSynchronize(db->stream));
    if (db->own_stream) { cudaStreamDestroy(db->stream); db->own_stream = false; }
    if (cuda_stream) db->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    else { SNPM_CUDA(cudaStreamCreateWithFlags(&db->stream, cudaStreamNonBlocking)); db->own_stream = true; }
    return SNPM_OK;
}

int snpm_db_load_int8(snpm_db *db, int64_t row0, int64_t n, const int8_t *snps) {
    if (!db || row0 < 0 || n < 0 || row0 + n > db->n_rows || (n > 0 && !snps)) return fail(SNPM_E_ARG, "snpm_db_load_int8: bad row range");
    if (n == 0) return SNPM_OK;
    SNPM_CUDA(cudaSetDevice(db->device));
    const int64_t max_rows = std::max<int64_t>(1, (int64_t(256) << 20) / db->n_acc);    // 256 MB staging
    const size_t stage_bytes = (size_t(std::min(n, max_rows)) * db->n_acc + 255) & ~size_t(255);
    SNPM_TRY(db->scratch.ensure(stage_bytes + 256));
    int *d_bad = reinterpret_cast<int *>(static_cast<char *>(db->scratch.p) + stage_bytes);
    SNPM_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), db->stream));
    for (int64_t r = 0; r < n; r += max_rows) {
        const int64_t k = std::min(max_rows, n - r);
        SNPM_CUDA(cudaMemcpyAsync(db->scratch.p, snps + r * db->n_acc, size_t(k) * db->n_acc, cudaMemcpyHostToDevice, db->stream));
        k_pack_int8<<<grid_for(k * db->stride * 32, 256, db->n_sm), 256, 0, db->stream>>>(
            db->scratch.as<int8_t>(), k, db->n_acc, db->stride, db->d_packed + (row0 + r) * db->stride, d_bad);
        SNPM_KERNEL_CHECK();
        SNPM_CUDA(cudaStreamSynchronize(db->stream));
    }
    int bad = 0;
    SNPM_CUDA(cudaMemcpy(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost));
    if (bad > 0) return fail(SNPM_E_RANGE, "snpm_db_load_int8: %d genotype codes above 2 (codes are 0 ref, 1 alt, 2 het, negative = missing; makedb.py:59)", bad);
    return SNPM_OK;
}

int snpm_db_load_packed(snpm_db *db, int64_t row0, int64_t n, const uint64_t *packed) {
    if (!db || row0 < 0 || n < 0 || row0 + n > db->n_rows || (n > 0 && !packed)) return fail(SNPM_E_ARG, "snpm_db_load_packed: bad row range");
    if (n == 0) return SNPM_OK;
    SNPM_CUDA(cudaSetDevice(db->device));
    SNPM_CUDA(cudaMemcpyAsync(db->d_packed + row0 * db->stride, packed, size_t(n) * db->stride * 8, cudaMemcpyHostToDevice, db->stream));
    SNPM_CUDA(cudaStreamSynchronize(db->stream));
    return SNPM_OK;
}

int snpm_db_fill_synthetic(snpm_db *db, uint64_t seed) {
    if (!db) return fail(SNPM_E_ARG, "snpm_db_fill_synthetic: db is NULL");
    SNPM_CUDA(cudaSetDevice(db->device));
    if (db->n_rows == 0) return SNPM_OK;
    k_fill_synthetic<<<grid_for(db->n_rows * db->stride, 256, db->n_sm, 32), 256, 0, db->stream>>>(
        db->d_packed, db->n_rows, db->n_acc, db->stride, seed, db->row0_global);
    SNPM_KERNEL_CHECK();
    SNPM_CUDA(cudaStreamSynchronize(db->stream));
    return SNPM_OK;
}

int snpm_db_read_rows_int8(snpm_db *db, const int64_t *rows, int64_t k, int8_t *out) {
    if (!db || k < 0 || (k > 0 && (!rows || !out))) return fail(SNPM_E_ARG, "snpm_db_read_rows_int8: bad arguments");
    if (k == 0) return SNPM_OK;
    for (int64_t i = 0; i < k; ++i)
        if (rows[i] < 0 || rows[i] >= db->n_rows) return fail(SNPM_E_ARG, "snpm_db_read_rows_int8: row %lld out of range", (long long)rows[i]);
    SNPM_CUDA(cudaSetDevice(db->device));
    DevBuf d_rows, d_out;
    SNPM_TRY(d_rows.ensure(size_t(k) * 8));
    SNPM_TRY(d_out.ensure(size_t(k) * db->n_acc));
    SNPM_CUDA(cudaMemcpyAsync(d_rows.p, rows, size_t(k) * 8, cudaMemcpyHostToDevice, db->stream));
    k_unpack_rows<<<grid_for(k * db->n_acc, 256, db->n_sm), 256, 0, db->stream>>>(db->d_packed, db->stride, db->n_acc, d_rows.as<int64_t>(), k, d_out.as<int8_t>());
    SNPM_CUDA(cudaGetLastError());
    SNPM_CUDA(cudaMemcpyAsync(out, d_out.p, size_t(k) * db->n_acc, cudaMemcpyDeviceToHost, db->stream));
    SNPM_CUDA(cudaStreamSynchronize(db->stream));
    return SNPM_OK;
}

int snpm_db_read_packed(snpm_db *db, int64_t row0, int64_t n, uint64_t *out) {
    if (!db || row0 < 0 || n < 0 || row0 + n > db->n_rows || (n > 0 && !out)) return fail(SNPM_E_ARG, "snpm_db_read_packed: bad row range");
    if (n == 0) return SNPM_OK;
    SNPM_CUDA(cudaSetDevice(db->device));
    SNPM_CUDA(cudaMemcpyAsync(out, db->d_packed + row0 * db->stride, size_t(n) * db->stride * 8, cudaMemcpyDeviceToHost, db->stream));
    SNPM_CUDA(cudaStreamSynchronize(db->stream));
    return SNPM_OK;
}

int snpm_db_segregating_rows(snpm_db *db, const int32_t *acc_idx, int32_t n_sel, uint8_t *flags) {
    if (!db || n_sel < 0 || (n_sel > 0 && !acc_idx) || (db->n_rows > 0 && !flags)) return fail(SNPM_E_ARG, "snpm_db_segregating_rows: bad arguments");
    std::vector<uint32_t> sel(size_t(db->stride), 0u);
    for (int32_t i = 0; i < n_sel; ++i) {
        if (acc_idx[i] < 0 || acc_idx[i] >= db->n_acc) return fail(SNPM_E_ARG, "snpm_db_segregating_rows: accession index %d out of range", acc_idx[i]);
        sel[size_t(acc_idx[i] >> 5)] |= 1u << (acc_idx[i] & 31);
    }
    if (db->n_rows == 0) return SNPM_OK;
    SNPM_CUDA(cudaSetDevice(db->device));
    DevBuf d_sel, d_flags;
    SNPM_TRY(d_sel.ensure(size_t(db->stride) * 4));
    SNPM_TRY(d_flags.ensure(size_t(db->n_rows)));
    SNPM_CUDA(cudaMemcpyAsync(d_sel.p, sel.data(), size_t(db->stride) * 4, cudaMemcpyHostToDevice, db->stream));
    k_segregating_rows<<<grid_for(db->n_rows * 32, 256, db->n_sm, 32), 256, 0, db->stream>>>(db->d_packed, db->n_rows, db->stride,
                                                                                          d_sel.as<uint32_t>(), d_flags.as<uint8_t>());
    SNPM_CUDA(cudaGetLastError());
    SNPM_CUDA(cudaMemcpyAsync(flags, d_flags.p, size_t(db->n_rows), cudaMemcpyDeviceToHost, db->stream));
    SNPM_CUDA(cudaStreamSynchronize(db->stream));
    return SNPM_OK;
}

int snpm_db_read_columns(snpm_db *db, const int32_t *acc_idx, int32_t n_sel, int8_t *out) {
    if (!db || n_sel < 0 || (n_sel > 0 && (!acc_idx || (db->n_rows > 0 && !out)))) return fail(SNPM_E_ARG, "snpm_db_read_columns: bad arguments");
    for (int32_t i = 0; i < n_sel; ++i)
        if (acc_idx[i] < 0 || acc_idx[i] >= db->n_acc) return fail(SNPM_E_ARG, "snpm_db_read_columns: accession index %d out of range", acc_idx[i]);
    if (n_sel == 0 || db->n_rows == 0) return SNPM_OK;
    SNPM_CUDA(cudaSetDevice(db->device));
    DevBuf d_out;
    const int32_t per = std::min<int32_t>(n_sel, RC_MAX_COLS);
    SNPM_TRY(d_out.ensure(size_t(per) * size_t(db->n_rows)));
    for (int32_t c0 = 0; c0 < n_sel; c0 += RC_MAX_COLS) {
        ColumnSel sel;
        sel.n = std::min<int32_t>(RC_MAX_COLS, n_sel - c0);
        for (int32_t c = 0; c < RC_MAX_COLS; ++c) {
            const int32_t a = c < sel.n ? acc_idx[c0 + c] : 0;
            sel.word[c] = a >> 5;
            sel.bit[c] = a & 31;
        }
        k_read_columns<<<grid_for(db->n_rows, 256, db->n_sm, 32), 256, 0, db->stream>>>(db->d_packed, db->n_rows, db->stride, sel, d_out.as<int8_t>());
        SNPM_CUDA(cudaGetLastError());
        SNPM_CUDA(cudaMemcpyAsync(out + size_t(c0) * size_t(db->n_rows), d_out.p, size_t(sel.n) * size_t(db->n_rows), cudaMemcpyDeviceToHost, db->stream));
        SNPM_CUDA(cudaStreamSynchronize(db->stream));
    }
    return SNPM_OK;
}

int snpm_pair_match_counts(int device, const int64_t *idx1, const int64_t *idx2, int64_t m, const int32_t *chrom1, const int32_t *gt1, int64_t n1,
                           const int32_t *gt2, int64_t n2, int32_t n_chr, int64_t *common, int64_t *matches) {
    if (m < 0 || n1 < 0 || n2 < 0 || n_chr < 0 || (m > 0 && (!idx1 || !idx2 || !chrom1 || !gt1 || !gt2)) || (n_chr > 0 && (!common || !matches)))
        return fail(SNPM_E_ARG, "snpm_pair_match_counts: bad arguments");
    for (int64_t k = 0; k < m; ++k)
        if (idx1[k] < 0 || idx1[k] >= n1 || idx2[k] < 0 || idx2[k] >= n2) return fail(SNPM_E_ARG, "snpm_pair_match_counts: pair %lld points outside the samples", (long long)k);
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return fail(SNPM_E_CUDA, "snpm_pair_match_counts: no CUDA device (there is no CPU fallback)");
    if (n_chr == 0) return SNPM_OK;
    SNPM_CUDA(cudaSetDevice(device));
    DevBuf d_i1, d_i2, d_c1, d_g1, d_g2, d_cnt;
    std::vector<unsigned long long> cnt(size_t(2) * n_chr, 0ull);
    SNPM_TRY(d_cnt.ensure(size_t(2) * n_chr * 8));
    SNPM_CUDA(cudaMemset(d_cnt.p, 0, size_t(2) * n_chr * 8));
    if (m > 0) {
        SNPM_TRY(d_i1.ensure(size_t(m) * 8));
        SNPM_TRY(d_i2.ensure(size_t(m) * 8));
        SNPM_TRY(d_c1.ensure(size_t(n1) * 4));
        SNPM_TRY(d_g1.ensure(size_t(n1) * 4));
        SNPM_TRY(d_g2.ensure(size_t(n2) * 4));
        SNPM_CUDA(cudaMemcpy(d_i1.p, idx1, size_t(m) * 8, cudaMemcpyHostToDevice));
        SNPM_CUDA(cudaMemcpy(d_i2.p, idx2, size_t(m) * 8, cudaMemcpyHostToDevice));
        SNPM_CUDA(cudaMemcpy(d_c1.p, chrom1, size_t(n1) * 4, cudaMemcpyHostToDevice));
        SNPM_CUDA(cudaMemcpy(d_g1.p, gt1, size_t(n1) * 4, cudaMemcpyHostToDevice));
        SNPM_CUDA(cudaMemcpy(d_g2.p, gt2, size_t(n2) * 4, cudaMemcpyHostToDevice));
        const int grid = int(std::min<int64_t>(ceil_div64(m, 256), 1184));
        k_pair_counts<<<grid, 256>>>(d_i1.as<int64_t>(), d_i2.as<int64_t>(), m, d_c1.as<int32_t>(), d_g1.as<int32_t>(), d_g2.as<int32_t>(), n_chr,
                                     d_cnt.as<unsigned long long>());
        SNPM_CUDA(cudaGetLastError());
        SNPM_CUDA(cudaDeviceSynchronize());
    }
    SNPM_CUDA(cudaMemcpy(cnt.data(), d_cnt.p, size_t(2) * n_chr * 8, cudaMemcpyDeviceToHost));
    for (int32_t c = 0; c < n_chr; ++c) {
        common[c] = int64_t(cnt[size_t(c)]);
        matches[c] = int64_t(cnt[size_t(n_chr) + c]);
    }
    return SNPM_OK;
}

// ---- all-against-all pairsnp -----------------------------------------------------------------
int snpm_pair_matrix(int device, int64_t S, const int64_t *offsets, const int32_t *col, const uint8_t *cls, int32_t n_cls, int64_t K,
                     const int64_t *chr_start, int32_t C, int64_t chunk_markers, int32_t *common, int32_t *same, float *ms) {
    // every check runs on the host, before anything is allocated
    if (S < 1 || S > SNPM_PAIR_MAX_SAMPLES) return fail(SNPM_E_ARG, "snpm_pair_matrix: %lld samples; 1 to %d are allowed", (long long)S, SNPM_PAIR_MAX_SAMPLES);
    if (!offsets || n_cls < 1 || n_cls > 8 || K < 0 || C < 0 || !chr_start || chunk_markers < 0 || (C > 0 && (!common || !same)))
        return fail(SNPM_E_ARG, "snpm_pair_matrix: bad arguments");
    if (K > INT32_MAX) return fail(SNPM_E_ARG, "snpm_pair_matrix: %lld columns; column indices are int32", (long long)K);
    if (chr_start[0] != 0 || chr_start[C] != K) return fail(SNPM_E_ARG, "snpm_pair_matrix: chr_start must run from 0 to K = %lld", (long long)K);
    for (int32_t c = 0; c < C; ++c) {
        if (chr_start[c + 1] < chr_start[c]) return fail(SNPM_E_ARG, "snpm_pair_matrix: chr_start decreases at chromosome %d", c);
        if (chr_start[c + 1] - chr_start[c] >= (int64_t(1) << 31))
            return fail(SNPM_E_RANGE, "snpm_pair_matrix: chromosome %d has 2^31 columns or more; the counts are int32", c);
    }
    if (offsets[0] != 0) return fail(SNPM_E_ARG, "snpm_pair_matrix: offsets[0] must be 0");
    if (offsets[S] > 0 && (!col || !cls)) return fail(SNPM_E_ARG, "snpm_pair_matrix: bad arguments");
    for (int64_t s = 0; s < S; ++s) {
        if (offsets[s + 1] < offsets[s]) return fail(SNPM_E_ARG, "snpm_pair_matrix: offsets decrease at sample %lld", (long long)s);
        for (int64_t i = offsets[s]; i < offsets[s + 1]; ++i) {
            if (col[i] < 0 || col[i] >= K) return fail(SNPM_E_ARG, "snpm_pair_matrix: sample %lld: column %d is outside 0..K-1", (long long)s, col[i]);
            if (i > offsets[s] && col[i] <= col[i - 1]) return fail(SNPM_E_ARG, "snpm_pair_matrix: sample %lld: columns are not strictly ascending", (long long)s);
            if (cls[i] >= n_cls) return fail(SNPM_E_ARG, "snpm_pair_matrix: sample %lld: class %d is not below n_cls = %d", (long long)s, int(cls[i]), n_cls);
        }
    }
    const int64_t n = offsets[S];
    const int slots = n_cls <= 4 ? 4 : 8, mk = 128 / slots;
    const int m_blocks = int(ceil_div64(S, 64)), n_blocks = int(ceil_div64(S, OG_BN)), ld_out = n_blocks * OG_BN;
    const int64_t kb_bytes = int64_t(m_blocks) * OG_A_TILE + int64_t(n_blocks) * OG_B_TILE;
    int64_t widest = 0;
    for (int32_t c = 0; c < C; ++c) widest = std::max(widest, chr_start[c + 1] - chr_start[c]);
    int64_t step = chunk_markers > 0 ? chunk_markers : std::max<int64_t>(1, SNPM_PAIR_CHUNK_BYTES / kb_bytes) * mk;
    step = std::max<int64_t>(1, std::min(step, widest));
    const int64_t max_kb = ceil_div64(step, mk);
    const size_t cells = size_t(C) * size_t(S) * size_t(S);

    SNPM_CUDA(cudaSetDevice(device));
    int n_sm = 0;
    SNPM_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));
    struct Res {
        DevBuf off, col, cls, at, bt, ps, pc, same, common;
        cudaStream_t st = nullptr;
        std::vector<cudaEvent_t> ev;
        ~Res() {
            for (cudaEvent_t e : ev) cudaEventDestroy(e);
            if (st) cudaStreamDestroy(st);
        }
    } r;
    // events: call start / end, then per chunk of a ring of RING: start, operands ready, GEMM done
    constexpr int RING = 64;
    r.ev.assign(2 + 3 * RING, nullptr);
    for (cudaEvent_t &e : r.ev) SNPM_CUDA(cudaEventCreate(&e));
    SNPM_CUDA(cudaStreamCreateWithFlags(&r.st, cudaStreamNonBlocking));
    cudaStream_t st = r.st;
    SNPM_TRY(r.off.ensure(size_t(S + 1) * 8));
    SNPM_TRY(r.col.ensure(size_t(n) * 4));
    SNPM_TRY(r.cls.ensure(size_t(n)));
    SNPM_TRY(r.same.ensure(cells * 4));
    SNPM_TRY(r.common.ensure(cells * 4));
    if (K > 0) {
        SNPM_TRY(r.at.ensure(size_t(m_blocks) * max_kb * OG_A_TILE));
        SNPM_TRY(r.bt.ensure(size_t(n_blocks) * max_kb * OG_B_TILE));
        SNPM_TRY(r.ps.ensure(size_t(S) * ld_out * 4));
        SNPM_TRY(r.pc.ensure(size_t(S) * ld_out * 4));
    }
    const size_t smem = size_t(OG_STAGES) * (OG_A_TILE + OG_B_TILE) + 1024;
    SNPM_CUDA(smem_attr<k_onehot_gemm>(int(smem)));

    SNPM_CUDA(cudaEventRecord(r.ev[0], st));
    SNPM_CUDA(cudaMemcpyAsync(r.off.p, offsets, size_t(S + 1) * 8, cudaMemcpyHostToDevice, st));
    if (n > 0) {
        SNPM_CUDA(cudaMemcpyAsync(r.col.p, col, size_t(n) * 4, cudaMemcpyHostToDevice, st));
        SNPM_CUDA(cudaMemcpyAsync(r.cls.p, cls, size_t(n), cudaMemcpyHostToDevice, st));
    }
    if (cells) {
        SNPM_CUDA(cudaMemsetAsync(r.same.p, 0, cells * 4, st));
        SNPM_CUDA(cudaMemsetAsync(r.common.p, 0, cells * 4, st));
    }
    float t_expand = 0.f, t_gemm = 0.f;
    auto collect = [&](int q) -> int {                          // the times of the chunk in ring slot q
        cudaEvent_t *e = &r.ev[2 + 3 * q];
        float a = 0.f, b = 0.f;
        SNPM_CUDA(cudaEventSynchronize(e[2]));
        SNPM_CUDA(cudaEventElapsedTime(&a, e[0], e[1]));
        SNPM_CUDA(cudaEventElapsedTime(&b, e[1], e[2]));
        t_expand += a;
        t_gemm += b;
        return SNPM_OK;
    };
    const int warps = 8;
    const dim3 acc_grid(unsigned(ceil_div64(S, 256)), unsigned(S));
    int64_t chunk = 0;
    for (int32_t c = 0; c < C; ++c) {
        for (int64_t c0 = chr_start[c]; c0 < chr_start[c + 1]; c0 += step, ++chunk) {  // a chunk never spans two chromosomes
            const int64_t c1 = std::min(c0 + step, chr_start[c + 1]);
            const int32_t n_kb = int32_t(ceil_div64(c1 - c0, mk));
            const int q = int(chunk % RING);
            if (chunk >= RING) SNPM_TRY(collect(q));
            cudaEvent_t *e = &r.ev[2 + 3 * q];
            SNPM_CUDA(cudaEventRecord(e[0], st));
            SNPM_CUDA(cudaMemsetAsync(r.at.p, 0, size_t(m_blocks) * n_kb * OG_A_TILE, st));
            SNPM_CUDA(cudaMemsetAsync(r.bt.p, 0, size_t(n_blocks) * n_kb * OG_B_TILE, st));
            const unsigned eg = unsigned(ceil_div64(S, warps));
            if (slots == 4)
                k_pair_expand<4><<<eg, 32 * warps, 0, st>>>(r.off.as<int64_t>(), r.col.as<int32_t>(), r.cls.as<uint8_t>(), int32_t(S), int32_t(c0),
                                                           int32_t(c1), n_kb, r.at.as<unsigned char>(), r.bt.as<unsigned char>());
            else
                k_pair_expand<8><<<eg, 32 * warps, 0, st>>>(r.off.as<int64_t>(), r.col.as<int32_t>(), r.cls.as<uint8_t>(), int32_t(S), int32_t(c0),
                                                           int32_t(c1), n_kb, r.at.as<unsigned char>(), r.bt.as<unsigned char>());
            SNPM_KERNEL_CHECK();
            SNPM_CUDA(cudaEventRecord(e[1], st));
            OneHotGemmArgs g = {};
            g.a_tiled = r.at.as<unsigned char>(); g.b_tiled = r.bt.as<unsigned char>(); g.n_kb = n_kb; g.m_blocks = m_blocks; g.n_blocks = n_blocks;
            g.S = int32_t(S); g.out_score = r.ps.as<int32_t>(); g.out_ninfo = r.pc.as<int32_t>(); g.ld_out = ld_out;
            k_onehot_gemm<<<unsigned(std::min(m_blocks * n_blocks, n_sm)), OG_THREADS, smem, st>>>(g);
            SNPM_KERNEL_CHECK();
            SNPM_CUDA(cudaEventRecord(e[2], st));
            const size_t at = size_t(c) * S * S;
            k_pair_accumulate<<<acc_grid, 256, 0, st>>>(g.out_score, g.out_ninfo, ld_out, int32_t(S), r.same.as<int32_t>() + at, r.common.as<int32_t>() + at);
            SNPM_KERNEL_CHECK();
        }
    }
    for (int64_t k = std::max<int64_t>(0, chunk - RING); k < chunk; ++k) SNPM_TRY(collect(int(k % RING)));
    if (cells) {
        SNPM_CUDA(cudaMemcpyAsync(same, r.same.p, cells * 4, cudaMemcpyDeviceToHost, st));
        SNPM_CUDA(cudaMemcpyAsync(common, r.common.p, cells * 4, cudaMemcpyDeviceToHost, st));
    }
    SNPM_CUDA(cudaEventRecord(r.ev[1], st));
    SNPM_CUDA(cudaStreamSynchronize(st));
    if (ms) {
        ms[0] = t_expand;
        ms[1] = t_gemm;
        ms[2] = 0.f;
        SNPM_CUDA(cudaEventElapsedTime(&ms[2], r.ev[0], r.ev[1]));
    }
    return SNPM_OK;
}

int64_t snpm_db_n_rows(const snpm_db *db) { return db ? db->n_rows : -1; }
int32_t snpm_db_n_acc(const snpm_db *db) { return db ? db->n_acc : -1; }
int32_t snpm_db_row_words(const snpm_db *db) { return db ? db->stride : -1; }
int64_t snpm_db_packed_bytes(const snpm_db *db) { return db ? db->n_rows * int64_t(db->stride) * 8 : -1; }

// ---- batches --------------------------------------------------------------------------------------
// the sample offsets of every upload: S >= 1 samples, offsets from 0, non-decreasing, fewer than 2^31 - 2048 markers in all
static int check_offsets(const char *fn, int64_t S, const int64_t *offsets) {
    if (S < 1 || !offsets) return fail(SNPM_E_ARG, "%s: need at least one sample and its offsets", fn);
    if (offsets[0] != 0) return fail(SNPM_E_ARG, "%s: offsets[0] must be 0", fn);
    for (int64_t s = 0; s < S; ++s)
        if (offsets[s + 1] < offsets[s]) return fail(SNPM_E_ARG, "%s: offsets must be non-decreasing", fn);
    if (offsets[S] >= (int64_t(1) << 31) - 2048) return fail(SNPM_E_ARG, "%s: %lld markers exceed the 2^31 limit", fn, (long long)offsets[S]);
    return SNPM_OK;
}

// the end of every upload: the next run waits for the copies, and the results of the last run are no longer the batch's
static int upload_done(snpm_batch *b) {
    SNPM_CUDA(cudaEventRecord(b->ev_uploaded, b->copy_stream));
    b->ran = b->ran_windows = b->epilogue_done = false;
    return SNPM_OK;
}

static int batch_upload(snpm_batch *b, int64_t S, const int64_t *offsets, const int32_t *chrom, const int32_t *pos, const double *wei,
                        const uint16_t *wei_idx = nullptr, const double *table = nullptr, int32_t n_table = 0) {
    SNPM_TRY(check_offsets("batch", S, offsets));
    const int64_t n = offsets[S];
    if (n > 0 && (!chrom || !pos || (!wei && !wei_idx))) return fail(SNPM_E_ARG, "batch: NULL marker arrays");
    if (wei_idx && (!table || n_table < 1 || n_table > 65536)) return fail(SNPM_E_ARG, "batch: weight table must hold 1..65536 entries");
    b->S = S;
    b->n = n;
    b->grouped = false;
    b->coded = false;
    b->chunk_rows = b->chunk_rows_req;                           // latched: the buffers below and the next runs use this value
    b->h_off.assign(offsets, offsets + S + 1);
    int64_t nseg = 0;
    for (int64_t s = 0; s < S; ++s) nseg += ceil_div64(offsets[s + 1] - offsets[s], b->chunk_rows);
    b->nseg_cap = nseg;
    SNPM_TRY(b->d_off.ensure(size_t(S + 1) * 8));
    SNPM_TRY(b->d_chrom.ensure(size_t(n) * 4));
    SNPM_TRY(b->d_pos.ensure(size_t(n) * 4));
    SNPM_TRY(b->d_wei.ensure(size_t(n) * 24));
    // copies go to the batch's copy stream, after the last kernels that read the previous inputs
    cudaStream_t st = b->copy_stream;
    SNPM_CUDA(cudaStreamWaitEvent(st, b->ev_inputs_free, 0));
    SNPM_CUDA(cudaMemcpyAsync(b->d_off.p, offsets, size_t(S + 1) * 8, cudaMemcpyHostToDevice, st));
    if (n) {
        SNPM_CUDA(cudaMemcpyAsync(b->d_chrom.p, chrom, size_t(n) * 4, cudaMemcpyHostToDevice, st));
        SNPM_CUDA(cudaMemcpyAsync(b->d_pos.p, pos, size_t(n) * 4, cudaMemcpyHostToDevice, st));
        if (wei_idx) {
            SNPM_TRY(b->d_wei_idx.ensure(size_t(n) * 6));
            SNPM_TRY(b->d_wei_table.ensure(size_t(n_table) * 8));
            SNPM_CUDA(cudaMemcpyAsync(b->d_wei_idx.p, wei_idx, size_t(n) * 6, cudaMemcpyHostToDevice, st));
            SNPM_CUDA(cudaMemcpyAsync(b->d_wei_table.p, table, size_t(n_table) * 8, cudaMemcpyHostToDevice, st));
            k_expand_weights<<<int(ceil_div64(n * 3, 256)), 256, 0, st>>>(b->d_wei_idx.as<uint16_t>(), b->d_wei_table.as<double>(), n * 3,
                                                                         b->d_wei.as<double>());
            SNPM_KERNEL_CHECK();
        } else {
            SNPM_CUDA(cudaMemcpyAsync(b->d_wei.p, wei, size_t(n) * 24, cudaMemcpyHostToDevice, st));
        }
    }
    return upload_done(b);
}

static int batch_new(snpm_db *db, snpm_batch **out) {
    snpm_batch *b = new snpm_batch();
    b->db = db;
    for (int i = 0; i < SNPM_N_EVENTS; ++i) {
        if (cudaEventCreate(&b->ev[i]) != cudaSuccess) { snpm_batch_destroy(b); return fail(SNPM_E_CUDA, "cudaEventCreate failed"); }
    }
    if (cudaStreamCreateWithFlags(&b->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&b->ev_uploaded, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&b->ev_inputs_free, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreate(&b->ev_joined) != cudaSuccess) {
        snpm_batch_destroy(b);
        return fail(SNPM_E_CUDA, "snpm_batch_create: copy stream / events");
    }
    if (cudaMallocHost(reinterpret_cast<void **>(&b->h_status), 8 * sizeof(int)) != cudaSuccess) {
        snpm_batch_destroy(b);
        return fail(SNPM_E_NOMEM, "cudaMallocHost failed");
    }
    *out = b;
    return SNPM_OK;
}

int snpm_batch_create(snpm_db *db, int64_t n_samples, const int64_t *offsets, const int32_t *s_chrom_id, const int32_t *s_pos,
                      const double *wei, snpm_batch **out) {
    if (!db || !out) return fail(SNPM_E_ARG, "snpm_batch_create: NULL handle");
    *out = nullptr;
    SNPM_CUDA(cudaSetDevice(db->device));
    snpm_batch *b = nullptr;
    SNPM_TRY(batch_new(db, &b));
    int rc = batch_upload(b, n_samples, offsets, s_chrom_id, s_pos, wei);
    if (rc == SNPM_OK && cudaStreamSynchronize(b->copy_stream) != cudaSuccess) rc = fail(SNPM_E_CUDA, "snpm_batch_create: upload failed");
    if (rc != SNPM_OK) { snpm_batch_destroy(b); return rc; }
    *out = b;
    return SNPM_OK;
}

int snpm_batch_upload(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const int32_t *s_chrom_id, const int32_t *s_pos,
                      const double *wei) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_upload: NULL batch");
    SNPM_CUDA(cudaSetDevice(b->db->device));
    return batch_upload(b, n_samples, offsets, s_chrom_id, s_pos, wei);
}

int snpm_batch_upload_indexed(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const int32_t *s_chrom_id, const int32_t *s_pos,
                              const uint16_t *wei_idx, const double *table, int32_t n_table) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_upload_indexed: NULL batch");
    if (!wei_idx && offsets && n_samples >= 1 && offsets[n_samples] > 0) return fail(SNPM_E_ARG, "snpm_batch_upload_indexed: NULL weight indices");
    SNPM_CUDA(cudaSetDevice(b->db->device));
    return batch_upload(b, n_samples, offsets, s_chrom_id, s_pos, nullptr, wei_idx, table, n_table);
}


// ---- grouped order (k_score_grouped) ---------------------------------------------------------------
// Host-side preparation, done once per sample set at parse time: order every sample's markers by their weight triple.
int snpm_group_markers(int64_t n_samples, const int64_t *offsets, const int32_t *s_chrom_id, const int32_t *s_pos, const double *wei,
                       uint8_t *out_chrom, int32_t *out_pos, uint16_t *out_gid, int64_t *out_order, double *table, int32_t table_cap,
                       int32_t *n_table) {
    if (n_samples < 1 || !offsets || !n_table || !table || table_cap < 1) return fail(SNPM_E_ARG, "snpm_group_markers: bad arguments");
    const int64_t n = offsets[n_samples];
    if (n > 0 && (!s_chrom_id || !s_pos || !wei || !out_chrom || !out_pos || !out_gid)) return fail(SNPM_E_ARG, "snpm_group_markers: NULL marker arrays");
    struct Key {
        uint64_t a, b, c;
        bool operator==(const Key &o) const { return a == o.a && b == o.b && c == o.c; }
    };
    struct KeyHash {
        size_t operator()(const Key &k) const {
            uint64_t h = k.a * 0x9E3779B97F4A7C15ull;
            h ^= (k.b + 0x7F4A7C15ull) * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2);
            h ^= (k.c + 0x165667B19E3779F9ull) * 0xFF51AFD7ED558CCDull + (h << 6) + (h >> 2);
            return size_t(h ^ (h >> 29));
        }
    };
    std::unordered_map<Key, int32_t, KeyHash> ids;
    ids.reserve(4096);
    const int32_t cap = std::min<int32_t>(table_cap, 65536);
    std::vector<int32_t> gid(static_cast<size_t>(n));
    for (int64_t i = 0; i < n; ++i) {
        const double w0 = wei[3 * i], w1 = wei[3 * i + 1], w2 = wei[3 * i + 2];
        if (!(w0 >= 0.0 && w1 >= 0.0 && w2 >= 0.0) || std::isinf(w0) || std::isinf(w1) || std::isinf(w2))
            return fail(SNPM_E_ARG, "snpm_group_markers: weights must be finite and non-negative (marker %lld)", (long long)i);
        Key k;
        memcpy(&k.a, &w0, 8);
        memcpy(&k.b, &w1, 8);
        memcpy(&k.c, &w2, 8);
        if (w0 == 0.0) k.a = 0;        // -0.0 and 0.0 weigh the same
        if (w1 == 0.0) k.b = 0;
        if (w2 == 0.0) k.c = 0;
        auto it = ids.find(k);
        if (it == ids.end()) {
            const int32_t id = int32_t(ids.size());
            if (id >= cap) return fail(SNPM_E_RANGE, "snpm_group_markers: more than %d distinct weight triples", cap);
            table[3 * size_t(id)] = w0;
            table[3 * size_t(id) + 1] = w1;
            table[3 * size_t(id) + 2] = w2;
            it = ids.emplace(k, id).first;
        }
        gid[size_t(i)] = it->second;
        const int32_t c = s_chrom_id[i];
        if (c >= 255) return fail(SNPM_E_RANGE, "snpm_group_markers: chromosome id %d does not fit one byte", c);
    }
    const int32_t T = int32_t(ids.size());
    *n_table = T;
    // Order the triples so that along a sample's markers every class weight changes as rarely as possible (the kernel reads a
    // class counter out only when THAT class's weight changes): first by the called class (the one whose weight is 1.0, else
    // the largest), then by the remaining class with fewer distinct values, then by the other one.
    {
        std::vector<int32_t> called(static_cast<size_t>(T));
        std::vector<std::vector<double>> seen(9);
        for (int32_t t = 0; t < T; ++t) {
            const double *w = table + 3 * size_t(t);
            int c = 0;
            if (w[0] == 1.0) c = 0; else if (w[2] == 1.0) c = 2; else if (w[1] == 1.0) c = 1;
            else { c = 0; if (w[2] > w[c]) c = 2; if (w[1] > w[c]) c = 1; }
            called[size_t(t)] = c;
            for (int k = 0; k < 3; ++k) seen[size_t(3 * c + k)].push_back(w[k]);
        }
        int slow[3], fast[3];
        for (int c = 0; c < 3; ++c) {
            size_t distinct[3] = {0, 0, 0};
            for (int k = 0; k < 3; ++k) {
                auto &v = seen[size_t(3 * c + k)];
                std::sort(v.begin(), v.end());
                distinct[k] = size_t(std::unique(v.begin(), v.end()) - v.begin());
            }
            const int o1 = (c + 1) % 3, o2 = (c + 2) % 3;
            if (distinct[o1] <= distinct[o2]) { slow[c] = o1; fast[c] = o2; } else { slow[c] = o2; fast[c] = o1; }
        }
        std::vector<int32_t> perm(static_cast<size_t>(T)), rank(static_cast<size_t>(T));
        for (int32_t t = 0; t < T; ++t) perm[size_t(t)] = t;
        std::sort(perm.begin(), perm.end(), [&](int32_t x, int32_t y) {
            const int cx = called[size_t(x)], cy = called[size_t(y)];
            if (cx != cy) return cx < cy;
            const double *wx_ = table + 3 * size_t(x), *wy_ = table + 3 * size_t(y);
            if (wx_[cx] != wy_[cx]) return wx_[cx] > wy_[cx];
            if (wx_[slow[cx]] != wy_[slow[cx]]) return wx_[slow[cx]] > wy_[slow[cx]];
            if (wx_[fast[cx]] != wy_[fast[cx]]) return wx_[fast[cx]] > wy_[fast[cx]];
            return x < y;
        });
        std::vector<double> sorted(static_cast<size_t>(T) * 3);
        for (int32_t r = 0; r < T; ++r) {
            rank[size_t(perm[size_t(r)])] = r;
            memcpy(&sorted[3 * size_t(r)], table + 3 * size_t(perm[size_t(r)]), 24);
        }
        memcpy(table, sorted.data(), size_t(T) * 24);
        for (int64_t i = 0; i < n; ++i) gid[size_t(i)] = rank[size_t(gid[size_t(i)])];
    }
    std::vector<int64_t> cnt(static_cast<size_t>(T) + 1);
    for (int64_t s = 0; s < n_samples; ++s) {
        const int64_t b0 = offsets[s], b1 = offsets[s + 1];
        std::fill(cnt.begin(), cnt.end(), 0);
        for (int64_t i = b0; i < b1; ++i) ++cnt[size_t(gid[size_t(i)]) + 1];
        for (int32_t t = 0; t < T; ++t) cnt[size_t(t) + 1] += cnt[size_t(t)];
        for (int64_t i = b0; i < b1; ++i) {                       // stable: position order is kept inside a group
            const int32_t g = gid[size_t(i)];
            const int64_t o = b0 + cnt[size_t(g)]++;
            out_chrom[o] = s_chrom_id[i] < 0 ? uint8_t(255) : uint8_t(s_chrom_id[i]);
            out_pos[o] = s_pos[i];
            out_gid[o] = uint16_t(g);
            if (out_order) out_order[o] = i;
        }
    }
    return SNPM_OK;
}

static int upload_grouped(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint8_t *chrom_u8, const int32_t *s_pos,
                          const uint32_t *packed_cp, const uint16_t *gid, const double *table, int32_t n_table,
                          const uint16_t *run_gid = nullptr, const uint32_t *run_end = nullptr, int64_t n_runs = 0) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_upload_grouped: NULL batch");
    snpm_db *db = b->db;
    SNPM_TRY(check_offsets("snpm_batch_upload_grouped", n_samples, offsets));
    const int64_t n = offsets[n_samples];
    if (n > 0 && ((!gid && !run_gid) || (!packed_cp && (!chrom_u8 || !s_pos)))) return fail(SNPM_E_ARG, "snpm_batch_upload_grouped: NULL marker arrays");
    if (run_gid && n > 0) {
        if (!run_end || n_runs < 1 || n_runs > n) return fail(SNPM_E_ARG, "snpm_batch_upload_grouped_runs: need 1..n runs");
        if (int64_t(run_end[n_runs - 1]) != n || run_end[0] == 0) return fail(SNPM_E_ARG, "snpm_batch_upload_grouped_runs: the runs must cover markers 0..n");
    }
    if (!table || n_table < 1 || n_table > 65536) return fail(SNPM_E_ARG, "snpm_batch_upload_grouped: weight table must hold 1..65536 triples");
    std::vector<double> t4(size_t(n_table) * 4);
    for (int32_t t = 0; t < n_table; ++t) {
        const double w0 = table[3 * size_t(t)], w1 = table[3 * size_t(t) + 1], w2 = table[3 * size_t(t) + 2];
        if (!(w0 >= 0.0 && w1 >= 0.0 && w2 >= 0.0) || std::isinf(w0) || std::isinf(w1) || std::isinf(w2))
            return fail(SNPM_E_ARG, "snpm_batch_upload_grouped: weights must be finite and non-negative (triple %d)", t);
        t4[4 * size_t(t)] = w0;            // (w_ref, w_alt, w_het, 0): the order of pair_w
        t4[4 * size_t(t) + 1] = w2;
        t4[4 * size_t(t) + 2] = w1;
        t4[4 * size_t(t) + 3] = 0.0;
    }
    SNPM_CUDA(cudaSetDevice(db->device));
    b->S = n_samples;
    b->n = n;
    b->grouped = true;
    b->coded = false;
    b->pending_expand = 0;
    b->n_gtable = n_table;
    b->gchunk = b->gchunk_req;                                  // latched: the buffers below and the next runs use this value
    b->h_off.assign(offsets, offsets + n_samples + 1);
    int64_t nseg = 0;                                           // bound by the markers alone (a repeated marker matches its row twice)
    for (int64_t s = 0; s < n_samples; ++s) nseg += ceil_div64(offsets[s + 1] - offsets[s], b->gchunk);
    b->nseg_cap = nseg;
    SNPM_TRY(b->d_off.ensure(size_t(n_samples + 1) * 8));
    SNPM_TRY(b->d_chrom8.ensure(size_t(n)));
    SNPM_TRY(b->d_chrom.ensure(size_t(n) * 4));
    SNPM_TRY(b->d_pos.ensure(size_t(n) * 4));
    SNPM_TRY(b->d_gid.ensure(size_t(n) * 2));
    SNPM_TRY(b->d_gtable.ensure(size_t(n_table) * 32));
    cudaStream_t st = b->copy_stream;
    SNPM_CUDA(cudaStreamWaitEvent(st, b->ev_inputs_free, 0));
    SNPM_CUDA(cudaMemcpyAsync(b->d_off.p, offsets, size_t(n_samples + 1) * 8, cudaMemcpyHostToDevice, st));
    // the table is staged in a buffer the batch owns so that the caller's (and this function's) copy may go away
    b->h_gtable.assign(t4.begin(), t4.end());
    SNPM_CUDA(cudaMemcpyAsync(b->d_gtable.p, b->h_gtable.data(), size_t(n_table) * 32, cudaMemcpyHostToDevice, st));
    if (n) {
        if (run_gid) {
            const size_t bad_off = (size_t(n_runs) * 6 + 15) & ~size_t(15);
            SNPM_TRY(b->d_runs.ensure(bad_off + 16));
            uint32_t *d_end = b->d_runs.as<uint32_t>();
            uint16_t *d_rg = reinterpret_cast<uint16_t *>(d_end + n_runs);
            b->d_runs_bad = reinterpret_cast<int *>(static_cast<char *>(b->d_runs.p) + bad_off);
            SNPM_CUDA(cudaMemsetAsync(b->d_runs_bad, 0, sizeof(int), st));
            SNPM_CUDA(cudaMemcpyAsync(d_end, run_end, size_t(n_runs) * 4, cudaMemcpyHostToDevice, st));
            SNPM_CUDA(cudaMemcpyAsync(d_rg, run_gid, size_t(n_runs) * 2, cudaMemcpyHostToDevice, st));
            b->pending_expand |= 1;
            b->pending_runs = n_runs;
        } else {
            b->d_runs_bad = nullptr;
            SNPM_CUDA(cudaMemcpyAsync(b->d_gid.p, gid, size_t(n) * 2, cudaMemcpyHostToDevice, st));
        }
        if (packed_cp) {
            SNPM_TRY(b->d_wei_idx.ensure(size_t(n) * 4));      // staging of the packed words (the buffer is free in grouped mode)
            SNPM_CUDA(cudaMemcpyAsync(b->d_wei_idx.p, packed_cp, size_t(n) * 4, cudaMemcpyHostToDevice, st));
            b->pending_expand |= 2;
        } else {
            SNPM_CUDA(cudaMemcpyAsync(b->d_chrom8.p, chrom_u8, size_t(n), cudaMemcpyHostToDevice, st));
            SNPM_CUDA(cudaMemcpyAsync(b->d_pos.p, s_pos, size_t(n) * 4, cudaMemcpyHostToDevice, st));
            b->pending_expand |= 4;
        }
    }
    return upload_done(b);
}

int snpm_batch_upload_grouped(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint8_t *chrom_u8, const int32_t *s_pos,
                              const uint16_t *gid, const double *table, int32_t n_table) {
    return upload_grouped(b, n_samples, offsets, chrom_u8, s_pos, nullptr, gid, table, n_table);
}

int snpm_batch_upload_grouped_packed(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint32_t *chrom_pos, const uint16_t *gid,
                                     const double *table, int32_t n_table) {
    return upload_grouped(b, n_samples, offsets, nullptr, nullptr, chrom_pos, gid, table, n_table);
}

int snpm_batch_upload_grouped_runs(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint32_t *chrom_pos, const uint16_t *run_gid,
                                   const uint32_t *run_end, int64_t n_runs, const double *table, int32_t n_table) {
    return upload_grouped(b, n_samples, offsets, nullptr, nullptr, chrom_pos, nullptr, table, n_table, run_gid, run_end, n_runs);
}

static int upload_coded(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint32_t *chrom_pos, const uint16_t *codes,
                        const uint32_t *codes32, const double *wtable, int32_t n_wtable) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_upload_coded: NULL batch");
    if (codes32 && n_wtable > 1024) return fail(SNPM_E_ARG, "snpm_batch_upload_coded32: three codes share one word only up to 1024 weight values (%d given)", n_wtable);
    snpm_db *db = b->db;
    SNPM_TRY(check_offsets("snpm_batch_upload_coded", n_samples, offsets));
    const int64_t n = offsets[n_samples];
    if (n > 0 && (!chrom_pos || (!codes && !codes32))) return fail(SNPM_E_ARG, "snpm_batch_upload_coded: NULL marker arrays");
    if (!wtable || n_wtable < 1 || n_wtable > 65536) return fail(SNPM_E_ARG, "snpm_batch_upload_coded: the weight table must hold 1..65536 values");
    for (int32_t t = 0; t < n_wtable; ++t)
        if (!(wtable[t] >= 0.0) || std::isinf(wtable[t])) return fail(SNPM_E_ARG, "snpm_batch_upload_coded: weights must be finite and non-negative (entry %d)", t);
    // segment length unless the caller chose one: 320 rows balance the seven teams of a CTA best on one-slice panels (1135
    // accessions: 0.250 ms against 0.317 / 0.326 at 400 / 496 rows); on wider panels, where the eight teams of a CTA score eight
    // slices of the SAME segment, longer segments only save partial sums and their combine (20 000 accessions: 1.88 ms per step
    // at 496 rows against 2.08 at 320)
    if (!b->gchunk_set) b->gchunk_req = db->stride > G2_WX ? G2_MAX_CHUNK : 320;
    if (b->gchunk_req % GR_BLOCK || b->gchunk_req > G2_MAX_CHUNK)
        return fail(SNPM_E_ARG, "snpm_batch_upload_coded: the group chunk must be a multiple of %d and at most %d rows (it is %d)", GR_BLOCK, G2_MAX_CHUNK, b->gchunk_req);
    SNPM_CUDA(cudaSetDevice(db->device));
    b->S = n_samples;
    b->n = n;
    b->grouped = true;
    b->coded = true;
    b->codes_packed = codes32 != nullptr;
    b->pending_expand = 2;                                      // packed words -> chromosome ids + positions at the head of the run
    b->d_runs_bad = nullptr;
    b->n_wtable = n_wtable;
    int bits = 1;
    while ((1 << bits) < n_wtable) ++bits;
    b->code_bits = bits;
    b->key_bits = 3 * bits + 2;
    b->gchunk = b->gchunk_req;
    b->h_off.assign(offsets, offsets + n_samples + 1);
    int64_t nseg = 0;
    std::vector<int32_t> tile_first(size_t(n_samples) + 1), tile_sample;
    for (int64_t s = 0; s < n_samples; ++s) {
        const int64_t ns = offsets[s + 1] - offsets[s];
        nseg += ceil_div64(ns, b->gchunk);
        tile_first[size_t(s)] = int32_t(tile_sample.size());
        for (int64_t t = 0; t < ceil_div64(ns, RS_TILE); ++t) tile_sample.push_back(int32_t(s));
    }
    tile_first[size_t(n_samples)] = int32_t(tile_sample.size());
    b->nseg_cap = nseg;
    b->n_sort_tiles = int64_t(tile_sample.size());
    const size_t key_bytes = b->key_bits <= 32 ? 4 : 8;
    SNPM_TRY(b->d_off.ensure(size_t(n_samples + 1) * 8));
    SNPM_TRY(b->d_chrom.ensure(size_t(n) * 4));
    SNPM_TRY(b->d_pos.ensure(size_t(n) * 4));
    SNPM_TRY(b->d_wei_idx.ensure(size_t(n) * 4));               // staging of the packed words
    SNPM_TRY(b->d_codes.ensure(size_t(n) * 6));
    SNPM_TRY(b->d_wtable.ensure(size_t(n_wtable) * 8));
    SNPM_TRY(b->d_key_a.ensure(size_t(n) * key_bytes));
    SNPM_TRY(b->d_pair_db_tmp.ensure(size_t(n) * 4));
    SNPM_TRY(b->d_pair_s_tmp.ensure(size_t(n) * 4));
    SNPM_TRY(b->d_tile_sample.ensure(std::max<size_t>(tile_sample.size(), 1) * 4));
    SNPM_TRY(b->d_tile_first.ensure(size_t(n_samples + 1) * 4));
    SNPM_TRY(b->d_tile_hist.ensure(std::max<size_t>(tile_sample.size(), 1) * (size_t(GH_MAX_GROUPS) * 4 + 8)));      // id counts per tile + the tile ranges
    // block words of every segment, their cost estimates, the bucket counts of the work order (zeroed together), then (bucket, rank)
    SNPM_TRY(b->d_blk_chg.ensure(size_t(std::max<int64_t>(nseg, 1)) * (size_t(b->gchunk / GR_BLOCK) * 8 + 12) + size_t(SO_BUCKETS) * 4 + 16));
    SNPM_TRY(b->d_seg_order.ensure(size_t(std::max<int64_t>(nseg, 1)) * 16));
    SNPM_TRY(b->d_work_counter.ensure(256));
    SNPM_TRY(b->d_hash.ensure(size_t(n_samples) * GH_SLOTS * 8));
    SNPM_TRY(b->d_slot_gid.ensure(size_t(n_samples) * GH_SLOTS * 2));
    SNPM_TRY(b->d_ngroups.ensure(size_t(n_samples) * 4));
    SNPM_TRY(b->d_group_overflow.ensure(size_t(n_samples) * 4));
    SNPM_TRY(b->d_gkeys.ensure(size_t(n_samples) * GH_MAX_GROUPS * key_bytes));
    SNPM_TRY(b->d_gw.ensure(size_t(n_samples) * GH_MAX_GROUPS * 32));
    SNPM_TRY(b->d_goff.ensure(size_t(n_samples) * (GH_MAX_GROUPS + 1) * 4));
    SNPM_TRY(b->d_gid.ensure(size_t(n) * 2));
    cudaStream_t st = b->copy_stream;
    SNPM_CUDA(cudaStreamWaitEvent(st, b->ev_inputs_free, 0));
    // small host-built tables are staged in buffers the batch owns (the copies are asynchronous)
    b->h_gtable.assign(wtable, wtable + n_wtable);
    b->h_tiles.assign(tile_first.begin(), tile_first.end());
    b->h_tiles.insert(b->h_tiles.end(), tile_sample.begin(), tile_sample.end());
    SNPM_CUDA(cudaMemcpyAsync(b->d_off.p, offsets, size_t(n_samples + 1) * 8, cudaMemcpyHostToDevice, st));
    SNPM_CUDA(cudaMemcpyAsync(b->d_wtable.p, b->h_gtable.data(), size_t(n_wtable) * 8, cudaMemcpyHostToDevice, st));
    SNPM_CUDA(cudaMemcpyAsync(b->d_tile_first.p, b->h_tiles.data(), size_t(n_samples + 1) * 4, cudaMemcpyHostToDevice, st));
    if (!tile_sample.empty())
        SNPM_CUDA(cudaMemcpyAsync(b->d_tile_sample.p, b->h_tiles.data() + n_samples + 1, tile_sample.size() * 4, cudaMemcpyHostToDevice, st));
    if (n) {
        SNPM_CUDA(cudaMemcpyAsync(b->d_wei_idx.p, chrom_pos, size_t(n) * 4, cudaMemcpyHostToDevice, st));
        if (codes32) SNPM_CUDA(cudaMemcpyAsync(b->d_codes.p, codes32, size_t(n) * 4, cudaMemcpyHostToDevice, st));
        else SNPM_CUDA(cudaMemcpyAsync(b->d_codes.p, codes, size_t(n) * 6, cudaMemcpyHostToDevice, st));
    }
    return upload_done(b);
}

int snpm_batch_upload_coded(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint32_t *chrom_pos, const uint16_t *codes,
                            const double *wtable, int32_t n_wtable) {
    return upload_coded(b, n_samples, offsets, chrom_pos, codes, nullptr, wtable, n_wtable);
}

int snpm_batch_upload_coded32(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint32_t *chrom_pos, const uint32_t *codes32,
                              const double *wtable, int32_t n_wtable) {
    return upload_coded(b, n_samples, offsets, chrom_pos, nullptr, codes32, wtable, n_wtable);
}

int snpm_batch_coded_timings(snpm_batch *b, float *ms, int n) {
    if (!b || !ms || n < 4) return fail(SNPM_E_ARG, "snpm_batch_coded_timings: need room for 4 floats");
    if (!b->coded || !b->ran) return fail(SNPM_E_STATE, "snpm_batch_coded_timings: run a coded batch first");
    SNPM_CUDA(cudaSetDevice(b->db->device));
    SNPM_CUDA(cudaStreamSynchronize(b->db->stream));
    for (int i = 0; i < n; ++i) ms[i] = 0.f;
    cudaEventElapsedTime(&ms[0], b->ev[SNPM_EV_START], b->ev_joined);
    cudaEventElapsedTime(&ms[1], b->ev_joined, b->ev[SNPM_EV_JOIN]);
    cudaEventElapsedTime(&ms[2], b->ev[SNPM_EV_JOIN], b->ev[SNPM_EV_SCORE]);
    cudaEventElapsedTime(&ms[3], b->ev[SNPM_EV_SCORE], b->ev[SNPM_EV_COMBINE]);
    return SNPM_OK;
}

int snpm_pack_markers(int64_t n, const uint8_t *chrom_u8, const int32_t *pos, uint32_t *out) {
    if (n < 0 || (n > 0 && (!chrom_u8 || !pos || !out))) return fail(SNPM_E_ARG, "snpm_pack_markers: bad arguments");
    for (int64_t i = 0; i < n; ++i) {
        const uint32_t c = chrom_u8[i] == 255 ? 31u : uint32_t(chrom_u8[i]);
        if ((chrom_u8[i] != 255 && c > 30u) || pos[i] < 0 || pos[i] >= (1 << 27))
            return fail(SNPM_E_RANGE, "snpm_pack_markers: marker %lld (chromosome id %u, position %d) does not fit 5 + 27 bits", (long long)i, c, pos[i]);
        out[i] = (c << 27) | uint32_t(pos[i]);
    }
    return SNPM_OK;
}

int snpm_pack_coded(int64_t n, const int32_t *chrom_id, const int32_t *pos, const uint16_t *codes, uint32_t *chrom_pos, uint32_t *codes32) {
    if (n < 0 || (n > 0 && (!chrom_id || !pos || !chrom_pos || (codes32 && !codes)))) return fail(SNPM_E_ARG, "snpm_pack_coded: bad arguments");
    uint32_t bad = 0u;
    for (int64_t i = 0; i < n; ++i) {
        const int32_t c = chrom_id[i], p = pos[i];
        bad |= uint32_t(c > 30) | uint32_t(p < 0) | uint32_t(p >= (1 << 27));
        chrom_pos[i] = ((c < 0 ? 31u : uint32_t(c)) << 27) | (uint32_t(p) & ((1u << 27) - 1u));
    }
    if (codes32)
        for (int64_t i = 0; i < n; ++i) {
            const uint32_t a = codes[3 * i], h = codes[3 * i + 1], t = codes[3 * i + 2];
            bad |= uint32_t((a | h | t) > 1023u);
            codes32[i] = a | (h << 10) | (t << 20);
        }
    if (bad) return fail(SNPM_E_RANGE, "snpm_pack_coded: a chromosome id above 30, a position outside 27 bits or a code above 1023");
    return SNPM_OK;
}

int snpm_batch_guard_counts(snpm_batch *b, int32_t *counts) {
    if (!b || !counts) return fail(SNPM_E_ARG, "snpm_batch_guard_counts: NULL argument");
    if (!b->grouped) { for (int64_t s = 0; s < b->rangen(); ++s) counts[s] = 0; return SNPM_OK; }
    if (!b->epilogue_done) return fail(SNPM_E_STATE, "snpm_batch_guard_counts: run the epilogue first");
    if (b->rangen() == 0) return SNPM_OK;
    SNPM_CUDA(cudaSetDevice(b->db->device));
    SNPM_CUDA(cudaMemcpyAsync(counts, b->d_guard.as<int32_t>() + b->range0(), size_t(b->rangen()) * 4, cudaMemcpyDeviceToHost, b->db->stream));
    SNPM_CUDA(cudaStreamSynchronize(b->db->stream));
    return SNPM_OK;
}

int snpm_batch_set_result_range(snpm_batch *b, int64_t first_sample, int64_t n_samples) {
    if (!b || first_sample < 0 || n_samples < -1) return fail(SNPM_E_ARG, "snpm_batch_set_result_range: bad range");
    b->res0 = first_sample;
    b->resn = n_samples;
    return SNPM_OK;
}

int snpm_batch_set_track_pairs(snpm_batch *b, int on) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_set_track_pairs: NULL batch");
    b->track_pairs = on != 0;
    return SNPM_OK;
}

int snpm_batch_set_chunk_rows(snpm_batch *b, int32_t rows) {
    if (!b || rows < 1 || rows > 1000000) return fail(SNPM_E_ARG, "snpm_batch_set_chunk_rows: 1..1000000 rows");
    b->chunk_rows_req = rows;
    return SNPM_OK;
}

int snpm_batch_set_group_chunk(snpm_batch *b, int32_t rows) {
    if (!b || rows < 16 || rows > GR_MAX_CHUNK || rows % 8) return fail(SNPM_E_ARG, "snpm_batch_set_group_chunk: 16..%d rows, a multiple of 8", GR_MAX_CHUNK);
    b->gchunk_req = rows;
    b->gchunk_set = true;
    return SNPM_OK;
}

static void ipc_close_peers(snpm_batch *b);

int snpm_batch_destroy(snpm_batch *b) {
    if (!b) return SNPM_OK;
    cudaSetDevice(b->db->device);
    cudaStreamSynchronize(b->db->stream);
    if (b->copy_stream) { cudaStreamSynchronize(b->copy_stream); cudaStreamDestroy(b->copy_stream); }
    if (b->ev_uploaded) cudaEventDestroy(b->ev_uploaded);
    if (b->ev_inputs_free) cudaEventDestroy(b->ev_inputs_free);
    if (b->ev_joined) cudaEventDestroy(b->ev_joined);
    if (b->ev_fork) cudaEventDestroy(b->ev_fork);
    if (b->ev_join) cudaEventDestroy(b->ev_join);
    for (int i = 0; i < SNPM_N_EVENTS; ++i)
        if (b->ev[i]) cudaEventDestroy(b->ev[i]);
    if (b->h_status) cudaFreeHost(b->h_status);
    if (b->h_tail) cudaFreeHost(b->h_tail);
    if (b->ev_fetched) cudaEventDestroy(b->ev_fetched);
    if (b->ev_results) cudaEventDestroy(b->ev_results);
    ipc_close_peers(b);
    delete b;
    return SNPM_OK;
}

int snpm_batch_set_row_filter(snpm_batch *b, const int64_t *sorted_rows, int64_t n) {
    if (!b || n < 0) return fail(SNPM_E_ARG, "snpm_batch_set_row_filter: bad arguments");
    for (int64_t i = 1; i < n; ++i)
        if (sorted_rows[i] <= sorted_rows[i - 1]) return fail(SNPM_E_ARG, "snpm_batch_set_row_filter: rows must be strictly ascending");
    SNPM_CUDA(cudaSetDevice(b->db->device));
    // NULL clears the filter; a non-NULL list of n = 0 rows is an EMPTY filter that keeps no pair (the reference's
    // filter_pos_ix of length 0 leaves no common SNP, snpmatch.py:211-216)
    b->has_filter = sorted_rows != nullptr;
    b->n_filter = b->has_filter ? n : 0;
    SNPM_TRY(b->d_filter.ensure(size_t(std::max<int64_t>(n, 1)) * 8));
    if (b->has_filter && n) {
        SNPM_CUDA(cudaMemcpyAsync(b->d_filter.p, sorted_rows, size_t(n) * 8, cudaMemcpyHostToDevice, b->db->stream));
        SNPM_CUDA(cudaStreamSynchronize(b->db->stream));
    }
    return SNPM_OK;
}

int snpm_batch_set_segregation_filter(snpm_batch *b, const uint32_t *sel, int64_t S, int32_t words) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_set_segregation_filter: NULL batch");
    if (!sel) {
        b->has_seg = false;
        b->seg_S = 0;
        return SNPM_OK;
    }
    snpm_db *db = b->db;
    if (S < 1 || words != db->stride)
        return fail(SNPM_E_ARG, "snpm_batch_set_segregation_filter: need S >= 1 selections of snpm_db_row_words() = %d words (got S = %lld, %d words)",
                    db->stride, (long long)S, words);
    std::vector<int32_t> off(size_t(S) + 1, 0);
    std::vector<uint32_t> pairs;                                // (word, mask) of every touched word, sample by sample
    for (int64_t s = 0; s < S; ++s) {
        for (int32_t w = 0; w < words; ++w) {
            const uint32_t m = sel[size_t(s) * words + w];
            const int64_t first = int64_t(w) * 32;
            const uint32_t valid = first >= db->n_acc ? 0u : (db->n_acc - first >= 32 ? 0xffffffffu : (1u << (db->n_acc - first)) - 1u);
            if (m & ~valid) return fail(SNPM_E_ARG, "snpm_batch_set_segregation_filter: sample %lld selects accessions beyond the panel's %d", (long long)s, db->n_acc);
            if (m) {
                pairs.push_back(uint32_t(w));
                pairs.push_back(m);
            }
        }
        if (pairs.size() / 2 > size_t(INT32_MAX)) return fail(SNPM_E_ARG, "snpm_batch_set_segregation_filter: selections too large");
        off[size_t(s) + 1] = int32_t(pairs.size() / 2);
    }
    SNPM_CUDA(cudaSetDevice(db->device));
    SNPM_TRY(b->d_segsel.ensure(std::max<size_t>(pairs.size(), 2) * 4));
    SNPM_TRY(b->d_segsel_off.ensure(off.size() * 4));
    // the copies queue behind the runs that may still read the previous selections; the host arrays are gone on return
    if (!pairs.empty()) SNPM_CUDA(cudaMemcpyAsync(b->d_segsel.p, pairs.data(), pairs.size() * 4, cudaMemcpyHostToDevice, db->stream));
    SNPM_CUDA(cudaMemcpyAsync(b->d_segsel_off.p, off.data(), off.size() * 4, cudaMemcpyHostToDevice, db->stream));
    SNPM_CUDA(cudaStreamSynchronize(db->stream));
    b->has_seg = true;
    b->seg_S = S;
    return SNPM_OK;
}

int snpm_batch_count_flagged_pairs(snpm_batch *b, const uint8_t *flags, int64_t *counts) {
    if (!b || !counts || (b->n > 0 && !flags)) return fail(SNPM_E_ARG, "snpm_batch_count_flagged_pairs: bad arguments");
    if (!b->ran) return fail(SNPM_E_STATE, "snpm_batch_count_flagged_pairs: run the batch first");
    snpm_db *db = b->db;
    SNPM_CUDA(cudaSetDevice(db->device));
    cudaStream_t st = db->stream;
    SNPM_TRY(b->d_flag_counts.ensure(size_t(b->S) * 8));
    SNPM_CUDA(cudaMemsetAsync(b->d_flag_counts.p, 0, size_t(b->S) * 8, st));
    if (b->n > 0) {
        SNPM_TRY(b->d_flags.ensure(size_t(b->n)));
        SNPM_CUDA(cudaMemcpyAsync(b->d_flags.p, flags, size_t(b->n), cudaMemcpyHostToDevice, st));
        k_count_flagged_pairs<<<int(ceil_div64(b->n, 256)), 256, 0, st>>>(b->d_match_row.as<int32_t>(), b->d_flags.as<uint8_t>(), b->n,
                                                                          b->d_off.as<int64_t>(), b->S, b->d_flag_counts.as<unsigned long long>());
        SNPM_KERNEL_CHECK();
    }
    SNPM_CUDA(cudaMemcpyAsync(counts, b->d_flag_counts.p, size_t(b->S) * 8, cudaMemcpyDeviceToHost, st));
    SNPM_CUDA(cudaStreamSynchronize(st));
    return SNPM_OK;
}

// join + compaction + per-sample ranges (queued on the stream)
static int batch_join(snpm_batch *b, int algo) {
    snpm_db *db = b->db;
    cudaStream_t st = db->stream;
    const int64_t n = b->n, S = b->S;
    const int64_t n_tiles = ceil_div64(n, JOIN_TILE);
    SNPM_TRY(b->d_match_row.ensure(size_t(n) * 4));
    SNPM_TRY(b->d_tile_cnt.ensure(size_t(n_tiles) * 4));
    SNPM_TRY(b->d_tile_off.ensure(size_t(n_tiles) * 4));
    SNPM_TRY(b->d_prefix.ensure(size_t(n + 1) * 4));
    SNPM_TRY(b->d_pair_db.ensure(size_t(n) * 4));
    SNPM_TRY(b->d_pair_s.ensure(size_t(n) * 4));
    if (b->coded) { /* keys and temporaries were sized at upload */ }
    else if (b->grouped) SNPM_TRY(b->d_pair_gid.ensure(size_t(n) * 2 + 16));
    else SNPM_TRY(b->d_pair_w.ensure(size_t(n) * 32));
    SNPM_TRY(b->d_mstart.ensure(size_t(S + 1) * 4));
    SNPM_TRY(b->d_seg_off.ensure(size_t(S + 1) * 4));
    SNPM_TRY(b->d_status.ensure(8 * sizeof(int)));
    SNPM_CUDA(cudaStreamWaitEvent(st, b->ev_uploaded, 0));       // the samples are on the device
    SNPM_CUDA(cudaMemsetAsync(b->d_status.p, 0, 8 * sizeof(int), st));
    if (b->grouped && b->pending_expand && n > 0) {               // compact upload forms -> the arrays the join reads (once per upload)
        if (b->pending_expand & 1) {
            const uint32_t *d_end = b->d_runs.as<uint32_t>();
            k_expand_runs<<<int(ceil_div64(b->pending_runs * 32, 256)), 256, 0, st>>>(d_end, reinterpret_cast<const uint16_t *>(d_end + b->pending_runs),
                                                                                 int32_t(b->pending_runs), n, b->d_gid.as<uint16_t>(), b->d_runs_bad);
        }
        // packed chromosome/position words (bit 1) are unpacked by the join itself (grouped batches always take k_join_search)
        if (b->pending_expand & 4) k_expand_chrom<<<int(ceil_div64(n, 256)), 256, 0, st>>>(b->d_chrom8.as<uint8_t>(), n, b->d_chrom.as<int32_t>());
        SNPM_KERNEL_CHECK();
        b->pending_expand &= 2;                               // the packed words stay where they are
    }
    // run ends that do not ascend were counted by k_expand_runs: reported at wait / fetch (status slot 4, next to ids outside the table)
    if (b->grouped && b->d_runs_bad) SNPM_CUDA(cudaMemcpyAsync(b->d_status.as<int>() + 4, b->d_runs_bad, sizeof(int), cudaMemcpyDeviceToDevice, st));
    if (!b->peer_red.empty() && b->ipc_step > 0 && b->d_red.p == b->ipc_ptr) {      // the peers have pulled their rows of the last step
        k_wait_peers_done<<<1, 32, 0, st>>>(reinterpret_cast<const uint32_t *>(static_cast<const char *>(b->d_red.p) + b->ipc_flags_off),
                                            int32_t(b->peer_red.size()), b->ipc_step, b->d_status.as<int>());
        SNPM_KERNEL_CHECK();
    }
    // auto: per-marker binary search for low-coverage samples (n << N: a tile of markers spans a long panel slice), merge-path
    // once a sample carries more than an eighth of the panel rows (measured at m = N = 10.7 M: 0.40 ms vs 0.47 ms)
    if (algo == 0) algo = (n / S) * 8 >= db->n_rows ? 2 : 1;
    if (b->grouped) algo = 1;                                    // markers are not in position order
    const int64_t *filter = b->has_filter ? b->d_filter.as<int64_t>() : nullptr;
    // the grouping's overflow flags, read by k_combine_grouped: zero also for a batch without markers
    if (b->coded && S > 0) SNPM_CUDA(cudaMemsetAsync(b->d_group_overflow.p, 0, size_t(S) * 4, st));
    if (n_tiles > 0) {
        if (algo == 2)
            k_join_mergepath<<<int(n_tiles), 256, 0, st>>>(b->d_chrom.as<int32_t>(), b->d_pos.as<int32_t>(), n, b->d_off.as<int64_t>(), S,
                                                         db->d_pos, db->d_chr_regions, db->n_chr, filter, b->n_filter, db->row0_global,
                                                         b->d_match_row.as<int32_t>(), b->d_tile_cnt.as<int32_t>(), b->d_status.as<int>());
        else
            k_join_search<<<int(n_tiles), JOIN_TILE, 0, st>>>(b->d_chrom.as<int32_t>(), b->d_pos.as<int32_t>(), n, b->d_off.as<int64_t>(), S,
                                                            db->d_pos, db->d_chr_regions, db->n_chr, db->d_bucket, db->d_bucket_off, db->bucket_shift,
                                                            filter, b->n_filter, db->row0_global,
                                                            b->d_match_row.as<int32_t>(), b->d_tile_cnt.as<int32_t>(), b->d_status.as<int>(), (b->grouped && !b->coded) ? 0 : 1,
                                                            db->d_bitmap, db->d_bm_first_row, db->d_bm_off,
                                                            (b->grouped && (b->pending_expand & 2)) ? b->d_wei_idx.as<uint32_t>() : nullptr);
        SNPM_KERNEL_CHECK();
        if (b->has_seg) {
            static_assert(SEGP_THREADS == JOIN_TILE, "the segregation filter recounts the join's tiles");
            k_segregating_pairs<<<int(n_tiles), SEGP_THREADS, 0, st>>>(db->d_packed, db->stride, b->d_off.as<int64_t>(), S, n, b->d_segsel.as<uint2>(),
                                                                      b->d_segsel_off.as<int32_t>(), b->d_match_row.as<int32_t>(), b->d_tile_cnt.as<int32_t>());
            SNPM_KERNEL_CHECK();
            b->launches += 1;
        }
        k_scan_tiles<<<1, 1024, 0, st>>>(b->d_tile_cnt.as<int32_t>(), n_tiles, b->d_tile_off.as<int32_t>(), b->d_prefix.as<int32_t>() + n);
        SNPM_KERNEL_CHECK();
        if (b->coded) {
            unsigned long long *hash = b->d_hash.as<unsigned long long>();
            SNPM_CUDA(cudaMemsetAsync(hash, 0, size_t(S) * GH_SLOTS * 8, st));
            if (b->key_bits <= 32)
                k_scatter_pairs_coded<uint32_t><<<int(n_tiles), SC_THREADS, 0, st>>>(b->d_match_row.as<int32_t>(), n, b->d_tile_off.as<int32_t>(), b->d_codes.as<uint16_t>(),
                        b->d_wtable.as<double>(), b->n_wtable, b->code_bits, b->d_prefix.as<int32_t>(), b->d_pair_db_tmp.as<int32_t>(), b->d_pair_s_tmp.as<int32_t>(),
                        b->d_key_a.as<uint32_t>(), b->d_status.as<int>(), b->d_off.as<int64_t>(), S, hash, b->d_group_overflow.as<int>(),
                        b->codes_packed ? b->d_codes.as<uint32_t>() : nullptr);
            else
                k_scatter_pairs_coded<uint64_t><<<int(n_tiles), SC_THREADS, 0, st>>>(b->d_match_row.as<int32_t>(), n, b->d_tile_off.as<int32_t>(), b->d_codes.as<uint16_t>(),
                        b->d_wtable.as<double>(), b->n_wtable, b->code_bits, b->d_prefix.as<int32_t>(), b->d_pair_db_tmp.as<int32_t>(), b->d_pair_s_tmp.as<int32_t>(),
                        b->d_key_a.as<uint64_t>(), b->d_status.as<int>(), b->d_off.as<int64_t>(), S, hash, b->d_group_overflow.as<int>(),
                        b->codes_packed ? b->d_codes.as<uint32_t>() : nullptr);
        } else if (b->grouped)
            k_scatter_pairs_grouped<<<int(n_tiles), JOIN_TILE, 0, st>>>(b->d_match_row.as<int32_t>(), n, b->d_tile_off.as<int32_t>(),
                                                                      b->d_gid.as<uint16_t>(), b->n_gtable, b->d_prefix.as<int32_t>(), b->d_pair_db.as<int32_t>(),
                                                                      b->d_pair_s.as<int32_t>(), b->d_pair_gid.as<uint16_t>(), b->d_status.as<int>());
        else
            k_scatter_pairs<<<int(n_tiles), JOIN_TILE, 0, st>>>(b->d_match_row.as<int32_t>(), n, b->d_tile_off.as<int32_t>(), b->d_wei.as<double>(),
                                                              b->d_prefix.as<int32_t>(), b->d_pair_db.as<int32_t>(), b->d_pair_s.as<int32_t>(),
                                                              b->d_pair_w.as<double>());
        SNPM_KERNEL_CHECK();
        b->launches += 3;
    } else {
        SNPM_CUDA(cudaMemsetAsync(b->d_prefix.p, 0, 4, st));
    }
    k_sample_ranges<<<1, 1024, 0, st>>>(b->d_prefix.as<int32_t>(), b->d_off.as<int64_t>(), S, b->grouped ? b->gchunk : b->chunk_rows, b->d_mstart.as<int32_t>(),
                                        b->d_seg_off.as<int32_t>());
    SNPM_KERNEL_CHECK();
    b->launches += 1;
    return SNPM_OK;
}

}  // extern "C" (templates below)

// coded batches: dense group ids from the per-sample key tables, ONE stable partition pass that moves the panel rows into
// (group, position) order, block words (change masks + first group) from the group table
template <typename KeyT>
static int batch_group_sort_t(snpm_batch *b) {
    snpm_db *db = b->db;
    cudaStream_t st = db->stream;
    const int tiles = int(b->n_sort_tiles);
    if (tiles == 0 || b->n == 0) return SNPM_OK;
    const int32_t *mstart = b->d_mstart.as<int32_t>(), *tsample = b->d_tile_sample.as<int32_t>(), *tfirst = b->d_tile_first.as<int32_t>();
    uint32_t *hist = b->d_tile_hist.as<uint32_t>();
    int2 *range = reinterpret_cast<int2 *>(hist + (size_t(tiles) << 11));
    SNPM_CUDA(smem_attr<k_group_place>(64 * 1024));
    KeyT *gkeys = b->d_gkeys.as<KeyT>();
    k_group_rank<KeyT><<<int(b->S), 1024, 0, st>>>(b->d_hash.as<unsigned long long>(), b->d_wtable.as<double>(), b->code_bits, b->d_slot_gid.as<uint16_t>(),
                                                   b->d_ngroups.as<int32_t>(), gkeys, b->d_gw.as<double4>(), b->d_group_overflow.as<int>());
    int64_t n_max = 0, jcap1 = 1;
    for (int64_t s = 0; s < b->S; ++s) {
        n_max = std::max(n_max, b->h_off[size_t(s) + 1] - b->h_off[size_t(s)]);
        jcap1 = std::max(jcap1, ceil_div64(b->h_off[size_t(s) + 1] - b->h_off[size_t(s)], b->gchunk));
    }
    // One kernel per sample (a CTA walks its sample's pairs twice, ~2.4 us per 1000 pairs) or five kernels over tiles of 2048 pairs
    // (~0.07 ms of latency whatever the batch)?  Measured, group stage in ms, one kernel / tiles: 64 samples x 45 000 pairs 0.151 /
    // 0.112; 128 x 22 500 (a 2-GPU rank) 0.108 / 0.114; 256 x 11 250: 0.110 / 0.129; 512 x 5 600: 0.136 / 0.164; 64 x 5 600: 0.048 / 0.062.
    const char *force = getenv("SNPM_GROUP_KERNEL");                        // measurement / test switch: "tiled" or "sample"
    const bool fits = n_max <= GP_MAX_PAIRS;
    const bool want = force ? !strcmp(force, "sample") : (n_max <= 32768 || b->S >= 128);
    if (fits && want) {
        // every sample's counters fit shared memory: ids, offsets, placement, block words and segment costs in one kernel per sample
        SNPM_CUDA(smem_attr<k_group_sample<KeyT>>(int(GP_SMEM)));
        const size_t ncap = size_t(std::max<int64_t>(b->nseg_cap, 1));
        int32_t *cost = reinterpret_cast<int32_t *>(b->d_blk_chg.as<unsigned long long>() + ncap * size_t(b->gchunk / GR_BLOCK));
        int32_t *buckets = cost + ncap;
        const size_t zbytes = ncap * (size_t(b->gchunk / GR_BLOCK) * 8 + 4) + size_t(SO_BUCKETS) * 4;
        int2 *br = reinterpret_cast<int2 *>(reinterpret_cast<unsigned char *>(b->d_blk_chg.p) + ((zbytes + 7) & ~size_t(7)));
        SNPM_CUDA(cudaMemsetAsync(b->d_blk_chg.p, 0, zbytes, st));
        k_group_sample<KeyT><<<int(b->S), 32 * GP_WARPS, GP_SMEM, st>>>(
            b->d_key_a.as<KeyT>(), b->d_hash.as<unsigned long long>(), b->d_slot_gid.as<uint16_t>(), b->d_ngroups.as<int32_t>(), b->d_gid.as<uint16_t>(),
            b->d_pair_db_tmp.as<int32_t>(), b->d_pair_s_tmp.as<int32_t>(), b->d_pair_db.as<int32_t>(), b->track_pairs ? b->d_pair_s.as<int32_t>() : nullptr,
            b->d_goff.as<int32_t>(), gkeys, mstart, b->d_seg_off.as<int32_t>(), b->gchunk, b->code_bits, b->d_blk_chg.as<unsigned long long>(), cost,
            int32_t(jcap1), buckets, br, b->d_work_counter.as<unsigned int>());
        k_order_place<<<int(b->S), 256, 0, st>>>(buckets, br, b->d_seg_off.as<int32_t>(), mstart, b->gchunk, b->d_seg_order.as<int4>());
        SNPM_KERNEL_CHECK();
        b->launches += 3;
        return SNPM_OK;
    }
    k_tile_ranges<<<(tiles + 255) / 256, 256, 0, st>>>(mstart, tsample, tfirst, tiles, range);
    k_group_ids<KeyT><<<tiles, RS_THREADS, 0, st>>>(b->d_key_a.as<KeyT>(), range, tsample, b->d_hash.as<unsigned long long>(), b->d_slot_gid.as<uint16_t>(),
                                                    b->d_ngroups.as<int32_t>(), b->d_gid.as<uint16_t>(), hist);
    k_group_scan<<<int(b->S), 1024, 0, st>>>(hist, tfirst, b->d_ngroups.as<int32_t>(), b->d_goff.as<int32_t>());
    const size_t nseg_cap = size_t(std::max<int64_t>(b->nseg_cap, 1));
    int32_t *seg_cost = reinterpret_cast<int32_t *>(b->d_blk_chg.as<unsigned long long>() + nseg_cap * size_t(b->gchunk / GR_BLOCK));
    int32_t *bucket_cnt = seg_cost + nseg_cap;
    const size_t zero_bytes = nseg_cap * (size_t(b->gchunk / GR_BLOCK) * 8 + 4) + size_t(SO_BUCKETS) * 4;
    int2 *seg_br = reinterpret_cast<int2 *>(reinterpret_cast<unsigned char *>(b->d_blk_chg.p) + ((zero_bytes + 7) & ~size_t(7)));
    int64_t jcap = 1;
    for (int64_t s = 0; s < b->S; ++s) jcap = std::max(jcap, ceil_div64(b->h_off[size_t(s) + 1] - b->h_off[size_t(s)], b->gchunk));
    // The block words and the work order need the group table only, not the placed rows: they run on the batch's second stream
    // (idle between its upload and its read-back) next to the partition pass.
    cudaStream_t aux = b->copy_stream;
    if (!b->ev_fork) SNPM_CUDA(cudaEventCreateWithFlags(&b->ev_fork, cudaEventDisableTiming));
    if (!b->ev_join) SNPM_CUDA(cudaEventCreateWithFlags(&b->ev_join, cudaEventDisableTiming));
    SNPM_CUDA(cudaEventRecord(b->ev_fork, st));
    SNPM_CUDA(cudaStreamWaitEvent(aux, b->ev_fork, 0));
    SNPM_CUDA(cudaMemsetAsync(b->d_blk_chg.p, 0, zero_bytes, aux));
    k_group_marks<KeyT><<<int(b->S), 1024, 0, aux>>>(b->d_goff.as<int32_t>(), gkeys, b->d_ngroups.as<int32_t>(), mstart, b->d_seg_off.as<int32_t>(), b->gchunk,
                                                     b->code_bits, b->d_blk_chg.as<unsigned long long>(), seg_cost, int32_t(jcap), bucket_cnt, seg_br);
    k_order_place<<<int(b->S), 256, 0, aux>>>(bucket_cnt, seg_br, b->d_seg_off.as<int32_t>(), mstart, b->gchunk, b->d_seg_order.as<int4>());
    SNPM_CUDA(cudaEventRecord(b->ev_join, aux));
    k_group_place<<<tiles, RS_THREADS, size_t(GH_MAX_GROUPS) * 20, st>>>(b->d_gid.as<uint16_t>(), b->d_pair_db_tmp.as<int32_t>(), b->d_pair_s_tmp.as<int32_t>(),
                                                                        b->d_pair_db.as<int32_t>(), b->track_pairs ? b->d_pair_s.as<int32_t>() : nullptr, mstart, tsample,
                                                                        tfirst, range, hist, b->d_ngroups.as<int32_t>(), b->d_goff.as<int32_t>(), b->d_work_counter.as<unsigned int>());
    SNPM_CUDA(cudaStreamWaitEvent(st, b->ev_join, 0));
    SNPM_KERNEL_CHECK();
    b->launches += 7;
    return SNPM_OK;
}

static int launch_grouped2(snpm_batch *b, bool skip_db_hets) {
    snpm_db *db = b->db;
    cudaStream_t st = db->stream;
    Group2Args g = {};
    g.packed = db->d_packed; g.stride = db->stride; g.pair_db = b->d_pair_db.as<int32_t>();
    g.blk_chg = b->d_blk_chg.as<unsigned long long>(); g.gw = b->d_gw.as<double>();
    g.seg_off = b->d_seg_off.as<int32_t>(); g.mstart = b->d_mstart.as<int32_t>(); g.S = int32_t(b->S); g.chunk = b->gchunk;
    g.part_score = b->d_part_score.as<double>(); g.part_int = b->d_part_int.as<int32_t>(); g.a_pad = db->stride * 32;
    // a row of up to 36 words (1135 accessions) is one slice; wider rows are cut into warp-aligned slices of 32 words
    if (db->stride <= G2_WX) { g.n_slices = 1; g.wx = (db->stride + 1) & ~1; }
    else { g.wx = 32; g.n_slices = (db->stride + 31) / 32; }
    g.teams = std::min(G2_THREADS / g.wx, G2_MAX_TEAMS);
    g.order = b->d_seg_order.as<int4>();
    g.work_counter = b->d_work_counter.as<unsigned int>();
    const int64_t n_items = std::max<int64_t>(b->nseg_cap, 1) * g.n_slices;      // upper bound (segments by markers; the kernel counts matched ones)
    if (n_items >= (int64_t(1) << 31) - (int64_t(1) << 20)) return fail(SNPM_E_ARG, "snpm_batch_run: %lld work items exceed the 2^31 limit", (long long)n_items);
    constexpr int ring = 64;                 // rows of a team's gather ring: 3 blocks in flight while one is scored
    const size_t smem = size_t(g.teams) * g2_team_smem(g.wx, g.chunk, ring);
    if (smem > 226 * 1024) return fail(SNPM_E_ARG, "snpm_batch_run: group chunk %d needs %zu bytes of shared memory", g.chunk, smem);
    const int grid = int(std::min<int64_t>(db->n_sm, ceil_div64(n_items, g.teams)));
#define G2_LAUNCH(SK, WXV)                                                                                                        \
    do {                                                                                                                          \
        SNPM_CUDA((smem_attr<k_score_grouped2<SK, WXV, ring>>(226 * 1024)));                                                    \
        k_score_grouped2<SK, WXV, ring><<<grid, G2_THREADS, smem, st>>>(g);                                                       \
    } while (0)
    if (g.wx == G2_WX) {
        if (skip_db_hets) G2_LAUNCH(true, G2_WX); else G2_LAUNCH(false, G2_WX);
    } else if (g.wx == 32) {
        if (skip_db_hets) G2_LAUNCH(true, 32); else G2_LAUNCH(false, 32);
    } else {
        if (skip_db_hets) G2_LAUNCH(true, 0); else G2_LAUNCH(false, 0);
    }
#undef G2_LAUNCH
    SNPM_KERNEL_CHECK();
    b->launches += 1;
    return SNPM_OK;
}

extern "C" {

static int batch_alloc_outputs(snpm_batch *b, int64_t nseg) {
    snpm_db *db = b->db;
    const int64_t a_pad = int64_t(db->stride) * 32;
    const int64_t SA = b->S * int64_t(db->n_acc);
    SNPM_TRY(b->d_part_score.ensure(size_t(std::max<int64_t>(nseg, 1)) * a_pad * 8));
    SNPM_TRY(b->d_part_ninfo.ensure(size_t(std::max<int64_t>(nseg, 1)) * a_pad * 4));
    SNPM_TRY(b->d_red.ensure(size_t(b->S) * size_t(b->red_pitch()) * 8));
    if (b->grouped) SNPM_TRY(b->d_part_int.ensure(size_t(std::max<int64_t>(nseg, 1)) * a_pad * 4));
    SNPM_TRY(b->d_matches.ensure(size_t(SA) * 8));
    SNPM_TRY(b->d_ninfo64.ensure(size_t(SA) * 8));
    SNPM_TRY(b->d_prob.ensure(size_t(SA) * 8));
    SNPM_TRY(b->d_L.ensure(size_t(SA) * 8));
    SNPM_TRY(b->d_LR.ensure(size_t(SA) * 8));
    return SNPM_OK;
}

static void rec(snpm_batch *b, int which) {
    cudaEventRecord(b->ev[which], b->db->stream);
    b->ev_rec[which] = true;
}

// the end of every run: the next upload may overwrite the inputs behind its kernels, and the epilogue is still to come
static int run_done(snpm_batch *b) {
    rec(b, SNPM_EV_COMBINE);
    SNPM_CUDA(cudaEventRecord(b->ev_inputs_free, b->db->stream));
    b->ran = true;
    b->ran_windows = false;
    b->epilogue_done = false;
    return SNPM_OK;
}

int snpm_batch_run(snpm_batch *b, int skip_db_hets, int mode) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_run: NULL batch");
    snpm_db *db = b->db;
    SNPM_CUDA(cudaSetDevice(db->device));
    cudaStream_t st = db->stream;
    const int kernel_mode = mode & 0xff, algo = (mode >> 8) & 0xff;
    if (kernel_mode < 0 || kernel_mode > 2) return fail(SNPM_E_ARG, "snpm_batch_run: unknown kernel mode %d", kernel_mode);
    if ((kernel_mode == 2) != b->grouped)
        return fail(SNPM_E_STATE, "snpm_batch_run: kernel mode 2 scores batches uploaded with snpm_batch_upload_grouped, and only those");
    if (algo > 2) return fail(SNPM_E_ARG, "snpm_batch_run: unknown join algorithm %d", algo);
    if (b->has_seg && kernel_mode == 2)
        return fail(SNPM_E_STATE, "snpm_batch_run: the segregation filter is honoured by kernel modes 0 and 1 only; clear it first");
    if (b->has_seg && b->seg_S != b->S)
        return fail(SNPM_E_ARG, "snpm_batch_run: the segregation filter holds %lld selections for %lld samples", (long long)b->seg_S, (long long)b->S);
    b->launches = 0;
    for (int i = 0; i < SNPM_N_EVENTS; ++i) b->ev_rec[i] = false;
    SNPM_TRY(batch_alloc_outputs(b, b->nseg_cap));
    rec(b, SNPM_EV_START);
    SNPM_TRY(batch_join(b, algo));
    rec(b, SNPM_EV_JOIN);
    ScoreArgs a = {};
    a.packed = db->d_packed;
    a.stride = db->stride;
    a.pair_db = b->d_pair_db.as<int32_t>();
    a.pair_w = b->d_pair_w.as<double>();
    a.seg_off = b->d_seg_off.as<int32_t>();
    a.mstart = b->d_mstart.as<int32_t>();
    a.S = int32_t(b->S);
    a.chunk = b->chunk_rows;
    a.table = 0;
    a.part_score = b->d_part_score.as<double>();
    a.part_ninfo = b->d_part_ninfo.as<int32_t>();
    a.a_pad = db->stride * 32;
    if (kernel_mode == 2 && b->coded) {
        cudaEventRecord(b->ev_joined, st);
        if (b->key_bits <= 32) SNPM_TRY(batch_group_sort_t<uint32_t>(b)); else SNPM_TRY(batch_group_sort_t<uint64_t>(b));
        rec(b, SNPM_EV_JOIN);                      // for coded batches "join" ends after the grouping: score_ms is the scoring kernel alone
        if (b->nseg_cap > 0 && b->n > 0) {
            SNPM_TRY(launch_grouped2(b, skip_db_hets != 0));
        }
        rec(b, SNPM_EV_SCORE);
        dim3 cgrid((a.a_pad + 31) / 32, unsigned(b->S));
        k_combine_grouped<<<cgrid, 32 * CG_PARTS, 0, st>>>(a.part_score, b->d_part_int.as<int32_t>(), a.a_pad, db->stride, db->n_acc, a.seg_off, a.mstart,
                                                 b->d_group_overflow.as<int>(), b->d_red.as<double>());
        SNPM_KERNEL_CHECK();
        b->launches += 1;
        return run_done(b);
    }
    if (kernel_mode == 2) {
        if (b->nseg_cap > 0) {
            GroupArgs g = {};
            g.packed = db->d_packed; g.stride = db->stride; g.pair_db = a.pair_db; g.pair_gid = b->d_pair_gid.as<uint16_t>();
            g.table = b->d_gtable.as<double>(); g.seg_off = a.seg_off; g.mstart = a.mstart; g.S = a.S; g.chunk = b->gchunk;
            g.part_score = a.part_score; g.part_int = b->d_part_int.as<int32_t>(); g.a_pad = a.a_pad;
            const int nsl = (db->stride + GR_MAX_WX - 1) / GR_MAX_WX;
            g.wx = ((db->stride + nsl - 1) / nsl + 1) & ~1;          // even: neighbouring threads copy 16-byte pairs of columns
            g.spc = std::min(GR_THREADS / g.wx, GR_MAX_TEAMS);
            const size_t gsmem = size_t(g.spc) * grouped_team_smem(g.wx, g.chunk);
            int64_t jmax = 0;
            for (int64_t smp = 0; smp < b->S; ++smp)
                jmax = std::max(jmax, ceil_div64(b->h_off[size_t(smp) + 1] - b->h_off[size_t(smp)], b->gchunk));
            g.jmax = int32_t(jmax);
            dim3 ggrid(unsigned(ceil_div64(b->S * jmax, g.spc)), unsigned((db->stride + g.wx - 1) / g.wx));
#define GR_LAUNCH(SK, WXV)                                                     \
    do {                                                                       \
        SNPM_CUDA((smem_attr<k_score_grouped<SK, WXV>>(220 * 1024)));          \
        k_score_grouped<SK, WXV><<<ggrid, GR_THREADS, gsmem, st>>>(g);         \
    } while (0)
            if (g.wx == GR_MAX_WX) {       // the 1135-accession row: addresses known at compile time
                if (skip_db_hets) GR_LAUNCH(true, GR_MAX_WX); else GR_LAUNCH(false, GR_MAX_WX);
            } else {
                if (skip_db_hets) GR_LAUNCH(true, 0); else GR_LAUNCH(false, 0);
            }
#undef GR_LAUNCH
            SNPM_KERNEL_CHECK();
            b->launches += 1;
        }
        rec(b, SNPM_EV_SCORE);
        dim3 cgrid((a.a_pad + 31) / 32, unsigned(b->S));
        k_combine_grouped<<<cgrid, 32 * CG_PARTS, 0, st>>>(a.part_score, b->d_part_int.as<int32_t>(), a.a_pad, db->stride, db->n_acc, a.seg_off, a.mstart,
                                                 nullptr, b->d_red.as<double>());
        SNPM_KERNEL_CHECK();
        b->launches += 1;
        return run_done(b);
    }
    if (kernel_mode == 1 && b->chunk_rows != SNPM_CHUNK_ROWS)
        return fail(SNPM_E_STATE, "snpm_batch_run: the popcount kernel works in %d-row chunks (its sums are exact in any chunking); set the chunk back", SNPM_CHUNK_ROWS);
    if (kernel_mode == 1 && b->nseg_cap > 0) {
        // called genotypes (one-hot weights): popcount kernel, exact in every summation order
        SNPM_TRY(b->d_pair_code.ensure(size_t(std::max<int64_t>(b->n, 1))));
        k_pair_codes<<<int(ceil_div64(b->n, 256)), 256, 0, st>>>(a.pair_w, b->d_prefix.as<int32_t>() + b->n, b->d_pair_code.as<uint8_t>());
        SNPM_KERNEL_CHECK();
        HardArgs h = {};
        h.packed = a.packed; h.stride = a.stride; h.pair_db = a.pair_db; h.pair_code = b->d_pair_code.as<uint8_t>();
        h.seg_off = a.seg_off; h.mstart = a.mstart; h.S = a.S; h.chunk = a.chunk;
        h.part_score = a.part_score; h.part_ninfo = a.part_ninfo; h.a_pad = a.a_pad; h.status = b->d_status.as<int>();
        const int wx = std::min<int>(db->stride, HC_THREADS), spc = std::min(HC_THREADS / wx, HC_MAX_SEGS);
        h.wx = wx;
        h.spc = spc;
        dim3 hgrid(unsigned(ceil_div64(b->nseg_cap, spc)), unsigned((db->stride + wx - 1) / wx));
        const size_t hsmem = size_t(spc) * SNPM_CHUNK_ROWS * 5;
        if (skip_db_hets) {
            SNPM_CUDA(smem_attr<k_score_hard<true>>(64 * 1024));
            k_score_hard<true><<<hgrid, HC_THREADS, hsmem, st>>>(h);
        } else {
            SNPM_CUDA(smem_attr<k_score_hard<false>>(64 * 1024));
            k_score_hard<false><<<hgrid, HC_THREADS, hsmem, st>>>(h);
        }
        SNPM_KERNEL_CHECK();
        b->launches += 2;
    } else {
        SNPM_TRY(launch_score(st, a, int(b->nseg_cap), skip_db_hets != 0));
        if (b->nseg_cap > 0) b->launches += 1;
    }
    rec(b, SNPM_EV_SCORE);
    // one warp per CTA: the per-accession chain is sequential, so spread the accessions over as many SMs as possible
    dim3 cgrid((db->n_acc + 31) / 32, unsigned(b->S));
    k_combine<<<cgrid, 32, 0, st>>>(a.part_score, a.part_ninfo, a.a_pad, db->n_acc, a.seg_off, a.mstart, 0, nullptr, nullptr, b->d_red.as<double>());
    SNPM_KERNEL_CHECK();
    b->launches += 1;
    return run_done(b);
}

int snpm_batch_epilogue(snpm_batch *b) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_epilogue: NULL batch");
    if (!b->ran) return fail(SNPM_E_STATE, "snpm_batch_epilogue: run the batch first");
    // k_grouped_finalize turns F into I + F in place: a second pass over the same totals would add I again
    if (b->grouped && b->epilogue_done) return fail(SNPM_E_STATE, "snpm_batch_epilogue: the epilogue of a grouped batch runs once per run");
    snpm_db *db = b->db;
    SNPM_CUDA(cudaSetDevice(db->device));
    const int64_t r0 = b->range0(), rn = b->rangen();
    if (r0 < 0 || rn < 0 || r0 + rn > b->S) return fail(SNPM_E_ARG, "snpm_batch_epilogue: result range [%lld, %lld) outside the %lld samples", (long long)r0, (long long)(r0 + rn), (long long)b->S);
    rec(b, SNPM_EV_EPI_START);
    const int64_t pitch = b->red_pitch(), A = db->n_acc;
    if (rn > 0) {
        if (b->grouped) {
            // totals (after any cross-GPU reduce) -> score with the reference's truncation, guard counts per sample
            SNPM_TRY(b->d_guard.ensure(size_t(b->S) * 4));
            SNPM_CUDA(cudaMemsetAsync(b->d_guard.as<int32_t>() + r0, 0, size_t(rn) * 4, db->stream));
            dim3 fgrid((db->n_acc + 255) / 256, unsigned(rn));
            k_grouped_finalize<<<fgrid, 256, 0, db->stream>>>(b->d_red.as<double>() + r0 * pitch, db->n_acc, b->d_guard.as<int32_t>() + r0);
            SNPM_KERNEL_CHECK();
            b->launches += 1;
        }
        SNPM_CUDA(launch_epilogue(db->stream, rn, b->d_red.as<double>() + r0 * pitch, pitch, db->n_acc, 1, 0, 0.0,
                                  b->d_matches.as<int64_t>() + r0 * A, b->d_ninfo64.as<int64_t>() + r0 * A,
                                  b->d_prob.as<double>() + r0 * A, b->d_L.as<double>() + r0 * A, b->d_LR.as<double>() + r0 * A));
    }
    SNPM_KERNEL_CHECK();
    b->launches += 1;
    rec(b, SNPM_EV_EPI_END);
    b->epilogue_done = true;
    return SNPM_OK;
}

// the argument and state errors the kernels count in the status slots (read back into h_status), in their order of precedence
static int status_error(const int *h_status) {
    if (h_status[0] > 0)
        return fail(SNPM_E_ARG, "sample markers are not sorted by (database chromosome order, position) or repeat a position (%d places)", h_status[0]);
    if (h_status[1] > 0)
        return fail(SNPM_E_ASSERT, "provided y is greater than n (%d window cells; likeliTest, snpmatch.py:43)", h_status[1]);
    if (h_status[2] > 0)
        return fail(SNPM_E_ARG, "identity table too short for %d window cells", h_status[2]);
    if (h_status[3] > 0)
        return fail(SNPM_E_ARG, "kernel mode 1 needs one-hot weights (called genotypes); %d matched markers are not", h_status[3]);
    if (h_status[4] > 0)
        return fail(SNPM_E_ARG, "%d matched markers carry a weight-triple id outside the table (or run-length coded ids do not ascend)", h_status[4]);
    if (h_status[5] > 0)
        return fail(SNPM_E_STATE, "peer reduce: a rank did not arrive within thirty seconds (every rank must run and reduce the same batches in the same order)");
    return SNPM_OK;
}

int snpm_batch_wait(snpm_batch *b, float *ms_device) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_wait: NULL batch");
    snpm_db *db = b->db;
    SNPM_CUDA(cudaSetDevice(db->device));
    if (b->d_status.p) SNPM_CUDA(cudaMemcpyAsync(b->h_status, b->d_status.p, 8 * sizeof(int), cudaMemcpyDeviceToHost, db->stream));
    else memset(b->h_status, 0, 8 * sizeof(int));
    SNPM_CUDA(cudaStreamSynchronize(db->stream));
    if (ms_device) {
        *ms_device = 0.f;
        if (b->ev_rec[SNPM_EV_START] && b->ev_rec[SNPM_EV_COMBINE]) {
            float t = 0.f;
            cudaEventElapsedTime(&t, b->ev[SNPM_EV_START], b->ev[SNPM_EV_COMBINE]);
            *ms_device += t;
        }
        if (b->ev_rec[SNPM_EV_EPI_START] && b->ev_rec[SNPM_EV_EPI_END]) {
            float t = 0.f;
            cudaEventElapsedTime(&t, b->ev[SNPM_EV_EPI_START], b->ev[SNPM_EV_EPI_END]);
            *ms_device += t;
        }
    }
    return status_error(b->h_status);
}

int snpm_batch_timings(snpm_batch *b, float *ms, int n) {
    if (!b || !ms || n < 6) return fail(SNPM_E_ARG, "snpm_batch_timings: need room for 6 floats");
    SNPM_CUDA(cudaSetDevice(b->db->device));
    SNPM_CUDA(cudaStreamSynchronize(b->db->stream));
    for (int i = 0; i < n; ++i) ms[i] = 0.f;
    auto el = [&](int a, int c) {
        float t = 0.f;
        if (b->ev_rec[a] && b->ev_rec[c]) cudaEventElapsedTime(&t, b->ev[a], b->ev[c]);
        return t;
    };
    ms[0] = el(SNPM_EV_START, SNPM_EV_JOIN);
    ms[1] = el(SNPM_EV_JOIN, SNPM_EV_SCORE);
    ms[2] = el(SNPM_EV_SCORE, SNPM_EV_COMBINE);
    ms[3] = el(SNPM_EV_EPI_START, SNPM_EV_EPI_END);
    ms[4] = el(SNPM_EV_START, SNPM_EV_COMBINE) + ms[3];
    ms[5] = float(b->launches);
    if (n >= 8) {                                  // one-shot peer reduce of the last step: the whole kernel, and its wait for the slowest rank
        ms[6] = el(SNPM_EV_RED_START, SNPM_EV_RED_END);
        int wait_ns = 0;
        if (b->ev_rec[SNPM_EV_RED_END] && b->d_status.p) cudaMemcpy(&wait_ns, b->d_status.as<int>() + 7, sizeof(int), cudaMemcpyDeviceToHost);
        ms[7] = float(wait_ns) * 1e-6f;
    }
    return SNPM_OK;
}

int snpm_batch_reduce_buffer(snpm_batch *b, void **dev_ptr, int64_t *n_doubles) {
    if (!b || !dev_ptr) return fail(SNPM_E_ARG, "snpm_batch_reduce_buffer: NULL argument");
    SNPM_CUDA(cudaSetDevice(b->db->device));
    SNPM_TRY(b->d_red.ensure(size_t(b->S) * size_t(b->red_pitch()) * 8));
    *dev_ptr = b->d_red.p;
    if (n_doubles) *n_doubles = b->S * b->red_pitch();
    return SNPM_OK;
}

// ---- one-shot reduce over peer memory ----------------------------------------------------------------------
static void ipc_close_peers(snpm_batch *b) {
    for (size_t r = 0; r < b->peer_red.size(); ++r)
        if (int32_t(r) != b->ipc_rank && b->peer_red[r]) cudaIpcCloseMemHandle(b->peer_red[r]);
    b->peer_red.clear();
    b->ipc_rank = -1;
}

int snpm_batch_ipc_export(snpm_batch *b, void *handle64, int64_t *n_doubles) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
    if (!b || !handle64) return fail(SNPM_E_ARG, "snpm_batch_ipc_export: NULL argument");
    SNPM_CUDA(cudaSetDevice(b->db->device));
    // at least 4 MB: large allocations are their own mapping, so the peers' pointer is the buffer itself (small cudaMalloc
    // blocks may be carved out of a shared 2 MB page, whose IPC handle maps the page).  The last 4 KB hold the flags.
    const size_t bytes = size_t(b->S) * size_t(b->red_pitch()) * 8;
    const size_t cap = std::max<size_t>(((bytes + 255) & ~size_t(255)) + PR_FLAG_BYTES, size_t(4) << 20);
    SNPM_CUDA(cudaStreamSynchronize(b->db->stream));
    if (b->d_red.cap != cap) {
        b->d_red.release();
        SNPM_TRY(b->d_red.ensure(cap));
    }
    b->ipc_flags_off = cap - PR_FLAG_BYTES;
    b->ipc_step = 0;
    SNPM_CUDA(cudaMemset(static_cast<char *>(b->d_red.p) + b->ipc_flags_off, 0, PR_FLAG_BYTES));
    SNPM_CUDA(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t *>(handle64), b->d_red.p));
    b->ipc_ptr = b->d_red.p;
    if (n_doubles) *n_doubles = b->S * b->red_pitch();
    return SNPM_OK;
}

int snpm_batch_ipc_open(snpm_batch *b, const void *handles, int32_t world, int32_t rank) {
    if (!b || !handles || world < 1 || world > PR_MAX_WORLD || rank < 0 || rank >= world) return fail(SNPM_E_ARG, "snpm_batch_ipc_open: bad arguments (at most %d ranks)", PR_MAX_WORLD);
    if (!b->ipc_ptr || b->ipc_ptr != b->d_red.p) return fail(SNPM_E_STATE, "snpm_batch_ipc_open: export this batch's buffer first (snpm_batch_ipc_export)");
    SNPM_CUDA(cudaSetDevice(b->db->device));
    ipc_close_peers(b);
    b->peer_red.assign(size_t(world), nullptr);
    b->ipc_rank = rank;
    const cudaIpcMemHandle_t *h = reinterpret_cast<const cudaIpcMemHandle_t *>(handles);
    for (int32_t r = 0; r < world; ++r) {
        if (r == rank) { b->peer_red[size_t(r)] = b->d_red.p; continue; }
        cudaError_t e = cudaIpcOpenMemHandle(&b->peer_red[size_t(r)], h[r], cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            b->peer_red[size_t(r)] = nullptr;
            ipc_close_peers(b);
            return fail(SNPM_E_CUDA, "snpm_batch_ipc_open: rank %d's buffer: %s", r, cudaGetErrorString(e));
        }
    }
    return SNPM_OK;
}

int snpm_batch_ipc_close(snpm_batch *b) {
    if (!b) return SNPM_OK;
    cudaSetDevice(b->db->device);
    cudaStreamSynchronize(b->db->stream);
    ipc_close_peers(b);
    b->ipc_ptr = nullptr;
    return SNPM_OK;
}

int snpm_batch_reduce_peers(snpm_batch *b) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_reduce_peers: NULL batch");
    if (!b->ran) return fail(SNPM_E_STATE, "snpm_batch_reduce_peers: run the batch first");
    const int32_t world = int32_t(b->peer_red.size());
    if (world < 1 || b->ipc_rank < 0) return fail(SNPM_E_STATE, "snpm_batch_reduce_peers: open the peers' buffers first (snpm_batch_ipc_open)");
    if (b->d_red.p != b->ipc_ptr) return fail(SNPM_E_STATE, "snpm_batch_reduce_peers: the reduce buffer moved since it was exported (batch grew): export and open again");
    const int64_t r0 = b->res0, rn = b->resn < 0 ? b->S - b->res0 : b->resn;
    if (r0 + rn > b->S) return fail(SNPM_E_ARG, "snpm_batch_reduce_peers: result range outside the batch");
    const int64_t pitch = b->red_pitch();
    int64_t first = r0 * pitch, count = rn * pitch;          // an empty share still takes part in the barrier
    SNPM_CUDA(cudaSetDevice(b->db->device));
    PeerPtrs pp;
    for (int32_t r = 0; r < PR_MAX_WORLD; ++r) {
        pp.p[r] = r < world ? static_cast<const double *>(b->peer_red[size_t(r)]) : nullptr;
        pp.flags[r] = r < world ? reinterpret_cast<uint32_t *>(static_cast<char *>(b->peer_red[size_t(r)]) + b->ipc_flags_off) : nullptr;
    }
    b->ipc_step += 1;
    rec(b, SNPM_EV_RED_START);
    const bool vec = ((first | count) & 1) == 0;
    const int grid = int(std::max<int64_t>(1, std::min<int64_t>(ceil_div64(vec ? count / 2 : count, 256), int64_t(b->db->n_sm) * 4)));
    if (vec) k_reduce_peers<double2><<<grid, 256, 0, b->db->stream>>>(pp, world, b->ipc_rank, b->ipc_step, first, count, b->d_red.as<double>(), b->d_status.as<int>());
    else k_reduce_peers<double><<<grid, 256, 0, b->db->stream>>>(pp, world, b->ipc_rank, b->ipc_step, first, count, b->d_red.as<double>(), b->d_status.as<int>());
    rec(b, SNPM_EV_RED_END);
    SNPM_KERNEL_CHECK();
    b->launches += 1;
    return SNPM_OK;
}

// queues on `st` the read-back of the result range: the (m, y > n count) pair of every sample into `tail` (2 doubles a sample),
// and whichever of the scores and the epilogue's outputs the caller asks for
static int queue_result_copies(snpm_batch *b, cudaStream_t st, double *tail, double *score, int64_t *matches, int64_t *ninfo, double *prob,
                               double *L, double *LR) {
    const size_t A = size_t(b->db->n_acc), S = size_t(b->rangen()), R0 = size_t(b->range0()), pitch = size_t(b->red_pitch()) * 8;
    const double *red = b->d_red.as<double>() + R0 * size_t(b->red_pitch());
    if (score) SNPM_CUDA(cudaMemcpy2DAsync(score, A * 8, red, pitch, A * 8, S, cudaMemcpyDeviceToHost, st));
    SNPM_CUDA(cudaMemcpy2DAsync(tail, 16, red + 2 * A, pitch, 16, S, cudaMemcpyDeviceToHost, st));
    if (matches) SNPM_CUDA(cudaMemcpyAsync(matches, b->d_matches.as<int64_t>() + R0 * A, S * A * 8, cudaMemcpyDeviceToHost, st));
    if (ninfo) SNPM_CUDA(cudaMemcpyAsync(ninfo, b->d_ninfo64.as<int64_t>() + R0 * A, S * A * 8, cudaMemcpyDeviceToHost, st));
    if (prob) SNPM_CUDA(cudaMemcpyAsync(prob, b->d_prob.as<double>() + R0 * A, S * A * 8, cudaMemcpyDeviceToHost, st));
    if (L) SNPM_CUDA(cudaMemcpyAsync(L, b->d_L.as<double>() + R0 * A, S * A * 8, cudaMemcpyDeviceToHost, st));
    if (LR) SNPM_CUDA(cudaMemcpyAsync(LR, b->d_LR.as<double>() + R0 * A, S * A * 8, cudaMemcpyDeviceToHost, st));
    return SNPM_OK;
}

// m of each of the S samples from the read-back tail; with `check` (after the epilogue) an accession with y > n fails the fetch
static int decode_tail(const double *tail, int64_t S, int64_t *m, bool check) {
    long long viol = 0;
    for (int64_t s = 0; s < S; ++s) {
        if (m) m[s] = int64_t(tail[2 * s]);
        viol += (long long)tail[2 * s + 1];
    }
    if (viol > 0 && check) return fail(SNPM_E_ASSERT, "provided y is greater than n (%lld accessions; likeliTest, snpmatch.py:43)", viol);
    return SNPM_OK;
}

int snpm_batch_fetch(snpm_batch *b, double *score, int64_t *matches, int64_t *ninfo, int64_t *m, double *prob, double *L, double *LR) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_fetch: NULL batch");
    if (!b->ran) return fail(SNPM_E_STATE, "snpm_batch_fetch: run the batch first");
    if ((matches || ninfo || prob || L || LR) && !b->epilogue_done) return fail(SNPM_E_STATE, "snpm_batch_fetch: run the epilogue first");
    SNPM_CUDA(cudaSetDevice(b->db->device));
    const size_t S = size_t(b->rangen()), R0 = size_t(b->range0());
    if (R0 + S > size_t(b->S)) return fail(SNPM_E_ARG, "snpm_batch_fetch: result range outside the batch");
    if (b->grouped && score && !b->epilogue_done) return fail(SNPM_E_STATE, "snpm_batch_fetch: grouped batches finalise their scores in the epilogue; run it first");
    std::vector<double> tail(2 * S + 2);
    if (S > 0) SNPM_TRY(queue_result_copies(b, b->db->stream, tail.data(), score, matches, ninfo, prob, L, LR));
    SNPM_TRY(snpm_batch_wait(b, nullptr));
    return decode_tail(tail.data(), int64_t(S), m, b->epilogue_done);
}


// Asynchronous variant of snpm_batch_fetch: queues the device-to-host copies behind the batch's kernels and returns; the
// host buffers (pinned, for the copies to be truly asynchronous) are valid after snpm_batch_fetch_wait.  Lets a caller queue
// the next batch's kernels before it waits for this one's results.
int snpm_batch_fetch_async(snpm_batch *b, double *score, int64_t *matches, int64_t *ninfo, int64_t *m, double *prob, double *L, double *LR,
                           int32_t *guard) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_fetch_async: NULL batch");
    if (!b->ran) return fail(SNPM_E_STATE, "snpm_batch_fetch_async: run the batch first");
    if (!b->epilogue_done) return fail(SNPM_E_STATE, "snpm_batch_fetch_async: run the epilogue first");
    snpm_db *db = b->db;
    SNPM_CUDA(cudaSetDevice(db->device));
    // the copies run on the batch's copy stream, behind an event that marks the end of its kernels: the read-back does not
    // hold up whatever is queued next on the compute stream
    cudaStream_t st = b->copy_stream;
    const size_t S = size_t(b->rangen()), R0 = size_t(b->range0());
    if (R0 + S > size_t(b->S) || S == 0) return fail(SNPM_E_ARG, "snpm_batch_fetch_async: empty result range or outside the batch");
    if (!b->ev_fetched) SNPM_CUDA(cudaEventCreateWithFlags(&b->ev_fetched, cudaEventDisableTiming));
    if (!b->ev_results) SNPM_CUDA(cudaEventCreateWithFlags(&b->ev_results, cudaEventDisableTiming));
    SNPM_CUDA(cudaEventRecord(b->ev_results, db->stream));
    SNPM_CUDA(cudaStreamWaitEvent(st, b->ev_results, 0));
    if (b->h_tail_cap < int64_t(S)) {
        if (b->h_tail) cudaFreeHost(b->h_tail);
        b->h_tail = nullptr;
        SNPM_CUDA(cudaMallocHost(reinterpret_cast<void **>(&b->h_tail), S * 16));
        b->h_tail_cap = int64_t(S);
    }
    SNPM_TRY(queue_result_copies(b, st, b->h_tail, score, matches, ninfo, prob, L, LR));
    if (guard) {
        if (b->grouped) SNPM_CUDA(cudaMemcpyAsync(guard, b->d_guard.as<int32_t>() + R0, S * 4, cudaMemcpyDeviceToHost, st));
        else memset(guard, 0, S * 4);
    }
    if (b->d_status.p) SNPM_CUDA(cudaMemcpyAsync(b->h_status, b->d_status.p, 8 * sizeof(int), cudaMemcpyDeviceToHost, st));
    else memset(b->h_status, 0, 8 * sizeof(int));
    SNPM_CUDA(cudaEventRecord(b->ev_fetched, st));
    b->pend_m = m;
    b->fetch_pending = true;
    return SNPM_OK;
}

int snpm_batch_fetch_wait(snpm_batch *b) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_fetch_wait: NULL batch");
    if (!b->fetch_pending) return fail(SNPM_E_STATE, "snpm_batch_fetch_wait: no fetch is pending");
    SNPM_CUDA(cudaSetDevice(b->db->device));
    SNPM_CUDA(cudaEventSynchronize(b->ev_fetched));
    b->fetch_pending = false;
    SNPM_TRY(status_error(b->h_status));
    return decode_tail(b->h_tail, b->rangen(), b->pend_m, true);
}

int snpm_batch_fetch_pairs(snpm_batch *b, int64_t s, int64_t *db_idx, int64_t *s_idx, int64_t capacity, int64_t *m) {
    if (!b || s < 0 || s >= b->S || !m) return fail(SNPM_E_ARG, "snpm_batch_fetch_pairs: bad arguments");
    if (!b->ran) return fail(SNPM_E_STATE, "snpm_batch_fetch_pairs: run the batch first");
    if (b->coded && !b->track_pairs) return fail(SNPM_E_STATE, "snpm_batch_fetch_pairs: the pairs of this coded batch are not tracked (snpm_batch_set_track_pairs)");
    snpm_db *db = b->db;
    SNPM_CUDA(cudaSetDevice(db->device));
    int32_t range[2];
    SNPM_CUDA(cudaMemcpyAsync(range, b->d_mstart.as<int32_t>() + s, 8, cudaMemcpyDeviceToHost, db->stream));
    SNPM_CUDA(cudaStreamSynchronize(db->stream));
    const int64_t cnt = range[1] - range[0];
    *m = cnt;
    if (cnt == 0 || (!db_idx && !s_idx)) return SNPM_OK;
    if (cnt > capacity) return fail(SNPM_E_ARG, "snpm_batch_fetch_pairs: capacity %lld < %lld pairs", (long long)capacity, (long long)cnt);
    std::vector<int32_t> tmp(size_t(cnt) * 2);
    SNPM_CUDA(cudaMemcpyAsync(tmp.data(), b->d_pair_db.as<int32_t>() + range[0], size_t(cnt) * 4, cudaMemcpyDeviceToHost, db->stream));
    SNPM_CUDA(cudaMemcpyAsync(tmp.data() + cnt, b->d_pair_s.as<int32_t>() + range[0], size_t(cnt) * 4, cudaMemcpyDeviceToHost, db->stream));
    SNPM_CUDA(cudaStreamSynchronize(db->stream));
    const int64_t base = b->h_off[size_t(s)];
    for (int64_t i = 0; i < cnt; ++i) {
        if (db_idx) db_idx[i] = int64_t(tmp[size_t(i)]) + db->row0_global;
        if (s_idx) s_idx[i] = int64_t(tmp[size_t(cnt + i)]) - base;
    }
    return SNPM_OK;
}

int snpm_score(snpm_db *db, const int32_t *s_chrom_id, const int32_t *s_pos, const double *wei, int64_t n, int skip_db_hets,
               const int64_t *filter_rows, int64_t n_filter, double *score, int64_t *matches, int64_t *ninfo, int64_t *m,
               double *prob, double *L, double *LR) {
    if (!db) return fail(SNPM_E_ARG, "snpm_score: db is NULL");
    SNPM_CUDA(cudaSetDevice(db->device));
    const int64_t off[2] = {0, n};
    // one batch object lives with the handle: repeated calls reuse its device buffers, stream and events
    if (!db->scratch_batch_) SNPM_TRY(batch_new(db, &db->scratch_batch_));
    snpm_batch *b = db->scratch_batch_;
    int rc = batch_upload(b, 1, off, s_chrom_id, s_pos, wei);
    if (rc == SNPM_OK) rc = snpm_batch_set_row_filter(b, filter_rows, n_filter);
    if (rc == SNPM_OK) rc = snpm_batch_run(b, skip_db_hets, 0);
    if (rc == SNPM_OK) rc = snpm_batch_epilogue(b);
    if (rc == SNPM_OK) rc = snpm_batch_fetch(b, score, matches, ninfo, m, prob, L, LR);
    if (rc != SNPM_OK) { cudaStreamSynchronize(b->copy_stream); cudaStreamSynchronize(db->stream); }   // the host arrays may go away
    return rc;
}

int snpm_intersect(snpm_db *db, const int32_t *s_chrom_id, const int32_t *s_pos, int64_t n, int algo, int64_t *db_idx, int64_t *s_idx,
                   int64_t *m) {
    if (!db || !m || algo < 0 || algo > 2) return fail(SNPM_E_ARG, "snpm_intersect: bad arguments");
    const int64_t off[2] = {0, n};
    std::vector<double> wei(size_t(n) * 3, 0.0);
    snpm_batch *b = nullptr;
    SNPM_TRY(snpm_batch_create(db, 1, off, s_chrom_id, s_pos, wei.data(), &b));
    b->launches = 0;
    int rc = batch_join(b, algo);
    if (rc == SNPM_OK) { b->ran = true; rc = snpm_batch_wait(b, nullptr); }
    if (rc == SNPM_OK) rc = snpm_batch_fetch_pairs(b, 0, db_idx, s_idx, n, m);
    snpm_batch_destroy(b);
    return rc;
}

// ---- A2 / A4 stand-alone operators ------------------------------------------------------------------
int snpm_match_gts_accs(int device, const double *wei, const int8_t *snps, int64_t k, int32_t n_acc, int skip_hets_db, double *score,
                        int64_t *ninfo) {
    if (k < 0 || n_acc <= 0 || !score || !ninfo || (k > 0 && (!wei || !snps))) return fail(SNPM_E_ARG, "snpm_match_gts_accs: bad arguments");
    if (k >= (int64_t(1) << 31)) return fail(SNPM_E_ARG, "snpm_match_gts_accs: too many rows");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return fail(SNPM_E_CUDA, "snpm_match_gts_accs: no CUDA device (there is no CPU fallback)");
    SNPM_CUDA(cudaSetDevice(device));
    const int32_t stride = (((n_acc + 31) / 32) + 1) & ~1;
    const int64_t a_pad = int64_t(stride) * 32;
    std::vector<int32_t> iota(size_t(k) + 2);
    std::vector<double> w4(size_t(k) * 4);
    for (int64_t r = 0; r < k; ++r) {
        iota[size_t(r)] = int32_t(r);
        w4[size_t(4 * r)] = wei[3 * r];
        w4[size_t(4 * r + 1)] = wei[3 * r + 2];      // (w_ref, w_alt, w_het, 0)
        w4[size_t(4 * r + 2)] = wei[3 * r + 1];
        w4[size_t(4 * r + 3)] = 0.0;
    }
    const int32_t seg[2] = {0, int32_t(k)};
    struct Stream {
        cudaStream_t s = nullptr;
        ~Stream() { if (s) cudaStreamDestroy(s); }
    } own;
    SNPM_CUDA(cudaStreamCreateWithFlags(&own.s, cudaStreamNonBlocking));
    cudaStream_t st = own.s;
    DevBuf d_snps, d_packed, d_rows, d_w, d_seg, d_ps, d_pn;
    SNPM_TRY(d_snps.ensure(size_t(k) * n_acc));
    SNPM_TRY(d_packed.ensure(size_t(k) * stride * 8));
    SNPM_TRY(d_rows.ensure(size_t(k) * 4));
    SNPM_TRY(d_w.ensure(size_t(k) * 32));
    SNPM_TRY(d_seg.ensure(8));
    SNPM_TRY(d_ps.ensure(size_t(a_pad) * 8));
    SNPM_TRY(d_pn.ensure(size_t(a_pad) * 4));
    if (k > 0) {
        SNPM_CUDA(cudaMemcpyAsync(d_snps.p, snps, size_t(k) * n_acc, cudaMemcpyHostToDevice, st));
        SNPM_CUDA(cudaMemcpyAsync(d_rows.p, iota.data(), size_t(k) * 4, cudaMemcpyHostToDevice, st));
        SNPM_CUDA(cudaMemcpyAsync(d_w.p, w4.data(), size_t(k) * 32, cudaMemcpyHostToDevice, st));
        int *d_bad = d_seg.as<int>() + 4;            // DevBuf allocations hold at least 256 bytes
        SNPM_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
        k_pack_int8<<<grid_for(k * stride * 32, 256, 148), 256, 0, st>>>(d_snps.as<int8_t>(), k, n_acc, stride, d_packed.as<uint64_t>(), d_bad);
        SNPM_CUDA(cudaGetLastError());
        int bad = 0;
        SNPM_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
        SNPM_CUDA(cudaStreamSynchronize(st));
        if (bad > 0) return fail(SNPM_E_RANGE, "snpm_match_gts_accs: %d genotype codes above 2 (codes are 0 ref, 1 alt, 2 het, negative = missing)", bad);
    }
    SNPM_CUDA(cudaMemcpyAsync(d_seg.p, seg, 8, cudaMemcpyHostToDevice, st));
    ScoreArgs a = {};
    a.packed = d_packed.as<uint64_t>();
    a.stride = stride;
    a.pair_db = d_rows.as<int32_t>();
    a.pair_w = d_w.as<double>();
    a.table = 1;
    a.nseg = 1;
    a.seg_begin = d_seg.as<int32_t>();
    a.seg_end = d_seg.as<int32_t>() + 1;
    a.part_score = d_ps.as<double>();
    a.part_ninfo = d_pn.as<int32_t>();
    a.a_pad = int32_t(a_pad);
    SNPM_TRY(launch_score(st, a, 1, skip_hets_db != 0));
    std::vector<int32_t> ni(static_cast<size_t>(n_acc), 0);
    SNPM_CUDA(cudaMemcpyAsync(score, d_ps.p, size_t(n_acc) * 8, cudaMemcpyDeviceToHost, st));
    SNPM_CUDA(cudaMemcpyAsync(ni.data(), d_pn.p, size_t(n_acc) * 4, cudaMemcpyDeviceToHost, st));
    SNPM_CUDA(cudaStreamSynchronize(st));
    for (int32_t i = 0; i < n_acc; ++i) ninfo[i] = ni[size_t(i)];
    return SNPM_OK;
}

int snpm_calculate_likelihoods(int device, const double *scores, const double *ninfo, int64_t n_acc, int amin_is_calc, double amin,
                               double *prob, double *L, double *LR) {
    return snpm_calculate_likelihoods_many(device, scores, ninfo, 1, n_acc, amin_is_calc, amin, prob, L, LR);
}

int snpm_calculate_likelihoods_many(int device, const double *scores, const double *ninfo, int64_t S, int64_t K, int amin_is_calc, double amin,
                                    double *prob, double *L, double *LR) {
    if (S < 0 || K <= 0 || K >= (int64_t(1) << 30) || S > (int64_t(1) << 31) / 8 || (S > 0 && (!scores || !ninfo)))
        return fail(SNPM_E_ARG, "snpm_calculate_likelihoods_many: bad arguments");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return fail(SNPM_E_CUDA, "snpm_calculate_likelihoods_many: no CUDA device (there is no CPU fallback)");
    if (S == 0) return SNPM_OK;
    SNPM_CUDA(cudaSetDevice(device));
    // rows of the reduce-buffer layout k_epilogue reads: score[K] | ninfo[K] | m | y > n count
    const size_t SK = size_t(S) * size_t(K), pitch = 2 * size_t(K) + 2;
    std::vector<double> red(size_t(S) * pitch, 0.0);
    for (int64_t s = 0; s < S; ++s) {
        memcpy(red.data() + size_t(s) * pitch, scores + size_t(s) * K, size_t(K) * 8);
        memcpy(red.data() + size_t(s) * pitch + K, ninfo + size_t(s) * K, size_t(K) * 8);
    }
    DevBuf d_red, d_out;
    SNPM_TRY(d_red.ensure(red.size() * 8));
    SNPM_TRY(d_out.ensure(3 * SK * 8));
    SNPM_CUDA(cudaMemcpy(d_red.p, red.data(), red.size() * 8, cudaMemcpyHostToDevice));
    double *o = d_out.as<double>();
    SNPM_CUDA(launch_epilogue(nullptr, S, d_red.as<double>(), int64_t(pitch), int32_t(K), 0, amin_is_calc ? 0 : 1, amin, nullptr, nullptr, o, o + SK, o + 2 * SK));
    SNPM_CUDA(cudaGetLastError());
    SNPM_CUDA(cudaDeviceSynchronize());
    std::vector<double> viol(size_t(S), 0.0);
    SNPM_CUDA(cudaMemcpy2D(viol.data(), 8, d_red.as<double>() + 2 * K + 1, pitch * 8, 8, size_t(S), cudaMemcpyDeviceToHost));
    if (prob) SNPM_CUDA(cudaMemcpy(prob, d_out.p, SK * 8, cudaMemcpyDeviceToHost));
    if (L) SNPM_CUDA(cudaMemcpy(L, d_out.as<double>() + SK, SK * 8, cudaMemcpyDeviceToHost));
    if (LR) SNPM_CUDA(cudaMemcpy(LR, d_out.as<double>() + 2 * SK, SK * 8, cudaMemcpyDeviceToHost));
    for (int64_t s = 0; s < S; ++s)
        if (viol[size_t(s)] > 0.0)
            return fail(SNPM_E_ASSERT, "provided y is greater than n (row %lld, %lld accessions; likeliTest, snpmatch.py:43)", (long long)s, (long long)viol[size_t(s)]);
    return SNPM_OK;
}

// ---- 8(f)-4: genotype_cross window calls -----------------------------------------------------------------
int snpm_cross_window_genotypes(int device, const int64_t *par_idx, const int64_t *vcf_idx, int64_t m, const int32_t *win_start, int32_t n_windows,
                                const int8_t *p1, const int8_t *p2, int64_t n_par, const int8_t *gt, int64_t n_vcf, int32_t n_samples,
                                double lr_thres, int32_t n_marker_thres, int32_t *counts, int8_t *geno, uint8_t *borderline) {
    if (m < 0 || n_windows < 0 || n_par < 0 || n_vcf < 0 || n_samples < 0 || !win_start || (m > 0 && (!par_idx || !vcf_idx || !p1 || !p2 || !gt)))
        return fail(SNPM_E_ARG, "snpm_cross_window_genotypes: bad arguments");
    if (m >= (int64_t(1) << 31)) return fail(SNPM_E_ARG, "snpm_cross_window_genotypes: at most 2^31 - 1 matched markers");
    if (win_start[0] != 0 || win_start[n_windows] != m) return fail(SNPM_E_ARG, "snpm_cross_window_genotypes: win_start must run from 0 to m");
    for (int32_t w = 0; w < n_windows; ++w)
        if (win_start[w + 1] < win_start[w]) return fail(SNPM_E_ARG, "snpm_cross_window_genotypes: win_start is not ascending");
    for (int64_t k = 0; k < m; ++k)
        if (par_idx[k] < 0 || par_idx[k] >= n_par || vcf_idx[k] < 0 || vcf_idx[k] >= n_vcf)
            return fail(SNPM_E_ARG, "snpm_cross_window_genotypes: pair %lld points outside the marker lists", (long long)k);
    const size_t cells = size_t(n_windows) * size_t(n_samples);
    if (cells > 0 && (!counts || !geno)) return fail(SNPM_E_ARG, "snpm_cross_window_genotypes: NULL outputs");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return fail(SNPM_E_CUDA, "snpm_cross_window_genotypes: no CUDA device (there is no CPU fallback)");
    if (cells == 0) return SNPM_OK;
    SNPM_CUDA(cudaSetDevice(device));
    DevBuf d_pi, d_vi, d_ws, d_p1, d_p2, d_gt, d_cnt, d_geno, d_border;
    const size_t n_gt = size_t(n_vcf) * size_t(n_samples);
    SNPM_TRY(d_pi.ensure(size_t(m) * 8));
    if (m) SNPM_CUDA(cudaMemcpy(d_pi.p, par_idx, size_t(m) * 8, cudaMemcpyHostToDevice));
    SNPM_TRY(d_vi.ensure(size_t(m) * 8));
    if (m) SNPM_CUDA(cudaMemcpy(d_vi.p, vcf_idx, size_t(m) * 8, cudaMemcpyHostToDevice));
    SNPM_TRY(d_ws.ensure((size_t(n_windows) + 1) * 4));
    SNPM_CUDA(cudaMemcpy(d_ws.p, win_start, (size_t(n_windows) + 1) * 4, cudaMemcpyHostToDevice));
    SNPM_TRY(d_p1.ensure(size_t(n_par)));
    if (n_par) SNPM_CUDA(cudaMemcpy(d_p1.p, p1, size_t(n_par), cudaMemcpyHostToDevice));
    SNPM_TRY(d_p2.ensure(size_t(n_par)));
    if (n_par) SNPM_CUDA(cudaMemcpy(d_p2.p, p2, size_t(n_par), cudaMemcpyHostToDevice));
    SNPM_TRY(d_gt.ensure(n_gt));
    if (n_gt) SNPM_CUDA(cudaMemcpy(d_gt.p, gt, n_gt, cudaMemcpyHostToDevice));
    SNPM_TRY(d_cnt.ensure(cells * 12));
    SNPM_TRY(d_geno.ensure(cells));
    SNPM_TRY(d_border.ensure(cells));
    dim3 grid(unsigned(n_windows), unsigned((n_samples + GC_THREADS - 1) / GC_THREADS));
    k_gc_window_calls<<<grid, GC_THREADS>>>(d_pi.as<int64_t>(), d_vi.as<int64_t>(), d_ws.as<int32_t>(), d_p1.as<int8_t>(), d_p2.as<int8_t>(),
                                            d_gt.as<int8_t>(), n_samples, lr_thres, n_marker_thres, d_cnt.as<int32_t>(), d_geno.as<int8_t>(),
                                            d_border.as<uint8_t>());
    SNPM_CUDA(cudaGetLastError());
    SNPM_CUDA(cudaDeviceSynchronize());
    SNPM_CUDA(cudaMemcpy(counts, d_cnt.p, cells * 12, cudaMemcpyDeviceToHost));
    SNPM_CUDA(cudaMemcpy(geno, d_geno.p, cells, cudaMemcpyDeviceToHost));
    if (borderline) SNPM_CUDA(cudaMemcpy(borderline, d_border.p, cells, cudaMemcpyDeviceToHost));
    return SNPM_OK;
}

// ---- A9 ------------------------------------------------------------------------------------------------
// A shared marker panel: the panel-side GEMM operand is expanded once (snpm_panel_create) and every snpm_panel_score call
// re-uses it and the panel's scratch buffers (no allocation after the first call of a given batch size).
struct snpm_panel {
    snpm_db *db = nullptr;
    int64_t K = 0, Kpad = 0;
    int32_t n_kb = 0, n_blocks = 0, ld_out = 0;
    DevBuf d_rows, d_bt, d_codes, d_at, d_os, d_on, d_red, d_m, d_n64, d_p, d_l, d_lr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    ~snpm_panel() {
        for (cudaEvent_t e : ev)
            if (e) cudaEventDestroy(e);
    }
};

int snpm_panel_create(snpm_db *db, const int64_t *panel_rows, int64_t K, int skip_db_hets, snpm_panel **out) {
    if (!db || !out || K < 0 || (K > 0 && !panel_rows)) return fail(SNPM_E_ARG, "snpm_panel_create: bad arguments");
    if (K >= (int64_t(1) << 29)) return fail(SNPM_E_ARG, "snpm_panel_create: int32 accumulators hold at most 2^29 markers");
    *out = nullptr;
    SNPM_CUDA(cudaSetDevice(db->device));
    cudaStream_t st = db->stream;
    std::unique_ptr<snpm_panel> p(new (std::nothrow) snpm_panel);
    if (!p) return fail(SNPM_E_NOMEM, "snpm_panel_create: out of host memory");
    p->db = db;
    p->K = K;
    p->Kpad = std::max<int64_t>(OG_ROWS, ceil_div64(K, OG_ROWS) * OG_ROWS);
    p->n_kb = int32_t(p->Kpad / OG_ROWS);
    p->ld_out = int32_t(ceil_div64(db->n_acc, OG_BN) * OG_BN);
    p->n_blocks = p->ld_out / OG_BN;
    std::vector<int32_t> rows(size_t(p->Kpad), -1);
    for (int64_t k = 0; k < K; ++k) {
        const int64_t r = panel_rows[k] - db->row0_global;
        if (r < 0 || r >= db->n_rows) return fail(SNPM_E_ARG, "snpm_panel_create: panel row %lld is not on this device", (long long)panel_rows[k]);
        rows[size_t(k)] = int32_t(r);
    }
    SNPM_TRY(p->d_rows.ensure(size_t(p->Kpad) * 4));
    SNPM_TRY(p->d_bt.ensure(size_t(p->n_blocks) * p->n_kb * OG_B_TILE));
    for (cudaEvent_t &e : p->ev) SNPM_CUDA(cudaEventCreate(&e));
    SNPM_CUDA(cudaMemcpyAsync(p->d_rows.p, rows.data(), size_t(p->Kpad) * 4, cudaMemcpyHostToDevice, st));
    k_onehot_expand_panel<<<dim3(p->n_kb, p->n_blocks), 256, 0, st>>>(db->d_packed, db->stride, p->d_rows.as<int32_t>(), int32_t(p->Kpad),
                                                                      skip_db_hets ? 1 : 0, p->d_bt.as<unsigned char>());
    SNPM_KERNEL_CHECK();
    SNPM_CUDA(cudaStreamSynchronize(st));                        // `rows` leaves scope
    *out = p.release();
    return SNPM_OK;
}

void snpm_panel_destroy(snpm_panel *p) {
    if (!p) return;
    cudaSetDevice(p->db->device);
    delete p;
}

int snpm_panel_score(snpm_panel *p, const uint8_t *codes, int packed, int64_t S, int32_t *score, int32_t *ninfo, double *prob, double *L,
                     double *LR, float *ms) {
    if (!p || S < 1 || S > SNPM_PANEL_MAX_SAMPLES || (p->K > 0 && !codes) || !score || !ninfo) return fail(SNPM_E_ARG, "snpm_panel_score: bad arguments");
    snpm_db *db = p->db;
    SNPM_CUDA(cudaSetDevice(db->device));
    cudaStream_t st = db->stream;
    const int64_t K = p->K, Kpad = p->Kpad;
    const int32_t A = db->n_acc, ld_out = p->ld_out;
    const int m_blocks = int(ceil_div64(S, 64));
    const bool like = prob || L || LR;
    const int64_t dev_pitch = packed ? Kpad / 4 : Kpad, host_pitch = packed ? ceil_div64(K, 4) : K;
    SNPM_TRY(p->d_codes.ensure(size_t(S) * dev_pitch));
    SNPM_TRY(p->d_at.ensure(size_t(m_blocks) * p->n_kb * OG_A_TILE));
    SNPM_TRY(p->d_os.ensure(size_t(S) * ld_out * 4));
    SNPM_TRY(p->d_on.ensure(size_t(S) * ld_out * 4));
    if (like) {
        SNPM_TRY(p->d_red.ensure(size_t(S) * (2 * size_t(A) + 2) * 8));
        SNPM_TRY(p->d_m.ensure(size_t(S) * A * 8));
        SNPM_TRY(p->d_n64.ensure(size_t(S) * A * 8));
        SNPM_TRY(p->d_p.ensure(size_t(S) * A * 8));
        SNPM_TRY(p->d_l.ensure(size_t(S) * A * 8));
        SNPM_TRY(p->d_lr.ensure(size_t(S) * A * 8));
    }
    SNPM_CUDA(cudaEventRecord(p->ev[0], st));
    // markers past K (up to the k-block boundary) are absent: code 3 everywhere, then the caller's codes on top
    if (host_pitch != dev_pitch || K == 0) SNPM_CUDA(cudaMemsetAsync(p->d_codes.p, packed ? 0xFF : 3, size_t(S) * dev_pitch, st));
    if (K > 0) SNPM_CUDA(cudaMemcpy2DAsync(p->d_codes.p, size_t(dev_pitch), codes, size_t(host_pitch), size_t(host_pitch), size_t(S), cudaMemcpyHostToDevice, st));
    if (packed && (K & 3) && K > 0) {
        // the last byte of a row holds 1-3 markers: whatever the caller left in its spare bits must read as absent
        k_onehot_mask_tail<<<int(ceil_div64(S, 256)), 256, 0, st>>>(p->d_codes.as<uint8_t>(), S, dev_pitch, K);
    }
    if (packed) k_onehot_expand_samples<true><<<dim3(p->n_kb, m_blocks), 128, 0, st>>>(p->d_codes.as<uint8_t>(), int32_t(S), int32_t(Kpad), dev_pitch, p->d_at.as<unsigned char>());
    else k_onehot_expand_samples<false><<<dim3(p->n_kb, m_blocks), 128, 0, st>>>(p->d_codes.as<uint8_t>(), int32_t(S), int32_t(Kpad), dev_pitch, p->d_at.as<unsigned char>());
    SNPM_KERNEL_CHECK();
    OneHotGemmArgs g = {};
    g.a_tiled = p->d_at.as<unsigned char>(); g.b_tiled = p->d_bt.as<unsigned char>(); g.n_kb = p->n_kb; g.m_blocks = m_blocks; g.n_blocks = p->n_blocks;
    g.S = int32_t(S); g.out_score = p->d_os.as<int32_t>(); g.out_ninfo = p->d_on.as<int32_t>(); g.ld_out = ld_out;
    const size_t smem = size_t(OG_STAGES) * (OG_A_TILE + OG_B_TILE) + 1024;
    SNPM_CUDA(smem_attr<k_onehot_gemm>(int(smem)));
    dim3 grid((unsigned)std::min(m_blocks * p->n_blocks, db->n_sm));      // persistent: one CTA per SM walks the tiles
    SNPM_CUDA(cudaEventRecord(p->ev[1], st));
    k_onehot_gemm<<<grid, OG_THREADS, smem, st>>>(g);
    SNPM_KERNEL_CHECK();
    SNPM_CUDA(cudaEventRecord(p->ev[2], st));
    if (like) {
        dim3 tgrid(unsigned(S), unsigned(std::min((A + 255) / 256, 65535)));      // samples on x: any S the API takes
        k_onehot_totals<<<tgrid, 256, 0, st>>>(g.out_score, g.out_ninfo, ld_out, A, int32_t(K), p->d_red.as<double>());
        SNPM_CUDA(launch_epilogue(st, S, p->d_red.as<double>(), 2 * int64_t(A) + 2, A, 1, 0, 0.0, p->d_m.as<int64_t>(), p->d_n64.as<int64_t>(),
                                  p->d_p.as<double>(), p->d_l.as<double>(), p->d_lr.as<double>()));
        SNPM_KERNEL_CHECK();
    }
    // with one-hot weights the score IS the number of matches: the int32 accumulators go back as they are (pitched copy)
    SNPM_CUDA(cudaMemcpy2DAsync(score, size_t(A) * 4, p->d_os.p, size_t(ld_out) * 4, size_t(A) * 4, size_t(S), cudaMemcpyDeviceToHost, st));
    SNPM_CUDA(cudaMemcpy2DAsync(ninfo, size_t(A) * 4, p->d_on.p, size_t(ld_out) * 4, size_t(A) * 4, size_t(S), cudaMemcpyDeviceToHost, st));
    if (prob) SNPM_CUDA(cudaMemcpyAsync(prob, p->d_p.p, size_t(S) * A * 8, cudaMemcpyDeviceToHost, st));
    if (L) SNPM_CUDA(cudaMemcpyAsync(L, p->d_l.p, size_t(S) * A * 8, cudaMemcpyDeviceToHost, st));
    if (LR) SNPM_CUDA(cudaMemcpyAsync(LR, p->d_lr.p, size_t(S) * A * 8, cudaMemcpyDeviceToHost, st));
    SNPM_CUDA(cudaEventRecord(p->ev[3], st));
    SNPM_CUDA(cudaStreamSynchronize(st));
    if (ms) {
        ms[0] = ms[1] = ms[2] = 0.f;
        cudaEventElapsedTime(&ms[0], p->ev[0], p->ev[1]);      // H2D + operand expansion
        cudaEventElapsedTime(&ms[1], p->ev[1], p->ev[2]);      // GEMM
        cudaEventElapsedTime(&ms[2], p->ev[0], p->ev[3]);      // everything on the device, copies included
    }
    return SNPM_OK;
}

// one-shot form: panel operand, scoring, int64 results
int snpm_score_shared_panel(snpm_db *db, const int64_t *panel_rows, int64_t K, const uint8_t *codes, int64_t S, int skip_db_hets,
                            int64_t *score, int64_t *ninfo, double *prob, double *L, double *LR, float *ms_gemm) {
    if (!db || K < 0 || S < 1 || S > SNPM_PANEL_MAX_SAMPLES || (K > 0 && (!panel_rows || !codes)) || !score || !ninfo)
        return fail(SNPM_E_ARG, "snpm_score_shared_panel: bad arguments");
    snpm_panel *p = nullptr;
    SNPM_TRY(snpm_panel_create(db, panel_rows, K, skip_db_hets, &p));
    const size_t SA = size_t(S) * size_t(db->n_acc);
    std::vector<int32_t> s32, n32;
    try {
        s32.resize(SA);
        n32.resize(SA);
    } catch (const std::bad_alloc &) {
        snpm_panel_destroy(p);
        return fail(SNPM_E_NOMEM, "snpm_score_shared_panel: out of host memory");
    }
    float ms[3] = {0.f, 0.f, 0.f};
    const int rc = snpm_panel_score(p, codes, 0, S, s32.data(), n32.data(), prob, L, LR, ms);
    snpm_panel_destroy(p);
    if (rc != SNPM_OK) return rc;
    for (size_t i = 0; i < SA; ++i) {
        score[i] = s32[i];
        ninfo[i] = n32[i];
    }
    if (ms_gemm) *ms_gemm = ms[1];
    return SNPM_OK;
}

// ---- A5 + A6 ----------------------------------------------------------------------------------------
// phase 1 of `cross` on this device's rows: join, window bounds, one order-exact segment per window of every sample
// (window w of sample s in slot s*W + w)
static int windows_begin(snpm_batch *b, int skip_db_hets, int64_t bin_len, const int32_t *win_count, const int32_t *win_off,
                         int32_t n_windows, const int32_t *kmax, int64_t kmax_len, double lr_thres) {
    if (!b || bin_len <= 0 || n_windows < 0 || !win_count || !win_off || !kmax || kmax_len < 1)
        return fail(SNPM_E_ARG, "snpm_batch_run_windows: bad arguments");
    if (b->S < 1) return fail(SNPM_E_ARG, "snpm_batch_run_windows: the batch holds no sample");
    if (b->S * int64_t(n_windows) > INT32_MAX / 2)
        return fail(SNPM_E_ARG, "snpm_batch_run_windows: %lld samples x %d windows is too many window slots for one run", (long long)b->S, n_windows);
    if (b->grouped) return fail(SNPM_E_STATE, "snpm_batch_run_windows: windows need the batch in position order (snpm_batch_upload)");
    if (b->has_seg) return fail(SNPM_E_STATE, "snpm_batch_run_windows: windows do not honour the segregation filter; clear it first");
    snpm_db *db = b->db;
    SNPM_CUDA(cudaSetDevice(db->device));
    cudaStream_t st = db->stream;
    const int32_t W = n_windows, SW = int32_t(b->S) * n_windows;
    b->launches = 0;
    for (int i = 0; i < SNPM_N_EVENTS; ++i) b->ev_rec[i] = false;
    SNPM_TRY(batch_alloc_outputs(b, std::max<int64_t>(SW, 1)));
    const size_t WA = size_t(std::max(SW, 1)) * db->n_acc;
    SNPM_TRY(b->d_win_count.ensure(size_t(std::max(db->n_chr, 1)) * 4));
    SNPM_TRY(b->d_win_off.ensure(size_t(std::max(db->n_chr, 1)) * 4));
    SNPM_TRY(b->d_win_begin.ensure(size_t(std::max(SW, 1)) * 4));
    SNPM_TRY(b->d_win_end.ensure(size_t(std::max(SW, 1)) * 4));
    SNPM_TRY(b->d_win_nrows.ensure(size_t(std::max(SW, 1)) * 4));
    SNPM_TRY(b->d_win_zero.ensure(size_t(std::max(SW, 1)) * 4));
    SNPM_TRY(b->d_kmax.ensure(size_t(kmax_len) * 4));
    SNPM_TRY(b->d_win_L.ensure(WA * 8));
    SNPM_TRY(b->d_win_LR.ensure(WA * 8));
    SNPM_TRY(b->d_win_ident.ensure(WA));
    SNPM_TRY(b->d_win_amb.ensure(size_t(std::max(SW, 1)) * 4));
    if (db->n_chr) {
        SNPM_CUDA(cudaMemcpyAsync(b->d_win_count.p, win_count, size_t(db->n_chr) * 4, cudaMemcpyHostToDevice, st));
        SNPM_CUDA(cudaMemcpyAsync(b->d_win_off.p, win_off, size_t(db->n_chr) * 4, cudaMemcpyHostToDevice, st));
    }
    SNPM_CUDA(cudaMemcpyAsync(b->d_kmax.p, kmax, size_t(kmax_len) * 4, cudaMemcpyHostToDevice, st));
    b->kmax_len = kmax_len;
    rec(b, SNPM_EV_START);
    SNPM_TRY(batch_join(b, 0));
    SNPM_CUDA(cudaMemsetAsync(b->d_win_begin.p, 0, size_t(std::max(SW, 1)) * 4, st));
    SNPM_CUDA(cudaMemsetAsync(b->d_win_end.p, 0, size_t(std::max(SW, 1)) * 4, st));
    SNPM_CUDA(cudaMemsetAsync(b->d_win_zero.p, 0, size_t(std::max(SW, 1)) * 4, st));
    SNPM_CUDA(cudaMemsetAsync(b->d_win_nrows.p, 0, size_t(std::max(SW, 1)) * 4, st));
    if (b->n > 0 && W > 0) {
        k_window_bounds<<<int(ceil_div64(b->n, 256)), 256, 0, st>>>(b->d_pair_s.as<int32_t>(), b->d_mstart.as<int32_t>(), int32_t(b->S), W,
                                                                 b->d_chrom.as<int32_t>(), b->d_pos.as<int32_t>(), b->d_win_count.as<int32_t>(),
                                                                 b->d_win_off.as<int32_t>(), bin_len, b->d_win_begin.as<int32_t>(),
                                                                 b->d_win_end.as<int32_t>());
        k_window_nrows<<<(SW + 255) / 256, 256, 0, st>>>(b->d_win_begin.as<int32_t>(), b->d_win_end.as<int32_t>(), SW, b->d_win_nrows.as<int32_t>());
        SNPM_KERNEL_CHECK();
        b->launches += 2;
    }
    rec(b, SNPM_EV_JOIN);
    ScoreArgs a = {};
    a.packed = db->d_packed;
    a.stride = db->stride;
    a.pair_db = b->d_pair_db.as<int32_t>();
    a.pair_w = b->d_pair_w.as<double>();
    a.table = 1;
    a.nseg = SW;
    a.seg_begin = b->d_win_begin.as<int32_t>();
    a.seg_end = b->d_win_end.as<int32_t>();
    a.part_score = b->d_part_score.as<double>();
    a.part_ninfo = b->d_part_ninfo.as<int32_t>();
    a.a_pad = db->stride * 32;
    SNPM_TRY(launch_score(st, a, SW, skip_db_hets != 0));
    if (SW > 0) b->launches += 1;
    rec(b, SNPM_EV_SCORE);
    b->n_windows = W;
    b->bin_len = bin_len;
    b->lr_thres = lr_thres;
    b->win_pending = true;
    b->ran = b->ran_windows = b->epilogue_done = false;
    return SNPM_OK;
}

// phase 2: totals over the windows in order, per-window likelihoods / identity calls, compaction of the rows the reference keeps —
// on this device's partials, or on the sums over all ranks
static int windows_finish(snpm_batch *b) {
    snpm_db *db = b->db;
    cudaStream_t st = db->stream;
    const int32_t W = b->n_windows, SW = int32_t(b->S) * W;
    const size_t WA = size_t(std::max(SW, 1)) * db->n_acc;
    const int32_t a_pad = db->stride * 32;
    const double *part_score = b->d_part_score.as<double>();
    const int32_t *part_ninfo = b->d_part_ninfo.as<int32_t>();
    const int32_t *zero = b->d_win_zero.as<int32_t>(), *nrows = b->d_win_nrows.as<int32_t>();
    // per sample: totals over its W windows in window order; m = the pairs inside its windows (sum of the rows per window)
    dim3 cgrid((db->n_acc + 31) / 32, unsigned(b->S));
    k_combine<<<cgrid, 32, 0, st>>>(part_score, part_ninfo, a_pad, db->n_acc, nullptr, nullptr, W, zero, nrows, b->d_red.as<double>());
    SNPM_KERNEL_CHECK();
    b->launches += 1;
    if (SW > 0) {
        k_window_epilogue<<<SW, 256, 0, st>>>(part_score, part_ninfo, a_pad, db->n_acc, zero, nrows, b->d_kmax.as<int32_t>(), b->kmax_len,
                                             b->lr_thres, b->d_win_L.as<double>(), b->d_win_LR.as<double>(), b->d_win_ident.as<uint8_t>(),
                                             b->d_win_amb.as<int32_t>(), b->d_status.as<int>());
        SNPM_KERNEL_CHECK();
        b->launches += 1;
        // the rows the reference keeps, compacted on the device (what snpm_batch_fetch_window_rows reads back)
        SNPM_TRY(b->d_win_row_off.ensure(size_t(SW + 1) * 4));
        SNPM_TRY(b->d_row_acc.ensure(WA * 4));
        SNPM_TRY(b->d_row_score.ensure(WA * 8));
        SNPM_TRY(b->d_row_ninfo.ensure(WA * 4));
        SNPM_TRY(b->d_row_L.ensure(WA * 8));
        SNPM_TRY(b->d_row_ident.ensure(WA));
        k_window_row_offsets<<<1, 1024, 0, st>>>(b->d_win_amb.as<int32_t>(), SW, db->n_acc, b->d_win_row_off.as<int32_t>());
        SNPM_KERNEL_CHECK();
        k_window_compact<<<SW, 256, 0, st>>>(part_score, part_ninfo, a_pad, db->n_acc, b->d_win_L.as<double>(), b->d_win_LR.as<double>(),
                                            b->d_win_ident.as<uint8_t>(), b->d_win_row_off.as<int32_t>(), b->lr_thres, b->d_row_acc.as<int32_t>(),
                                            b->d_row_score.as<double>(), b->d_row_ninfo.as<int32_t>(), b->d_row_L.as<double>(),
                                            b->d_row_ident.as<uint8_t>());
        SNPM_KERNEL_CHECK();
        b->launches += 2;
    }
    SNPM_TRY(run_done(b));
    b->win_pending = false;
    b->ran_windows = true;
    return SNPM_OK;
}

int snpm_batch_run_windows(snpm_batch *b, int skip_db_hets, int64_t bin_len, const int32_t *win_count, const int32_t *win_off,
                           int32_t n_windows, const int32_t *kmax, int64_t kmax_len, double lr_thres) {
    SNPM_TRY(windows_begin(b, skip_db_hets, bin_len, win_count, win_off, n_windows, kmax, kmax_len, lr_thres));
    b->win_reduced = false;
    return windows_finish(b);
}

int snpm_batch_run_windows_begin(snpm_batch *b, int skip_db_hets, int64_t bin_len, const int32_t *win_count, const int32_t *win_off,
                                 int32_t n_windows, const int32_t *kmax, int64_t kmax_len, double lr_thres, void **dev_ptr, int64_t *n_doubles) {
    if (!dev_ptr || !n_doubles) return fail(SNPM_E_ARG, "snpm_batch_run_windows_begin: NULL output");
    if (b && b->S != 1) return fail(SNPM_E_ARG, "snpm_batch_run_windows_begin: windows on a sharded panel are scored for a single-sample batch");
    SNPM_TRY(windows_begin(b, skip_db_hets, bin_len, win_count, win_off, n_windows, kmax, kmax_len, lr_thres));
    snpm_db *db = b->db;
    const int64_t cells = int64_t(std::max(n_windows, 1)) * db->stride * 32;
    SNPM_TRY(b->d_win_red.ensure(size_t(2 * cells + std::max(n_windows, 1)) * 8));
    k_window_pack<<<int(ceil_div64(cells, 256)), 256, 0, db->stream>>>(b->d_part_score.as<double>(), b->d_part_ninfo.as<int32_t>(), b->d_win_nrows.as<int32_t>(),
                                                                      cells, n_windows, b->d_win_red.as<double>());
    SNPM_KERNEL_CHECK();
    b->launches += 1;
    *dev_ptr = b->d_win_red.p;
    *n_doubles = 2 * cells + n_windows;
    return SNPM_OK;
}

int snpm_batch_run_windows_finish(snpm_batch *b) {
    if (!b || !b->win_pending) return fail(SNPM_E_STATE, "snpm_batch_run_windows_finish: call snpm_batch_run_windows_begin first");
    snpm_db *db = b->db;
    SNPM_CUDA(cudaSetDevice(db->device));
    const int64_t cells = int64_t(std::max(b->n_windows, 1)) * db->stride * 32;
    k_window_unpack<<<int(ceil_div64(cells, 256)), 256, 0, db->stream>>>(b->d_win_red.as<double>(), cells, b->n_windows, b->d_part_score.as<double>(),
                                                                        b->d_part_ninfo.as<int32_t>(), b->d_win_nrows.as<int32_t>());
    SNPM_KERNEL_CHECK();
    b->launches += 1;
    b->win_reduced = true;
    return windows_finish(b);
}

// the matched-marker ranges of all window slots of the last windows run, shared by the two window fetches
struct WindowBounds {
    std::vector<int32_t> begin, end;
    int32_t m_all = 0;       // matched pairs of the batch
    int64_t total = 0;       // of them inside the windows
};

// Queues the read-back of the bounds behind the caller's copies on the batch's stream, then waits for the batch; win_nrows (when
// given) receives the rows of every window, on all ranks after a sharded run.
static int read_window_bounds(snpm_batch *b, int32_t *win_nrows, WindowBounds &wb) {
    cudaStream_t st = b->db->stream;
    const size_t W = size_t(b->S) * size_t(b->n_windows);
    std::vector<int32_t> nr(W + 1);
    wb.begin.resize(W + 1);
    wb.end.resize(W + 1);
    if (W) {
        SNPM_CUDA(cudaMemcpyAsync(wb.begin.data(), b->d_win_begin.p, W * 4, cudaMemcpyDeviceToHost, st));
        SNPM_CUDA(cudaMemcpyAsync(wb.end.data(), b->d_win_end.p, W * 4, cudaMemcpyDeviceToHost, st));
        SNPM_CUDA(cudaMemcpyAsync(nr.data(), b->d_win_nrows.p, W * 4, cudaMemcpyDeviceToHost, st));
    }
    SNPM_CUDA(cudaMemcpyAsync(&wb.m_all, b->d_prefix.as<int32_t>() + b->n, 4, cudaMemcpyDeviceToHost, st));
    SNPM_TRY(snpm_batch_wait(b, nullptr));
    for (size_t w = 0; w < W; ++w) {
        if (win_nrows) win_nrows[w] = nr[w];
        wb.total += wb.end[w] - wb.begin[w];
    }
    return SNPM_OK;
}

// matched_s_idx (when given): the sample index of every matched marker inside the windows, in window order
static int gather_window_markers(snpm_batch *b, const WindowBounds &wb, const char *fn, int64_t *matched_s_idx, int64_t capacity) {
    if (!matched_s_idx || wb.total == 0) return SNPM_OK;
    if (wb.total > capacity) return fail(SNPM_E_ARG, "%s: capacity %lld < %lld matched markers", fn, (long long)capacity, (long long)wb.total);
    cudaStream_t st = b->db->stream;
    std::vector<int32_t> ps(size_t(wb.m_all));
    SNPM_CUDA(cudaMemcpyAsync(ps.data(), b->d_pair_s.p, size_t(wb.m_all) * 4, cudaMemcpyDeviceToHost, st));
    SNPM_CUDA(cudaStreamSynchronize(st));
    int64_t o = 0;
    for (size_t w = 0; w + 1 < wb.begin.size(); ++w)
        for (int32_t r = wb.begin[w]; r < wb.end[w]; ++r) matched_s_idx[o++] = ps[size_t(r)];
    return SNPM_OK;
}

int snpm_batch_fetch_windows(snpm_batch *b, double *win_score, int32_t *win_ninfo, double *win_L, double *win_LR, uint8_t *win_identical,
                             int32_t *win_num_amb, int32_t *win_nrows, int64_t *matched_s_idx, int64_t capacity, int64_t *n_matched) {
    if (!b) return fail(SNPM_E_ARG, "snpm_batch_fetch_windows: NULL batch");
    if (!b->ran_windows) return fail(SNPM_E_STATE, "snpm_batch_fetch_windows: run the windows first");
    snpm_db *db = b->db;
    SNPM_CUDA(cudaSetDevice(db->device));
    cudaStream_t st = db->stream;
    const size_t W = size_t(b->S) * size_t(b->n_windows), A = size_t(db->n_acc), a_pad = size_t(db->stride) * 32;     // all window slots
    if (W) {
        if (win_score) SNPM_CUDA(cudaMemcpy2DAsync(win_score, A * 8, b->d_part_score.p, a_pad * 8, A * 8, W, cudaMemcpyDeviceToHost, st));
        if (win_ninfo) SNPM_CUDA(cudaMemcpy2DAsync(win_ninfo, A * 4, b->d_part_ninfo.p, a_pad * 4, A * 4, W, cudaMemcpyDeviceToHost, st));
        if (win_L) SNPM_CUDA(cudaMemcpyAsync(win_L, b->d_win_L.p, W * A * 8, cudaMemcpyDeviceToHost, st));
        if (win_LR) SNPM_CUDA(cudaMemcpyAsync(win_LR, b->d_win_LR.p, W * A * 8, cudaMemcpyDeviceToHost, st));
        if (win_identical) SNPM_CUDA(cudaMemcpyAsync(win_identical, b->d_win_ident.p, W * A, cudaMemcpyDeviceToHost, st));
        if (win_num_amb) SNPM_CUDA(cudaMemcpyAsync(win_num_amb, b->d_win_amb.p, W * 4, cudaMemcpyDeviceToHost, st));
    }
    WindowBounds wb;
    SNPM_TRY(read_window_bounds(b, win_nrows, wb));
    if (n_matched) *n_matched = wb.total;
    return gather_window_markers(b, wb, "snpm_batch_fetch_windows", matched_s_idx, capacity);
}


// The rows of windowscore.txt as the reference keeps them (csmatch.py:57-60), compacted on the device: for every window
// with 1 <= num_amb < n_acc its accessions with LR < lr_thres, in accession order.  win_row_off int32 [W+1] cuts the row
// arrays into windows; win_num_amb / win_nrows int32 [W] as snpm_batch_fetch_windows.  capacity in rows; *n_rows receives
// the row count (call with NULL row arrays to learn it).
int snpm_batch_fetch_window_rows(snpm_batch *b, int32_t *win_row_off, int32_t *win_num_amb, int32_t *win_nrows, int32_t *row_acc,
                                 double *row_score, int32_t *row_ninfo, double *row_L, uint8_t *row_identical, int64_t capacity,
                                 int64_t *n_rows, int64_t *matched_s_idx, int64_t matched_capacity, int64_t *n_matched) {
    if (!b || !n_rows) return fail(SNPM_E_ARG, "snpm_batch_fetch_window_rows: NULL argument");
    if (!b->ran_windows) return fail(SNPM_E_STATE, "snpm_batch_fetch_window_rows: run the windows first");
    snpm_db *db = b->db;
    SNPM_CUDA(cudaSetDevice(db->device));
    cudaStream_t st = db->stream;
    const size_t W = size_t(b->S) * size_t(b->n_windows);      // all window slots
    std::vector<int32_t> off(W + 1, 0);
    if (W) {
        SNPM_CUDA(cudaMemcpyAsync(off.data(), b->d_win_row_off.p, (W + 1) * 4, cudaMemcpyDeviceToHost, st));
        if (win_num_amb) SNPM_CUDA(cudaMemcpyAsync(win_num_amb, b->d_win_amb.p, W * 4, cudaMemcpyDeviceToHost, st));
    }
    WindowBounds wb;
    SNPM_TRY(read_window_bounds(b, win_nrows, wb));
    const int64_t R = off[W];
    *n_rows = R;
    if (win_row_off) memcpy(win_row_off, off.data(), (W + 1) * 4);
    if (n_matched) *n_matched = wb.total;
    if (R > 0 && (row_acc || row_score || row_ninfo || row_L || row_identical)) {
        if (R > capacity) return fail(SNPM_E_ARG, "snpm_batch_fetch_window_rows: capacity %lld < %lld rows", (long long)capacity, (long long)R);
        if (row_acc) SNPM_CUDA(cudaMemcpyAsync(row_acc, b->d_row_acc.p, size_t(R) * 4, cudaMemcpyDeviceToHost, st));
        if (row_score) SNPM_CUDA(cudaMemcpyAsync(row_score, b->d_row_score.p, size_t(R) * 8, cudaMemcpyDeviceToHost, st));
        if (row_ninfo) SNPM_CUDA(cudaMemcpyAsync(row_ninfo, b->d_row_ninfo.p, size_t(R) * 4, cudaMemcpyDeviceToHost, st));
        if (row_L) SNPM_CUDA(cudaMemcpyAsync(row_L, b->d_row_L.p, size_t(R) * 8, cudaMemcpyDeviceToHost, st));
        if (row_identical) SNPM_CUDA(cudaMemcpyAsync(row_identical, b->d_row_ident.p, size_t(R), cudaMemcpyDeviceToHost, st));
    }
    SNPM_TRY(gather_window_markers(b, wb, "snpm_batch_fetch_window_rows", matched_s_idx, matched_capacity));
    SNPM_CUDA(cudaStreamSynchronize(st));                       // the row copies
    return SNPM_OK;
}

// ---- A7 ---------------------------------------------------------------------------------------------
int snpm_batch_f1_pairs(snpm_batch *b, const int32_t *acc_idx, int32_t n_top, double *pair_score, int64_t *pair_ninfo) {
    if (!b || !acc_idx || n_top < 2 || n_top > 4096 || !pair_score || !pair_ninfo) return fail(SNPM_E_ARG, "snpm_batch_f1_pairs: bad arguments");
    if (!b->ran) return fail(SNPM_E_STATE, "snpm_batch_f1_pairs: run the batch first");
    if (b->S < 1 || b->S > 65535) return fail(SNPM_E_ARG, "snpm_batch_f1_pairs: %lld samples (1 to 65535 per call)", (long long)b->S);
    if (b->grouped) return fail(SNPM_E_STATE, "snpm_batch_f1_pairs: needs the batch in position order (snpm_batch_upload)");
    snpm_db *db = b->db;
    const int64_t S = b->S, SK = S * n_top;
    for (int64_t i = 0; i < SK; ++i)
        if (acc_idx[i] < 0 || acc_idx[i] >= db->n_acc)
            return fail(SNPM_E_ARG, "snpm_batch_f1_pairs: accession index %d of sample %lld out of range", acc_idx[i], (long long)(i / n_top));
    SNPM_CUDA(cudaSetDevice(db->device));
    cudaStream_t st = db->stream;
    const int n_pairs = n_top * (n_top - 1) / 2;
    const size_t SP = size_t(S) * size_t(n_pairs);
    // row blocks of the largest sample (a sample's matched pairs never outnumber its markers); the other samples' surplus blocks add zeros
    int64_t n_max = 0;
    for (int64_t s = 0; s < S; ++s) n_max = std::max(n_max, b->h_off[size_t(s) + 1] - b->h_off[size_t(s)]);
    const int n_blocks = int(std::max<int64_t>(1, ceil_div64(n_max, F1_ROWS_PER_BLOCK)));
    SNPM_TRY(b->d_f1_acc.ensure(size_t(SK) * 4));
    SNPM_TRY(b->d_f1_part.ensure(SP * n_blocks * 32));
    SNPM_TRY(b->d_f1_out.ensure(SP * 16));
    SNPM_CUDA(cudaMemcpyAsync(b->d_f1_acc.p, acc_idx, size_t(SK) * 4, cudaMemcpyHostToDevice, st));
    dim3 grid(n_blocks, n_pairs, unsigned(S));
    k_f1_partial<<<grid, F1_THREADS, 0, st>>>(db->d_packed, db->stride, b->d_pair_db.as<int32_t>(), b->d_pair_w.as<double>(),
                                              b->d_mstart.as<int32_t>(), b->d_f1_acc.as<int32_t>(), n_top, b->d_f1_part.as<double>());
    SNPM_KERNEL_CHECK();
    k_f1_final<<<int((SP + 127) / 128), 128, 0, st>>>(b->d_f1_part.as<double>(), n_blocks, int(SP), b->d_f1_out.as<double>());
    SNPM_KERNEL_CHECK();
    b->launches += 2;
    std::vector<double> out(SP * 2);
    SNPM_CUDA(cudaMemcpyAsync(out.data(), b->d_f1_out.p, SP * 16, cudaMemcpyDeviceToHost, st));
    SNPM_CUDA(cudaStreamSynchronize(st));
    for (size_t p = 0; p < SP; ++p) {
        pair_score[p] = out[2 * p];
        pair_ninfo[p] = int64_t(out[2 * p + 1]);
    }
    return SNPM_OK;
}

}  // extern "C"
