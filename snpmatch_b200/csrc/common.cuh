// Shared host/device helpers of libsnpmatch_b200 (error convention, device buffers, handle structs).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>
#include <cmath>

#include "../../include/snpmatch_b200.h"

namespace snpm {

extern thread_local std::string g_last_error;

inline int fail(int code, const char *fmt, ...) __attribute__((format(printf, 2, 3)));
inline int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

#define SNPM_CUDA(call)                                                                          \
    do {                                                                                         \
        cudaError_t e__ = (call);                                                                \
        if (e__ != cudaSuccess)                                                                  \
            return snpm::fail(SNPM_E_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call,          \
                              cudaGetErrorString(e__));                                          \
    } while (0)

#define SNPM_TRY(call)                 \
    do {                               \
        int rc__ = (call);             \
        if (rc__ != SNPM_OK) return rc__; \
    } while (0)

// launch check; with SNPM_SYNC_DEBUG=1 in the environment every launch is also waited for, so that a device fault is
// reported at the kernel that caused it
static inline bool snpm_sync_debug() {
    static int v = -1;
    if (v < 0) v = getenv("SNPM_SYNC_DEBUG") ? 1 : 0;
    return v == 1;
}
#define SNPM_KERNEL_CHECK()                                              \
    do {                                                                 \
        SNPM_CUDA(cudaGetLastError());                                   \
        if (snpm_sync_debug()) SNPM_CUDA(cudaDeviceSynchronize());       \
    } while (0)

// Grow-only device allocation, freed with its owner.  The owner makes the buffer's device current before it destroys it.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    int ensure(size_t bytes) {
        if (bytes <= cap && p) return SNPM_OK;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes < 256 ? 256 : bytes;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            p = nullptr;
            return fail(SNPM_E_NOMEM, "cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
        }
        cap = want;
        return SNPM_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace snpm

// ---------------------------------------------------------------------------------------------
// Handles
// ---------------------------------------------------------------------------------------------
struct snpm_db {
    int device = 0;
    int64_t n_rows = 0;       // rows of this shard
    int32_t n_acc = 0;
    int32_t n_words = 0;      // ceil(n_acc / 32)
    int32_t stride = 0;       // words per row (even -> 16-byte multiple)
    int64_t row0_global = 0;
    int32_t n_chr = 0;
    int n_sm = 148;
    uint64_t *d_packed = nullptr;
    int32_t *d_pos = nullptr;
    int64_t *d_chr_regions = nullptr;   // [n_chr,2], local rows
    int32_t *d_bucket = nullptr;        // coarse position index (k_build_buckets)
    int32_t *d_bucket_off = nullptr;    // [n_chr + 1]
    int bucket_shift = 0;
    unsigned long long *d_bitmap = nullptr;   // exact position index (k_bitmap_set / k_bitmap_rows), or null: bucket search
    int32_t *d_bm_first_row = nullptr;
    int64_t *d_bm_off = nullptr;         // [n_chr + 1] first bit of every chromosome
    std::vector<int64_t> h_chr_regions;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    snpm::DevBuf scratch;               // upload staging for int8 rows
    struct snpm_batch *scratch_batch_ = nullptr;   // reused by snpm_score
};

enum { SNPM_EV_START = 0, SNPM_EV_JOIN, SNPM_EV_SCORE, SNPM_EV_COMBINE, SNPM_EV_EPI_START, SNPM_EV_EPI_END, SNPM_EV_RED_START, SNPM_EV_RED_END, SNPM_N_EVENTS };

struct snpm_batch {
    snpm_db *db = nullptr;
    int64_t S = 0;            // samples
    int64_t n = 0;            // markers over all samples
    int64_t nseg_cap = 0;     // upper bound of 1000-row chunks over all samples
    std::vector<int64_t> h_off;
    // inputs (device)
    snpm::DevBuf d_off, d_chrom, d_pos, d_wei, d_filter;
    int64_t n_filter = 0;
    bool has_filter = false;  // snpm_batch_set_row_filter: a filter is set (possibly an empty one, which keeps nothing)
    // snpm_batch_set_segregation_filter: per sample the (word, mask) pairs its accession selection touches, cut by d_segsel_off
    snpm::DevBuf d_segsel, d_segsel_off;
    int64_t seg_S = 0;
    bool has_seg = false;
    snpm::DevBuf d_flags, d_flag_counts;   // snpm_batch_count_flagged_pairs
    // join products
    snpm::DevBuf d_match_row, d_tile_cnt, d_tile_off, d_prefix, d_pair_db, d_pair_s, d_pair_w;
    snpm::DevBuf d_mstart, d_seg_off;
    // scoring products
    snpm::DevBuf d_part_score, d_part_ninfo, d_red, d_matches, d_ninfo64, d_prob, d_L, d_LR, d_status;
    // windows
    int32_t n_windows = 0;
    int64_t bin_len = 0;
    double lr_thres = 3.841;
    snpm::DevBuf d_win_count, d_win_off, d_win_begin, d_win_end, d_kmax, d_win_L, d_win_LR, d_win_ident, d_win_amb;
    snpm::DevBuf d_win_nrows, d_win_zero, d_win_red;     // rows per window (summed over the ranks of a sharded run), zeros, the packed partials
    int64_t kmax_len = 0;
    bool win_pending = false;                            // snpm_batch_run_windows_begin done, _finish not yet
    bool win_reduced = false;                            // the last windows run went through the packed buffer (sharded run)
    snpm::DevBuf d_win_row_off, d_row_acc, d_row_score, d_row_ninfo, d_row_L, d_row_ident;   // surviving rows, compacted
    // f1
    snpm::DevBuf d_f1_acc, d_f1_part, d_f1_out;
    snpm::DevBuf d_pair_code;
    snpm::DevBuf d_wei_idx, d_wei_table;
    // grouped mode (snpm_batch_upload_grouped): markers ordered by weight triple, scored by k_score_grouped
    bool grouped = false;
    int32_t n_gtable = 0;
    int32_t chunk_rows = SNPM_CHUNK_ROWS, chunk_rows_req = SNPM_CHUNK_ROWS;   // position-order batches: rows per chunk of the fp64 kernel (snpm_batch_set_chunk_rows; latched at upload)
    int32_t gchunk = 320;              // rows per segment of the grouped kernels for the samples now on the device (latched at upload)
    int32_t gchunk_req = 320;          // snpm_batch_set_group_chunk: takes effect at the next grouped / coded upload
    bool gchunk_set = false;           // false: coded uploads pick 320 rows, or 496 on panels wider than one 36-word slice (measured)
    // coded mode (snpm_batch_upload_coded): position-order markers + weight codes; grouped on the device (group_sort.cuh)
    bool coded = false;
    bool codes_packed = false;         // the three codes of a marker in one uint32 (snpm_batch_upload_coded32)
    int32_t n_wtable = 0, code_bits = 0, key_bits = 0;
    int64_t n_sort_tiles = 0;
    snpm::DevBuf d_codes, d_wtable, d_key_a, d_pair_db_tmp, d_pair_s_tmp, d_tile_sample, d_tile_first,
                 d_tile_hist, d_blk_chg, d_seg_order, d_work_counter, d_hash, d_slot_gid, d_ngroups, d_group_overflow, d_gkeys, d_gw, d_goff;
    bool track_pairs = true;           // coded runs: also move the marker index of every pair into grouped order (snpm_batch_fetch_pairs)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;   // coded runs: block words + work order on the copy stream next to the partition pass
    cudaEvent_t ev_joined = nullptr;   // coded runs: after join + compaction, before the key sort (snpm_batch_coded_timings)
    snpm::DevBuf d_chrom8, d_gid, d_gtable, d_pair_gid, d_part_int, d_guard, d_runs;
    std::vector<double> h_gtable;
    std::vector<int32_t> h_tiles;      // coded mode: tile_first [S+1] | tile_sample [tiles] (staging of the asynchronous copy)
    // expansion of the compact upload forms, deferred to the head of the next run ON THE COMPUTE STREAM: a kernel on the copy
    // stream next to the scoring kernel cost 0.15 ms per step end to end (bit 0: run-length ids, 1: packed words, 2: byte chromosomes)
    int pending_expand = 0;
    int64_t pending_runs = 0;
    int *d_runs_bad = nullptr;         // inside d_runs: run-length coded ids whose ends do not ascend (last grouped_runs upload), or null
    int64_t red_pitch() const { return (grouped ? 3 : 2) * int64_t(db->n_acc) + 2; }   // doubles per sample row of d_red
    // state
    bool ran = false, ran_windows = false, epilogue_done = false;
    int launches = 0;
    // uploads run on the batch's own copy stream so that the H2D of one batch overlaps the kernels of another
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_uploaded = nullptr, ev_inputs_free = nullptr;
    cudaEvent_t ev[SNPM_N_EVENTS] = {};
    bool ev_rec[SNPM_N_EVENTS] = {};
    int *h_status = nullptr;  // pinned, 8 ints
    // asynchronous fetch (snpm_batch_fetch_async / _wait)
    cudaEvent_t ev_fetched = nullptr, ev_results = nullptr;
    double *h_tail = nullptr;   // pinned, 2 doubles per sample (matched pairs, y>n count)
    int64_t h_tail_cap = 0;
    int64_t *pend_m = nullptr;
    bool fetch_pending = false;
    // result range (snpm_batch_set_result_range): the epilogue and the fetches work on samples [res0, res0 + resn); resn < 0 = all
    int64_t res0 = 0, resn = -1;
    // one-shot reduce over peer memory (snpm_batch_ipc_*): the reduce buffers of the other ranks' batches, opened through CUDA IPC
    void *ipc_ptr = nullptr;             // d_red.p at export time: the allocation the peers have mapped
    std::vector<void *> peer_red;        // [world]; [rank] = own buffer
    int32_t ipc_rank = -1;
    size_t ipc_flags_off = 0;            // byte offset of the flag block inside the exported allocation (the same on every rank)
    uint32_t ipc_step = 0;               // reduces done since the export: the value the flags carry
    int64_t range0() const { return resn < 0 ? 0 : res0; }
    int64_t rangen() const { return resn < 0 ? S : resn; }
};
