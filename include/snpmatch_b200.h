/*
 * libsnpmatch_b200 — C ABI of the B200-native genotype-matching hot path.
 *
 * The reference (Gregor-Mendel-Institute/SNPmatch 5.0.1, pure Python) has no FFI layer; the
 * operator boundary on this path is a set of NumPy-in / NumPy-out functions.  Every entry point
 * below names the reference function it replaces (file:line relative to the reference tree).
 * The Python host (snpmatch_b200/core/*.py) binds these with ctypes over NumPy buffers;
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative SNPM_E_* code; the message of the last
 *     failure on the calling thread is snpm_last_error();
 *   - all pointers are caller-owned, contiguous, host memory unless the name ends in _dev;
 *   - a snpm_db is bound to ONE CUDA device and ONE stream; calls on a handle are stream-ordered
 *     and synchronous on return (except the *_async / batch_run calls, which say so);
 *     handles are not thread-safe;
 *   - there is NO CPU fallback: without a CUDA device snpm_db_create fails with SNPM_E_CUDA.
 *
 * Genotype codes (makedb.py:59, parsers.py:32-34): 0 hom-ref, 1 hom-alt, 2 het, -1 missing.
 * Packed form: code & 3 (3 = missing) as two bit planes; per row and per group of 32 accessions
 * one 64-bit word, low half = bit 0 of the 32 codes, high half = bit 1 (accession g*32+j is bit j).
 * Row stride = snpm_db_row_words() words (padded to a multiple of 2 words = 16 bytes); padding
 * accessions are missing.
 */
#ifndef SNPMATCH_B200_H
#define SNPMATCH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNPM_VERSION 100           /* 0.1.0 */

#define SNPM_OK            0
#define SNPM_E_ARG        -1       /* bad argument (shape, null pointer, unsorted keys) */
#define SNPM_E_CUDA       -2       /* CUDA runtime error / no device */
#define SNPM_E_NOMEM      -3
#define SNPM_E_STATE      -4       /* call order (e.g. fetch before run) */
#define SNPM_E_ASSERT     -5       /* the reference would have tripped an assert (y > n, snpmatch.py:43) */
#define SNPM_E_RANGE      -6       /* a compact encoding does not fit (too many distinct weight triples, chromosome id > 254) */

#define SNPM_CHUNK_ROWS 1000       /* Genotyper chunk_size, snpmatch.py:173 */

typedef struct snpm_db snpm_db;          /* HBM-resident packed panel (A0) */
typedef struct snpm_batch snpm_batch;    /* one or more samples resident on the device + their results */

/* ---- diagnostics ------------------------------------------------------------------------- */
int          snpm_version(void);
const char  *snpm_last_error(void);
int          snpm_device_count(void);
/* name_buf receives the device name; sm = major*10+minor; mem_bytes total global memory */
int          snpm_device_info(int device, char *name_buf, int name_len, int *sm, int64_t *mem_bytes, int *n_sm);

/* ---- A0: database container ---------------------------------------------------------------
 * Replaces pygwas/genotype.py:534-673 (HDF5Genotype.snps/positions/chr_regions) and
 * snp_genotype.py:26-41 (Genotype.__init__) as the thing the kernels read.
 * positions int32[n_rows] sorted ascending inside each chromosome; chr_regions int64[n_chr,2]
 * row ranges [start,end) in database order.  row0_global: index of this shard's first row in the
 * whole panel (0 on a single GPU) — returned db indices are global. */
int snpm_db_create(int device, int64_t n_rows, int32_t n_acc,
                   const int32_t *positions, const int64_t *chr_regions, int32_t n_chr,
                   int64_t row0_global, snpm_db **out);
int snpm_db_destroy(snpm_db *db);
/* streaming loaders: rows [row0, row0+n) of the shard, int8 [n, n_acc] C-order or packed words.  int8 codes: 0 ref, 1 alt,
 * 2 het, any negative value = missing (the reference masks every value < 0, snpmatch.py:84-86); values above 2 do not occur in
 * the reference's databases (makedb.py:59) and make the load fail with SNPM_E_RANGE (the rows may have been overwritten). */
int snpm_db_load_int8(snpm_db *db, int64_t row0, int64_t n, const int8_t *snps);
int snpm_db_load_packed(snpm_db *db, int64_t row0, int64_t n, const uint64_t *packed);
/* deterministic synthetic panel generated in HBM: code = f(seed, global row, accession), the same
 * integer hash as snpmatch_b200/synth.py:panel_codes_cols */
int snpm_db_fill_synthetic(snpm_db *db, uint64_t seed);
/* read back (tests / HDF5Genotype.snps[rows,:] equivalent, snpmatch.py:222): local row indices */
int snpm_db_read_rows_int8(snpm_db *db, const int64_t *rows, int64_t k, int8_t *out);
int snpm_db_read_packed(snpm_db *db, int64_t row0, int64_t n, uint64_t *out);
/* --refine support: flags[r] = 1 when the selected accession columns carry at least two different called genotypes on
 * row r — Genotype.identify_segregating_snps (snp_genotype.py:188-211, segregting_snps :378-383).  flags uint8[n_rows]. */
int snpm_db_segregating_rows(snpm_db *db, const int32_t *acc_idx, int32_t n_sel, uint8_t *flags);
/* whole accession columns: out int8 [n_sel, n_rows] (row-contiguous per column) = g_acc.snps[:, acc_idx[c]] of the reference's
 * column-chunked file (simulate.py:15,36-37; genotype_cross.py:97-98; csmatch.py:116-117), served by the one resident copy. */
int snpm_db_read_columns(snpm_db *db, const int32_t *acc_idx, int32_t n_sel, int8_t *out);
int64_t snpm_db_n_rows(const snpm_db *db);
int32_t snpm_db_n_acc(const snpm_db *db);
int32_t snpm_db_row_words(const snpm_db *db);
int64_t snpm_db_packed_bytes(const snpm_db *db);
/* run the handle's work on a caller-provided CUDA stream (cudaStream_t as void*); NULL = own stream */
int snpm_db_set_stream(snpm_db *db, void *cuda_stream);

/* ---- A1: (chrom,pos) join -----------------------------------------------------------------
 * Replaces Genotype.get_common_positions (snp_genotype.py:46-68) for a sample against the
 * resident database.  s_chrom_id[i] = index of the marker's chromosome in the database's
 * chromosome list (after the 'chr'-stripping of parsers.py:161), -1 when absent; markers must be
 * grouped by chromosome in database order with positions strictly ascending inside a chromosome
 * (the reference's implicit precondition, SURVEY A.1) — SNPM_E_ARG otherwise.
 * Outputs db_idx/s_idx int64[>= n], paired, ascending in db order; *m = number of pairs.
 * algo: 0 auto, 1 per-marker binary search, 2 merge-path. */
int snpm_intersect(snpm_db *db, const int32_t *s_chrom_id, const int32_t *s_pos, int64_t n,
                   int algo, int64_t *db_idx, int64_t *s_idx, int64_t *m);

/* ---- A2: matchGTsAccs ---------------------------------------------------------------------
 * Drop-in for matchGTsAccs(sampleWei, t1001snps, skip_hets_db) (snpmatch.py:74-89): k rows of
 * int8 codes [k, n_acc] (host) and weights f64 [k,3] -> score f64[n_acc], ninfo int64[n_acc],
 * summed in the reference's floating-point order (sequential over rows per class, then
 * ((0+ref)+het)+alt).  Independent of any snpm_db (device = the device to run on). */
int snpm_match_gts_accs(int device, const double *wei, const int8_t *snps, int64_t k, int32_t n_acc,
                        int skip_hets_db, double *score, int64_t *ninfo);

/* ---- A4: likelihood epilogue --------------------------------------------------------------
 * GenotyperOutput.calculate_likelihoods (snpmatch.py:106-117) + likeliTest (:40-55) +
 * get_fraction (:25-28): L, LR = L/nanmin(L) (nan when the minimum is <= 0 or nan); prob = y/n
 * (nan when n <= 0).  amin_is_calc != 0 -> nanmin, else use amin.  SNPM_E_ASSERT if any y > n. */
int snpm_calculate_likelihoods(int device, const double *scores, const double *ninfo, int64_t n_acc,
                               int amin_is_calc, double amin, double *prob, double *L, double *LR);
/* the same for S tables of K entries in one call (GenotyperOutput.calculate_likelihoods of many `--refine` tables, snpmatch.py:106-117
 * called from :218-219): scores / ninfo / prob / L / LR f64 [S,K], one nanmin per row.  Rows shorter than K are padded with
 * ninfo = 0 (L = nan there, which leaves the row's minimum as it is); every row gets the bits snpm_calculate_likelihoods gives
 * for it alone.  SNPM_E_ASSERT if any y > n. */
int snpm_calculate_likelihoods_many(int device, const double *scores, const double *ninfo, int64_t S, int64_t K,
                                    int amin_is_calc, double amin, double *prob, double *L, double *LR);

/* ---- A1+A2+A3+A4: Genotyper.genotyper for one or many samples ------------------------------
 * Replaces Genotyper.genotyper (snpmatch.py:207-233) + GenotyperOutput (:94-120).
 * A batch holds S samples: offsets int64[S+1] into the concatenated marker arrays
 * (s_chrom_id int32, s_pos int32, wei f64 [n,3]).  Each sample is scored on its own, exactly as
 * S separate `snpmatch inbred` runs would (README.md:9: one process per sample). */
int snpm_batch_create(snpm_db *db, int64_t n_samples, const int64_t *offsets,
                      const int32_t *s_chrom_id, const int32_t *s_pos, const double *wei,
                      snpm_batch **out);
/* replace the samples of an existing batch, reusing its device buffers.  The copies are queued on the
 * batch's own copy stream (after the kernels that still read the previous samples), so the upload of
 * one batch overlaps the scoring of another; snpm_batch_run waits for them on the device.  The host
 * arrays must stay alive until the next wait/fetch of this batch. */
int snpm_batch_upload(snpm_batch *b, int64_t n_samples, const int64_t *offsets,
                      const int32_t *s_chrom_id, const int32_t *s_pos, const double *wei);
/* same as snpm_batch_upload with the weights dictionary-coded: wei_idx uint16 [n,3] indexes `table` (f64, n_table <= 65536
 * entries, the exact host values, e.g. exp(-PL/10) for every integer PL of the file, or {0.0, 1.0} for called genotypes);
 * the device expands them to the f64 [n,3] weights bit for bit.  6 instead of 24 bytes per marker cross the PCIe bus. */
int snpm_batch_upload_indexed(snpm_batch *b, int64_t n_samples, const int64_t *offsets,
                              const int32_t *s_chrom_id, const int32_t *s_pos, const uint16_t *wei_idx,
                              const double *table, int32_t n_table);
/* ---- grouped order: the throughput path of likelihood-weighted scoring (k_score_grouped) -----------------------------
 * matchGTsAccs (snpmatch.py:74-89) adds one of three weights per matched row; exp(-PL/10) takes few distinct values
 * (parsers.py:147-151), so rows that share a weight triple can be COUNTED per accession and weighted once.
 *
 * snpm_group_markers (host code, no device needed; run once per sample set at parse time, like ParseInputs' npz cache,
 * parsers.py:96-98): assigns every marker the id of its weight triple (table f64 [*n_table, 3] in wei's column order,
 * at most min(table_cap, 65536) triples per call -> SNPM_E_RANGE beyond), and writes each sample's markers ordered by
 * (id, original order): chromosome ids as one byte (255 = not in the panel), positions, ids, and (optional) out_order =
 * index of the marker in the input arrays.  Weights must be finite and >= 0 (SNPM_E_ARG otherwise: use the position-order
 * path for such inputs). */
int snpm_group_markers(int64_t n_samples, const int64_t *offsets, const int32_t *s_chrom_id, const int32_t *s_pos,
                       const double *wei, uint8_t *out_chrom, int32_t *out_pos, uint16_t *out_gid, int64_t *out_order,
                       double *table, int32_t table_cap, int32_t *n_table);
/* replace the samples of a batch by grouped ones (7 bytes per marker cross the PCIe bus); asynchronous like
 * snpm_batch_upload.  Such a batch is scored with snpm_batch_run(mode 2) only; windows and the F1 pass need position order. */
int snpm_batch_upload_grouped(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint8_t *chrom_u8,
                              const int32_t *s_pos, const uint16_t *gid, const double *table, int32_t n_table);
/* the same with chromosome id and position of a marker in one word (id << 27 | position; id 31 = not in the panel): 6 bytes per
 * marker cross the PCIe bus.  snpm_pack_markers (host code) builds the words from snpm_group_markers' output, or answers
 * SNPM_E_RANGE when a chromosome id exceeds 30 or a position 2^27 - 1 (use snpm_batch_upload_grouped then). */
int snpm_pack_markers(int64_t n, const uint8_t *chrom_u8, const int32_t *pos, uint32_t *out);
int snpm_batch_upload_grouped_packed(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint32_t *chrom_pos,
                                     const uint16_t *gid, const double *table, int32_t n_table);
/* the same with the weight-triple ids run-length coded: markers are ordered by id inside a sample, so run r covers markers
 * [run_end[r-1], run_end[r]) (global marker indices, strictly ascending, the last one = offsets[n_samples]; a run never
 * crosses a sample boundary unless both sides carry the same id, which is harmless) and carries run_gid[r].  About
 * 4 + 6 / (markers per run) bytes per marker cross the PCIe bus (4.1 for PL samples of 50 k markers). */
int snpm_batch_upload_grouped_runs(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint32_t *chrom_pos,
                                   const uint16_t *run_gid, const uint32_t *run_end, int64_t n_runs, const double *table, int32_t n_table);
/* ---- coded upload: the grouping done on the device (group_sort.cuh) ---------------------------------------------------
 * What a parser has in hand (parsers.py:141-157) goes up as it is: markers in POSITION order as chrom_pos words (chromosome
 * id << 27 | position, id 31 = not in the panel: snpm_pack_markers) and, per marker, three dictionary codes in wei's column
 * order (ref, het, alt) into wtable (n_wtable <= 65536 distinct weight values, finite and >= 0; for a VCF the code is the
 * integer PL and wtable[k] = exp(-k/10)).  10 bytes per marker cross the PCIe bus and the host does no per-marker work.
 * snpm_batch_run(mode 2) then joins, builds a sort key per matched pair from its codes (called class | its code | code of the
 * class with fewer distinct weights | code of the other), orders every sample's pairs by that key (dense ids of the distinct keys
 * of a sample + one stable partition pass), marks where each class weight changes and scores with the persistent counting kernel
 * k_score_grouped2.  A sample with more than 2048 distinct weight triples is reported through snpm_batch_guard_counts (re-score it).  Replaces
 * snpm_group_markers + snpm_batch_upload_grouped*; results are identical (counts do not depend on the order inside a group).
 * Group chunks (snpm_batch_set_group_chunk) must be multiples of 16 and at most 496 rows for coded batches. */
int snpm_batch_upload_coded(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint32_t *chrom_pos,
                            const uint16_t *codes, const double *wtable, int32_t n_wtable);
/* host code, one pass over the markers: the chrom_pos words (chromosome id << 27 | position; id < 0 -> 31) from int32 ids and
 * positions and, when codes32 is not NULL, the three codes of a marker in one word (ref | het << 10 | alt << 20).  What
 * ParseInputs holds after parsers.py:141-157 -> what snpm_batch_upload_coded / _coded32 take.  SNPM_E_RANGE when an id exceeds
 * 30, a position 2^27 - 1 or (codes32 wanted) a code 1023. */
int snpm_pack_coded(int64_t n, const int32_t *chrom_id, const int32_t *pos, const uint16_t *codes, uint32_t *chrom_pos,
                    uint32_t *codes32);
/* the same with the three codes of a marker in one word, ref | het << 10 | alt << 20 (n_wtable <= 1024: e.g. integer PLs up to
 * 1023): 8 bytes per marker cross the PCIe bus */
int snpm_batch_upload_coded32(snpm_batch *b, int64_t n_samples, const int64_t *offsets, const uint32_t *chrom_pos,
                              const uint32_t *codes32, const double *wtable, int32_t n_wtable);
/* coded batches: keep (1, default) or drop (0) the marker index of every matched pair in grouped order.  The scoring path only
 * needs the panel rows; with 0 snpm_batch_fetch_pairs answers SNPM_E_STATE for coded batches and the grouping moves one array
 * instead of two. */
int snpm_batch_set_track_pairs(snpm_batch *b, int on);
/* device times (ms) of the last coded run's stages: [0] marker expansion + join + compaction, [1] key sort + change masks,
 * [2] scoring kernel, [3] combine; n >= 4 */
int snpm_batch_coded_timings(snpm_batch *b, float *ms, int n);
/* after snpm_batch_epilogue on a grouped batch: counts[s] = accessions of sample s whose fractional score part lies
 * within the rounding-error bound of an integer, i.e. whose int(score) depends on the reference's own summation order
 * (probability ~1e-7 per accession).  Re-score those samples with mode 0.  All zeros for position-order batches. */
int snpm_batch_guard_counts(snpm_batch *b, int32_t *counts);
/* Genotyper(chunk_size=...) (snpmatch.py:173,218): rows per chunk of the order-exact fp64 kernel (default SNPM_CHUNK_ROWS).  The
 * reference adds chunk sums, so the chunk size is part of its floating-point summation order; takes effect at the next
 * position-order upload.  The popcount kernel (mode 1) keeps 1000-row chunks: its integer sums do not depend on them. */
int snpm_batch_set_chunk_rows(snpm_batch *b, int32_t rows);
/* rows per segment of the grouped kernel (16..1008, a multiple of 8; coded uploads: a multiple of 16, at most 496); takes
 * effect at the next grouped or coded upload (the value is latched there: buffers are sized from it).  Unless this is called,
 * host-grouped uploads use 320 rows and coded uploads 320 rows on panels of up to 36 words per row (1152 accessions), 496 on
 * wider ones (measured: DESIGN 4.2b) */
int snpm_batch_set_group_chunk(snpm_batch *b, int32_t rows);
int snpm_batch_destroy(snpm_batch *b);
/* optional Genotyper.genotyper(filter_pos_ix=...) (snpmatch.py:211-216): keep only pairs whose
 * GLOBAL database row is in the sorted list (applies to every sample of the batch).  sorted_rows == NULL clears the filter;
 * a non-NULL list with n = 0 is an empty filter: no pair is kept (scores 0, as the reference with an empty filter_pos_ix) */
int snpm_batch_set_row_filter(snpm_batch *b, const int64_t *sorted_rows, int64_t n);
/* --refine for many samples at once (snpmatch.py:189-205 with Genotype.identify_segregating_snps, snp_genotype.py:188-211): a
 * per-sample accession selection.  sel uint32 [S, words] with words == snpm_db_row_words(db); bit j of sel[s][w] selects
 * accession 32w + j (the bit layout of a packed row; bits at or beyond n_acc: SNPM_E_ARG).  A marker of sample s that the join
 * matched to row r keeps its pair only when r segregates among s's selected accessions: at least two of the called classes
 * ref, alt, het occur there (missing calls do not count, het counts whatever skip_db_hets says), the predicate of
 * snpm_db_segregating_rows.  A selection of fewer than two accessions keeps no pair.  Kept pairs and their order are those of
 * snpm_batch_set_row_filter(segregating rows of sel[s]) on sample s alone, so mode-0 scores are bit-identical to that.  ANDs with
 * the row filter.  Honoured by snpm_batch_run modes 0 and 1; S must equal the batch's sample count at run time (SNPM_E_ARG
 * otherwise); mode 2 and the window runs answer SNPM_E_STATE while it is set.  sel == NULL clears it.  Copies, then returns. */
int snpm_batch_set_segregation_filter(snpm_batch *b, const uint32_t *sel, int64_t S, int32_t words);
/* after snpm_batch_run: counts int64[S] = pairs of sample s the run kept whose marker has flags[i] != 0; flags uint8 [n], one per
 * marker in upload order.  With flags = heterozygous calls this is getHeterozygosity's count (snpmatch.py:244-253) of every
 * sample at once.  Waits for the result. */
int snpm_batch_count_flagged_pairs(snpm_batch *b, const uint8_t *flags, int64_t *counts);
/* join + chunked scoring + per-sample totals; device work is queued on the db's stream and the
 * call returns without waiting (inputs already resident).
 * mode bits 0-7: scoring kernel — 0 = fp64 kernel in the reference's summation order (any weights);
 *                1 = popcount kernel for called genotypes (every weight row one-hot, as ParseInputs.get_wei_from_GT
 *                    produces, parsers.py:132-139; exact in any order; SNPM_E_ARG at wait/fetch otherwise);
 *                2 = grouped counting kernel (batches uploaded with snpm_batch_upload_grouped, any finite weights >= 0):
 *                    integers bit-exact, fp64 scores within a few ulp of the reference; see snpm_batch_guard_counts.
 * mode bits 8-15: join algorithm (0 auto, 1 binary search, 2 merge-path). */
int snpm_batch_run(snpm_batch *b, int skip_db_hets, int mode);
/* likelihood epilogue on the (possibly all-reduced) totals; queued, not waited for.  Grouped batches finalise their totals in
 * place, so their epilogue runs once per snpm_batch_run (a second call answers SNPM_E_STATE); position-order batches may repeat it. */
int snpm_batch_epilogue(snpm_batch *b);
/* wait for the queued work; ms_device = GPU time of the last run+epilogue measured with CUDA
 * events on the db's stream (may be NULL) */
int snpm_batch_wait(snpm_batch *b, float *ms_device);
/* restrict snpm_batch_epilogue, the fetches and snpm_batch_guard_counts to samples [first_sample, first_sample + n_samples)
 * (host arrays then hold n_samples rows); n_samples = -1 restores "all".  For sharded panels: after a reduce-SCATTER of the
 * reduce buffer every rank finishes and reads back only its share of the samples.  Persists across uploads. */
int snpm_batch_set_result_range(snpm_batch *b, int64_t first_sample, int64_t n_samples);
/* device address of the f64 reduce buffer [S, 2*n_acc+2]: per sample score[n_acc],
 * ninfo[n_acc] (as f64, exact), m, y>n violation count — the payload of the cross-GPU sum (8e).
 * Grouped batches: [S, 3*n_acc+2] = fractional part F | ninfo | m | violations | integer part I; the epilogue
 * turns F into the score after the reduce.  Until then the violation slot of a coded batch holds the grouping's overflow flag
 * (0 or 1 per shard): summed with the rest, it flags the sample on whichever rank finishes it. */
int snpm_batch_reduce_buffer(snpm_batch *b, void **dev_ptr, int64_t *n_doubles);
/* ---- 8(e): the cross-GPU sum as a one-shot reduce over peer memory (NVLink / NVSwitch), one process per GPU -------------
 * Every rank exports the reduce buffer of its batch (snpm_batch_ipc_export: a 64-byte CUDA IPC handle; the buffer holds
 * n_doubles values), the handles are exchanged by the host (any transport: torch.distributed.all_gather_object, MPI, a
 * file), and snpm_batch_ipc_open maps the world's buffers (handles = world x 64 bytes, in rank order; at most 16 ranks).
 * Per step, AFTER a cross-rank barrier that orders every rank's snpm_batch_run before it on the stream (the host's job:
 * e.g. a one-element NCCL all-reduce), snpm_batch_reduce_peers queues one kernel that sums, for the samples of this rank's
 * result range (snpm_batch_set_result_range), the rows of all ranks with 16-byte peer loads in rank order into the own
 * buffer — the reduce-scatter of sharding.reduce_scatter_batch without a collective library on the data path.  Before the
 * NEXT snpm_batch_run of any rank a second barrier must have passed (the peers may still be reading).  The batch must keep
 * its size between export and use (SNPM_E_STATE otherwise). */
int snpm_batch_ipc_export(snpm_batch *b, void *handle64, int64_t *n_doubles);
int snpm_batch_ipc_open(snpm_batch *b, const void *handles, int32_t world, int32_t rank);
int snpm_batch_reduce_peers(snpm_batch *b);
int snpm_batch_ipc_close(snpm_batch *b);
/* copy results to the host (any pointer may be NULL).  score f64[S,A] (untruncated),
 * matches int64[S,A] (= int(score), snpmatch.py:96), ninfo int64[S,A], m int64[S],
 * prob/L/LR f64[S,A]. */
int snpm_batch_fetch(snpm_batch *b, double *score, int64_t *matches, int64_t *ninfo, int64_t *m,
                     double *prob, double *L, double *LR);
/* snpm_batch_fetch in two halves: _async queues the copies (into pinned host buffers) behind the batch's kernels and returns,
 * _wait blocks until they have landed and reports the errors snpm_batch_fetch would.  guard (optional) receives
 * snpm_batch_guard_counts.  Between the two calls another batch may be run: its kernels overlap this batch's read-back. */
int snpm_batch_fetch_async(snpm_batch *b, double *score, int64_t *matches, int64_t *ninfo, int64_t *m,
                           double *prob, double *L, double *LR, int32_t *guard);
int snpm_batch_fetch_wait(snpm_batch *b);
/* matched pairs of sample s (global db rows, marker index inside the sample) — commonSNPs,
 * snpmatch.py:186-187.  capacity in elements; *m receives the pair count. */
int snpm_batch_fetch_pairs(snpm_batch *b, int64_t s, int64_t *db_idx, int64_t *s_idx, int64_t capacity, int64_t *m);
/* per-stage device times of the last run (ms): [0] join, [1] scoring kernel, [2] combine,
 * [3] epilogue, [4] whole run; plus the number of kernel launches in ms[5]; with n >= 8 also [6] the one-shot peer
 * reduce kernel of the last step (snpm_batch_reduce_peers) and [7] the part of it spent waiting for the slowest rank */
int snpm_batch_timings(snpm_batch *b, float *ms, int n);

/* one-call host-buffer form of the above for a single sample (upload, run, epilogue, fetch) */
int snpm_score(snpm_db *db, const int32_t *s_chrom_id, const int32_t *s_pos, const double *wei, int64_t n,
               int skip_db_hets, const int64_t *filter_rows, int64_t n_filter,
               double *score, int64_t *matches, int64_t *ninfo, int64_t *m,
               double *prob, double *L, double *LR);

/* ---- A5+A6: CrossIdentifier.window_genotyper ----------------------------------------------
 * Replaces csmatch.py:64-104 + get_window_data (:44-61) + genomes.get_bins_* (genomes.py:73-127)
 * for every sample of the batch (S >= 1).  Per database chromosome c: win_count[c] windows of bin_len bp
 * (0 when the chromosome is not in the genome JSON), first global window number win_off[c]
 * (0-based, in genome-JSON order).  n_windows = W = total per sample; window w of sample s sits in
 * slot s*W + w of every per-window array below.  kmax int32[kmax_len]: identity table,
 * identical <=> floor(n - x - 1) + 1 <= kmax[n] (built by the host with scipy.stats.binom.sf,
 * snpmatch.py:57-72).  Per sample, every result equals a run of that sample alone; totals (snpm_batch_fetch)
 * hold one row per sample, m = matched markers inside the sample's windows.  Device work is queued; fetch waits. */
int snpm_batch_run_windows(snpm_batch *b, int skip_db_hets, int64_t bin_len,
                           const int32_t *win_count, const int32_t *win_off, int32_t n_windows,
                           const int32_t *kmax, int64_t kmax_len, double lr_thres);
/* The same in two halves for a panel sharded by SNP-row ranges over several GPUs (SURVEY 8e): _begin joins the sample with this
 * device's rows, finds the windows' bounds and scores every window's local rows (windows without rows here give zeros), then
 * packs score | ninfo | rows of all windows into ONE device buffer of *n_doubles f64 (integers are exact in f64): the caller
 * sums it over the ranks in place (one all-reduce: a window's rows lie in one shard except at the <= G-1 shard boundaries, where
 * two ranks contribute); _finish unpacks the sums and runs totals, per-window likelihoods, identity calls and the compaction on
 * them.  Fetches then return the window rows of ALL ranks' markers; matched_s_idx stays this rank's (the caller concatenates).
 * fp64 window scores of the boundary windows are sums of two in-order partial sums (last bits may differ from the reference's
 * single in-order sum; integers do not).  Single-sample batches only. */
int snpm_batch_run_windows_begin(snpm_batch *b, int skip_db_hets, int64_t bin_len, const int32_t *win_count, const int32_t *win_off,
                                 int32_t n_windows, const int32_t *kmax, int64_t kmax_len, double lr_thres, void **dev_ptr,
                                 int64_t *n_doubles);
int snpm_batch_run_windows_finish(snpm_batch *b);
/* With SW = S * W window slots: win_score f64[SW,A], win_ninfo int32[SW,A], win_L f64[SW,A], win_LR f64[SW,A],
 * win_identical uint8[SW,A], win_num_amb int32[SW], win_nrows int32[SW] (matched markers per window),
 * matched_s_idx int64[capacity] in slot order (matchedTarInd, csmatch.py:90: sample 0's windows, then sample 1's, ...;
 * indices into the concatenated upload) with *n_matched; totals come from snpm_batch_fetch. */
int snpm_batch_fetch_windows(snpm_batch *b, double *win_score, int32_t *win_ninfo, double *win_L, double *win_LR,
                             uint8_t *win_identical, int32_t *win_num_amb, int32_t *win_nrows,
                             int64_t *matched_s_idx, int64_t capacity, int64_t *n_matched);
/* The rows of windowscore.txt exactly as the reference keeps them (get_window_data, csmatch.py:57-60), compacted on the
 * device: for every window with 1 <= num_amb < n_acc its accessions with LR < lr_thres, in accession order.
 * win_row_off int32 [S*W+1] cuts the row arrays (accession index, float score, informative sites, likelihood, identity
 * call) into window slots; win_num_amb / win_nrows int32 [S*W] and matched_s_idx as in snpm_batch_fetch_windows.  capacity in
 * rows, *n_rows receives the row count (call with NULL row arrays to learn it).  A few KB instead of the 21 bytes x W x A of
 * the full arrays cross the bus. */
int snpm_batch_fetch_window_rows(snpm_batch *b, int32_t *win_row_off, int32_t *win_num_amb, int32_t *win_nrows,
                                 int32_t *row_acc, double *row_score, int32_t *row_ninfo, double *row_L,
                                 uint8_t *row_identical, int64_t capacity, int64_t *n_rows, int64_t *matched_s_idx,
                                 int64_t matched_capacity, int64_t *n_matched);

/* ---- A7: simulated F1 pass ----------------------------------------------------------------
 * Replaces the loop body of CrossIdentifier.match_insilico_f1s (csmatch.py:115-126) for every sample
 * of the batch over its whole-genome join: all P = n_top*(n_top-1)/2 pairs (i<j in list order) of the
 * sample's accession columns.  acc_idx int32[S, n_top] row-major, pair_score f64[S, P], pair_ninfo int64[S, P];
 * a sample's sums are the ones a single-sample batch of it gives, bit for bit.  Limits (SNPM_E_ARG, the value named):
 * 2 <= n_top <= 4096, every index in 0..n_acc-1 (a list may repeat one), 1 <= S <= 65535, S * P <= INT32_MAX, and at
 * most 65535 row blocks of 4096 markers (268 M markers) in the largest sample. */
int snpm_batch_f1_pairs(snpm_batch *b, const int32_t *acc_idx, int32_t n_top,
                        double *pair_score, int64_t *pair_ninfo);

/* ---- 8(f)-3: pairwiseScore ------------------------------------------------------------------
 * The counting loop of pairwiseScore (snpmatch.py:291-297) over the matched marker pairs (idx1, idx2: outputs of the join,
 * snpmatch.py:276-284) of two samples: common[c] = pairs on chromosome c, matches[c] = pairs whose genotype strings are
 * equal.  chrom1 int32[n1] = chromosome id of every marker of sample 1 (0..n_chr-1; others are not counted), gt1 int32[n1]
 * / gt2 int32[n2] = ids of the genotype strings in a table shared by both samples.  common/matches int64[n_chr]. */
int snpm_pair_match_counts(int device, const int64_t *idx1, const int64_t *idx2, int64_t m, const int32_t *chrom1, const int32_t *gt1,
                           int64_t n1, const int32_t *gt2, int64_t n2, int32_t n_chr, int64_t *common, int64_t *matches);

/* ---- 8(f)-3 for many samples: every pair's shared-marker identity in one tensor-core pass -------------------------
 * pairwiseScore (snpmatch.py:270-309) for all S x S pairs at once: its counting loop (:291-297) over the markers two
 * samples share becomes one-hot int8 GEMMs (tcgen05, int32 accumulation, exact) over the columns of the union of all
 * samples' markers.  Sample s has the markers offsets[s] .. offsets[s+1]-1 (offsets int64[S+1], offsets[0] = 0); col
 * int32[n] = the union column of each (strictly ascending inside a sample, < K), cls uint8[n] = the id of its GT string
 * (< n_cls, 1 <= n_cls <= 8: identical strings, identical ids).  chr_start int64[C+1] = the column range of each chromosome
 * (non-decreasing from 0 to K).  Out: common / same int32 [C,S,S] = per chromosome the columns samples i and j both have,
 * and how many of those carry the same class in both.
 * The columns are walked chromosome by chromosome in chunks of chunk_markers columns (0 = as many as fit
 * SNPM_PAIR_CHUNK_BYTES of operand tiles); a chunk never spans two chromosomes.  Only the CSR crosses PCIe (about 5 bytes
 * per marker); the operands of a chunk are expanded from it on the device.  Refused before any allocation: S outside
 * 1..SNPM_PAIR_MAX_SAMPLES, K >= 2^31, a chromosome of 2^31 columns or more (the counts are int32), and malformed input
 * (the error names the sample).  ms (optional) float[3]: device time of the operand expansion with its memsets, of the
 * GEMMs, and of the whole call including the copies. */
#define SNPM_PAIR_MAX_SAMPLES 8192          /* bounds the [C,S,S] outputs: 512 MB of both counts per chromosome at 8192 */
#define SNPM_PAIR_CHUNK_BYTES ((int64_t)1 << 30)
int snpm_pair_matrix(int device, int64_t S, const int64_t *offsets, const int32_t *col, const uint8_t *cls, int32_t n_cls, int64_t K,
                     const int64_t *chr_start, int32_t C, int64_t chunk_markers, int32_t *common, int32_t *same, float *ms);

/* ---- accession against accession: every pair of panel accessions in one tensor-core pass --------------------------
 * pairwiseScore's statistic for two accession columns of the resident panel, for every pair of the selection acc_idx
 * int32[n_sel] (indices into the panel's accessions, in output order), over the rows this handle holds:
 *   common[i, j] = rows on which accessions acc_idx[i] and acc_idx[j] are both called (code 0, 1 or 2),
 *   same[i, j]   = those of them with equal codes (het equals het).
 * With skip_db_hets, code 2 counts as missing.  Out: common / same int32 [n_sel, n_sel], full and symmetric; common[i, i] is the
 * number of called rows of accession i.  Two row shards of one panel give counts that sum to the whole panel's.
 * Both one-hot operands of a chunk of rows are expanded from the packed panel on the device (nothing but acc_idx crosses
 * PCIe on the way in) and multiplied with k_onehot_gemm: 12 n_sel operand bytes per row, and 16 n_i n_j int8 operations per
 * row for a block pair of n_i and n_j accessions (16 n_sel^2 when the selection is one block).
 * The rows are walked in chunks of chunk_rows rows (0 = as many as fit SNPM_PAIR_CHUNK_BYTES of operand tiles; a chunk may
 * span chromosomes).  The output is computed in blocks of block_acc accessions (0 = SNPM_ACC_BLOCK; a positive multiple of
 * 256): block pairs bi <= bj, the blocks below the diagonal mirrored from the ones above, so a selection of 20 000 runs as
 * 3 blocks and 6 block pairs.  Refused before any allocation, with the value named: n_sel < 1, an index outside 0..A-1,
 * block_acc not a positive multiple of 256, chunk_rows < 0, and a handle of 2^31 rows or more (the counts are int32).
 * ms (optional) float[3]: device time of the operand expansion, of the GEMMs, and of the whole call including the copies. */
#define SNPM_ACC_BLOCK 8192
int snpm_db_acc_pairs(snpm_db *db, const int32_t *acc_idx, int32_t n_sel, int skip_db_hets, int64_t chunk_rows, int32_t block_acc,
                      int32_t *common, int32_t *same, float *ms);

/* ---- 8(f)-4: genotype_cross -----------------------------------------------------------------
 * The window loop of GenotypeCross.genotype_cross (genotype_cross.py:210-241): for every genome window w and every sample s
 * of a multi-sample VCF, over the matched pairs k in [win_start[w], win_start[w+1]) (par_idx into the parents' segregating
 * markers, vcf_idx into the VCF markers; ordered by window): counts int32 [W,S,3] = calls equal to parent 1, heterozygous
 * calls, calls equal to parent 2 (get_window_genotype_gts :188-199), and geno int8 [W,S] = getWindowGenotype (:21-49) of
 * those counts with totalMarkers = pairs of the window: 0 parent 1, 1 het, 2 parent 2, -1 NA.  p1/p2 int8[n_par] parental
 * codes, gt int8 [n_vcf, S] parseGT codes.  borderline (optional) uint8 [W,S]: the call hangs on lr_next >= lr_thres
 * within 1e-9 relative. */
int snpm_cross_window_genotypes(int device, const int64_t *par_idx, const int64_t *vcf_idx, int64_t m, const int32_t *win_start, int32_t n_windows,
                                const int8_t *p1, const int8_t *p2, int64_t n_par, const int8_t *gt, int64_t n_vcf, int32_t n_samples,
                                double lr_thres, int32_t n_marker_thres, int32_t *counts, int8_t *geno, uint8_t *borderline);

/* ---- A9: batched scoring on a shared marker panel (tensor cores) ------------------------------
 * No reference symbol: the reference scores many samples as one process per sample (README.md:9).  S samples of CALLED
 * genotypes that share K markers (panel_rows int64[K], global rows; codes uint8 [S,K]: 0 ref, 1 alt, 2 het, 3 or more = sample
 * lacks the marker) are scored against every accession as one one-hot int8 GEMM on tcgen05 (int32 accumulation, exact):
 * score/ninfo int64 [S,A] equal what snpm_score returns per sample with one-hot weights; prob/L/LR f64 [S,A] optional.
 * 1 <= S <= SNPM_PANEL_MAX_SAMPLES (one launch row per 64 samples, at most 65 535 rows); more is SNPM_E_ARG.
 * ms_gemm (optional) receives the device time of the GEMM kernel. */
#define SNPM_PANEL_MAX_SAMPLES (65535 * 64)
int snpm_score_shared_panel(snpm_db *db, const int64_t *panel_rows, int64_t K, const uint8_t *codes, int64_t S, int skip_db_hets,
                            int64_t *score, int64_t *ninfo, double *prob, double *L, double *LR, float *ms_gemm);

/* The same as an object, for callers that score batch after batch on one marker panel: snpm_panel_create expands the panel-side
 * GEMM operand once (K markers x A accessions one-hot, 4 bytes per cell, resident), snpm_panel_score re-uses it and the
 * panel's scratch buffers (nothing is allocated after the first call of a given S).  codes: packed = 0 -> uint8 [S,K] as
 * above; packed = 1 -> 2 bits per marker, four markers per byte (marker k in bits 2(k&3), 2(k&3)+1 of byte k >> 2 of the
 * sample's row; rows are ceil(K/4) bytes; spare bits of the last byte are ignored), a quarter of the bytes over PCIe.
 * score / ninfo int32 [S,A]: with called genotypes the score is the number of matches (snpmatch.py:96 truncates nothing), so
 * the int32 accumulators are returned as they are; prob/L/LR f64 [S,A] optional (all three NULL skips the likelihood
 * epilogue).  Pass page-locked host buffers for full PCIe speed.  ms (optional) float[3]: device time of H2D + sample
 * operand expansion, of the GEMM, and of the whole call including the copies back. */
typedef struct snpm_panel snpm_panel;
int snpm_panel_create(snpm_db *db, const int64_t *panel_rows, int64_t K, int skip_db_hets, snpm_panel **out);
int snpm_panel_score(snpm_panel *p, const uint8_t *codes, int packed, int64_t S, int32_t *score, int32_t *ninfo, double *prob, double *L,
                     double *LR, float *ms);
void snpm_panel_destroy(snpm_panel *p);

/* ---- multi-sample VCF text on the device (`inbred --samples_vcf`, `cross --samples_vcf`) ----------------------------------
 * No reference symbol: the reference reads one sample column per scikit-allel call (parsers.py:184-213).  A handle parses the
 * genotype columns of the records of one VCF, chunk by chunk, for n_samples sample columns (the #CHROM line's).  The caller
 * passes whole lines: text [n_bytes] with 1 <= n_bytes <= chunk_bytes <= SNPM_VCF_MAX_CHUNK, ending in a line end; '\n',
 * "\r\n" and a lone '\r' each end a line (Python's universal newlines).  Lines starting with '#' and lines of fewer than 10
 * tab-separated fields are not records.
 * snpm_vcf_parse: info int64[5] = lines, cells of samples 0..n_samples-1 in records, called cells kept, 1 if the chunk holds a
 * byte >= 0x80, lines starting with "##INFO=<ID=DP,"; ms (optional) float[2] = device time of the copy up and of the kernels.
 * snpm_vcf_fetch, per line (n = info[0]): line_start int32[n+1] (byte offsets; line k is [line_start[k], line_start[k+1])
 * with its line end), flags int32[n] (1 record, 2 the device cannot reproduce the Python parser on this record: re-parse it,
 * 4 FORMAT has a PL key, 8 CHROM may differ from the previous record's), nsf int32[n] sample fields, pos int32[n], dp int32[n]
 * (INFO DP, -1 none), chrom_len int32[n] bytes of CHROM.  Per sample s, entries sample_off[s] .. sample_off[s+1]-1 (int32
 * [n_samples+1]) are its called cells in line order, records flagged 2 left out: line int32, cls uint16 = a1 * 111 + a2 of the
 * rendered GT's two alleles (0 '.', 1 + d for the digit d, 11 + 10x + y for the digits xy), pl int32 [3] (-1 missing). */
#define SNPM_VCF_MAX_CHUNK (int64_t(1) << 30)
typedef struct snpm_vcf snpm_vcf;
int snpm_vcf_create(int device, int32_t n_samples, int64_t chunk_bytes, snpm_vcf **out);
int snpm_vcf_parse(snpm_vcf *h, const char *text, int64_t n_bytes, int64_t *info, float *ms);
int snpm_vcf_fetch(snpm_vcf *h, int32_t *line_start, int32_t *flags, int32_t *nsf, int32_t *pos, int32_t *dp, int32_t *chrom_len,
                   int32_t *sample_off, int32_t *line, uint16_t *cls, int32_t *pl);
/* `makedb --no_csv`: the same handle and chunks, parsed with the rules of the reference's makedb CSV (makedb.py:34-62) into
 * rows of the packed panel, no per-cell array.  A record's calls are taken from the FIRST GT key of FORMAT; the GT text maps by
 * exact match: 0/0 0|0 -> 0, 1/1 1|1 -> 1, 0/1 0|1 1/0 1|0 -> 2, ./. .|. . -> missing; a record without GT and a cell without
 * that subfield are missing; any other text is missing and counted.
 * snpm_vcf_parse_gt_packed: info int64[4] = lines, rows, the counted calls, 1 if the chunk holds a byte >= 0x80; ms (optional)
 * float[2] as for snpm_vcf_parse.
 * snpm_vcf_fetch_gt_packed, per line (n = info[0]): line_start int32[n+1], flags int32[n] (1 record, 2 POS is not 1-9 plain
 * digits: pos is not set, convert the text on the host; 8 CHROM may differ from the previous record's), nsf int32[n], pos
 * int32[n], chrom_len int32[n] as for snpm_vcf_fetch; packed uint64 [info[1], stride] with stride = snpm_db_row_words of a
 * panel of n_samples accessions, in the layout of snpm_db_load_packed: one row per record with exactly n_samples sample fields,
 * in line order (a record with another count gets no row, and flag 8 is left unset on it). */
int snpm_vcf_parse_gt_packed(snpm_vcf *h, const char *text, int64_t n_bytes, int64_t *info, float *ms);
int snpm_vcf_fetch_gt_packed(snpm_vcf *h, int32_t *line_start, int32_t *flags, int32_t *nsf, int32_t *pos, int32_t *chrom_len,
                             uint64_t *packed);
/* `genotype_cross --gpu_parse`: the same handle and chunks, every record read into one row of int8 window-call codes, the codes
 * the reference's parseGT gives the GT strings of its import_vcf_file (parsers.py:12-35, 178-213).  A record's calls are taken
 * from the FIRST GT key of FORMAT, split at '/' and '|', the first two tokens kept (a missing or empty one is '.'), each matched
 * exactly: (1,1) -> 1, (0,1) (1,0) -> 2, (.,.) -> -1, any other pair -> 0; a record without GT, a cell without that subfield and
 * the cells past the record's sample fields are -1; sample fields past n_samples are ignored.  No cell is left to the host.
 * snpm_vcf_parse_gt_codes: info int64[3] = lines, rows, 1 if the chunk holds a byte >= 0x80; ms (optional) float[2] as for
 * snpm_vcf_parse.
 * snpm_vcf_fetch_gt_codes, per line (n = info[0]): line_start, flags, nsf, pos, chrom_len as for snpm_vcf_fetch_gt_packed (flag
 * 2: POS is not 1-9 plain digits, convert the text on the host); codes int8 [info[1], n_samples]: one row per record, in line
 * order, whatever its number of sample fields. */
int snpm_vcf_parse_gt_codes(snpm_vcf *h, const char *text, int64_t n_bytes, int64_t *info, float *ms);
int snpm_vcf_fetch_gt_codes(snpm_vcf *h, int32_t *line_start, int32_t *flags, int32_t *nsf, int32_t *pos, int32_t *chrom_len,
                            int8_t *codes);
void snpm_vcf_destroy(snpm_vcf *h);

/* ---- BGZF-compressed VCFs inflated on the device (the `.vcf.gz` input of the device VCF readers) --------------------------
 * No reference symbol: the reference reads `.vcf.gz` through scikit-allel and zlib on the host.  BGZF (bgzip, `bcftools -Oz`)
 * is a series of independent gzip members, each with FLG = FEXTRA, a `BC` extra subfield holding its size - 1, and at most
 * 65536 bytes of text (ISIZE); the file may end with the empty 28-byte EOF member.
 * snpm_bgzf_scan (host only, no device): walks the member headers of data[0..n_bytes).  *n_members = the number of members
 * when the file is all BGZF -- every member has ID1 ID2 = 1f 8b, CM 8, FLG exactly 4, an extra field with a BC subfield and
 * ISIZE <= 65536, and the members tile the data to its last byte -- or -1 otherwise (no member at all counts as not BGZF).
 * The first min(n, cap) members' byte offsets go to member_off (and member_off[n] = n_bytes when n <= cap; cap + 1 entries)
 * and their ISIZE to isize (cap entries).  Call again with cap >= n when n > cap.
 * snpm_bgzf_create: a handle with pinned staging for up to max_in_bytes of members and max_out_bytes of text per call
 * (each at most SNPM_BGZF_MAX_BYTES) and the device buffers.
 * snpm_bgzf_inflate: members i = comp[member_off[i] .. member_off[i+1]) for i < n (member_off int64 [n+1], offsets into comp;
 * comp_bytes <= max_in_bytes; each must have a BGZF header with FLG 4 and ISIZE <= 65536, and their ISIZEs must sum to at most
 * max_out_bytes: SNPM_E_ARG otherwise) go up in one copy; k_bgzf_inflate decodes each member's DEFLATE stream with one warp
 * into its place (the exclusive sum of the ISIZEs) and checks its length and CRC-32 against the trailer; the text comes back in
 * one copy.  info int64[3] = bytes of text, the index of the first refused member or -1, and its reason (1 invalid DEFLATE
 * stream, 2 length other than ISIZE, 3 CRC-32 mismatch).  The text goes to out (info[0] bytes) unless out is NULL; either way
 * it stays in the pinned staging that snpm_bgzf_text returns until the next call.  Nothing is copied back when a member is
 * refused.  ms (optional) float[3] = device time of the copy up, of the kernel alone, of the copy down of the text (the
 * per-member status copy in between is in none of the three). */
#define SNPM_BGZF_MAX_BYTES (int64_t(1) << 31)
typedef struct snpm_bgzf snpm_bgzf;
int snpm_bgzf_scan(const uint8_t *data, int64_t n_bytes, int64_t *member_off, int32_t *isize, int64_t cap, int64_t *n_members);
int snpm_bgzf_create(int device, int64_t max_in_bytes, int64_t max_out_bytes, snpm_bgzf **out);
int snpm_bgzf_inflate(snpm_bgzf *h, const uint8_t *comp, int64_t comp_bytes, const int64_t *member_off, int64_t n, uint8_t *out,
                      int64_t *info, float *ms);
const uint8_t *snpm_bgzf_text(snpm_bgzf *h);
void snpm_bgzf_destroy(snpm_bgzf *h);

#ifdef __cplusplus
}
#endif
#endif /* SNPMATCH_B200_H */
