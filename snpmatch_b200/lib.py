"""
ctypes binding of libsnpmatch_b200.so (include/snpmatch_b200.h).

The shared library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is no
CPU fallback: if the library is missing, or no CUDA device is present when a database is created,
the call raises.
"""
import ctypes as C
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SNPM_LIB_PATH") or os.path.join(_HERE, "libsnpmatch_b200.so")      # the override is for A/B runs of two builds

SNPM_OK = 0
SNPM_E_ARG = -1
SNPM_E_CUDA = -2
SNPM_E_NOMEM = -3
SNPM_E_STATE = -4
SNPM_E_ASSERT = -5
SNPM_E_RANGE = -6

CHUNK_ROWS = 1000
PAIR_MAX_SAMPLES = 8192        # SNPM_PAIR_MAX_SAMPLES

JOIN_AUTO, JOIN_SEARCH, JOIN_MERGEPATH = 0, 1, 2
KERNEL_FP64, KERNEL_POPCOUNT, KERNEL_GROUPED = 0, 1, 2


def weights_are_one_hot(wei):
    """True when every weight row is one of (1,0,0), (0,1,0), (0,0,1): called genotypes, as
    ParseInputs.get_wei_from_GT produces (parsers.py:132-139) — the popcount kernel applies."""
    w = np.asarray(wei)
    if w.ndim != 2 or w.shape[1] != 3 or len(w) == 0:
        return False
    return bool(np.all((w == 0.0) | (w == 1.0)) and np.all(w.sum(axis=1) == 1.0))


def index_weights(wei):
    """Dictionary-code a weight matrix: (idx uint16 [n,3], table f64) with table[idx] == wei bit for bit, or None when it
    holds more than 65536 distinct values.  Weights derived from integer PLs (exp(-PL/10), parsers.py:147-151) and one-hot
    weights of called genotypes always qualify.  Done once per sample at parse time; it shrinks the per-run H2D copy 4x."""
    w = np.ascontiguousarray(wei, dtype=np.float64)
    table, inv = np.unique(w.view(np.uint64).ravel(), return_inverse=True)      # bit patterns: keeps -0.0 / nan payloads apart
    if len(table) > 65536:
        return None
    return inv.astype(np.uint16).reshape(w.shape), table.view(np.float64)


class GroupedSamples(object):
    """Samples prepared for the grouped kernel (snpm_group_markers): every sample's markers ordered by weight triple.
    offsets int64 [S+1]; chrom uint8 [n] (255 = not in the panel); pos int32 [n]; gid uint16 [n]; table f64 [T,3] in the
    column order of `wei`; order int64 [n] = index of each marker in the arrays it was built from."""

    def __init__(self, offsets, chrom, pos, gid, table, order, packed=None, run_gid=None, run_end=None):
        self.offsets, self.chrom, self.pos, self.gid, self.table, self.order = offsets, chrom, pos, gid, table, order
        self.n_samples = len(offsets) - 1
        self.packed = packed          # uint32 [n] = chromosome id << 27 | position when everything fits, else None
        self.run_gid, self.run_end = run_gid, run_end     # the ids run-length coded (uint16 [R], uint32 [R] exclusive ends), or None

    def pack(self):
        """Chromosome id and position of every marker in one word (6 instead of 7 bytes per marker cross PCIe; leaves `packed`
        None when an id exceeds 30 or a position 2^27 - 1), and the weight-triple ids run-length coded when that is shorter
        (markers are ordered by id inside a sample: ~4.1 bytes per marker)."""
        n = len(self.pos)
        out = np.empty(max(n, 1), np.uint32)
        rc = load().snpm_pack_markers(n, ptr(self.chrom), ptr(self.pos), ptr(out))
        self.packed = out[:n] if rc == SNPM_OK else None
        self.run_gid = self.run_end = None
        if self.packed is not None and n > 0:
            change = np.flatnonzero(self.gid[1:] != self.gid[:-1]) + 1
            if 6 * (len(change) + 1) < 2 * n:
                self.run_end = np.ascontiguousarray(np.concatenate([change, [n]]), dtype=np.uint32)
                self.run_gid = np.ascontiguousarray(self.gid[np.concatenate([[0], change])], dtype=np.uint16)
        return self

    @property
    def h2d_bytes(self):
        marker_bytes = self.packed.nbytes if self.packed is not None else self.chrom.nbytes + self.pos.nbytes
        id_bytes = self.run_gid.nbytes + self.run_end.nbytes if self.run_gid is not None else self.gid.nbytes
        return int(self.offsets.nbytes + marker_bytes + id_bytes + self.table.size // 3 * 32)


def group_markers(offsets, s_chrom_id, s_pos, wei, table_cap=65536):
    """Order the markers of every sample by their weight triple (host code of the library, run once at parse time).
    Returns a GroupedSamples, or None when the weights do not qualify (more than 65536 distinct triples, a chromosome id
    above 254, negative / non-finite weights): score such samples in position order."""
    offsets = as_c(offsets, np.int64)
    s_chrom_id = as_c(s_chrom_id, np.int32)
    s_pos = as_c(s_pos, np.int32)
    wei = as_c(wei, np.float64).reshape(-1, 3)
    n = int(offsets[-1])
    assert len(s_chrom_id) == len(s_pos) == len(wei) == n
    chrom = np.empty(max(n, 1), np.uint8)
    pos = np.empty(max(n, 1), np.int32)
    gid = np.empty(max(n, 1), np.uint16)
    order = np.empty(max(n, 1), np.int64)
    table = np.empty((int(table_cap), 3), np.float64)
    nt = C.c_int32(0)
    rc = load().snpm_group_markers(len(offsets) - 1, ptr(offsets), ptr(s_chrom_id), ptr(s_pos), ptr(wei), ptr(chrom), ptr(pos),
                                   ptr(gid), ptr(order), ptr(table), int(table_cap), C.byref(nt))
    if rc in (SNPM_E_RANGE, SNPM_E_ARG):
        return None
    check(rc)
    return GroupedSamples(offsets, chrom[:n], pos[:n], gid[:n], np.ascontiguousarray(table[:max(nt.value, 1)]), order[:n]).pack()


class CodedSamples(object):
    """Samples as a parser hands them over (parsers.py:141-157), ready for snpm_batch_upload_coded: markers in POSITION order,
    chrom_pos uint32 [n] = chromosome id << 27 | position (id 31 = not in the panel), codes uint16 [n,3] = per marker the
    index of its three weights (columns ref, het, alt as in `wei`) in wtable f64 [V].  The grouping by weight triple
    happens on the device (csrc/group_sort.cuh)."""

    def __init__(self, offsets, chrom_pos, codes, wtable, codes32=None):
        self.offsets, self.chrom_pos, self.codes, self.wtable = offsets, chrom_pos, codes, wtable
        self.n_samples = len(offsets) - 1
        self.codes32 = codes32            # uint32 [n] = ref | het << 10 | alt << 20 when the table has at most 1024 values, else None

    def pack(self):
        """The three codes of a marker in one word (8 instead of 10 bytes per marker cross PCIe) when every code fits 10 bits."""
        if len(self.wtable) <= 1024 and self.codes32 is None:
            c = self.codes.astype(np.uint32)
            self.codes32 = np.ascontiguousarray(c[:, 0] | (c[:, 1] << np.uint32(10)) | (c[:, 2] << np.uint32(20)))
        return self

    @property
    def h2d_bytes(self):
        code_bytes = self.codes32.nbytes if self.codes32 is not None else self.codes.nbytes
        return int(self.offsets.nbytes + self.chrom_pos.nbytes + code_bytes + self.wtable.nbytes)


def pack_chrom_pos(s_chrom_id, s_pos):
    """chromosome id << 27 | position (id < 0 -> 31 = not in the panel), or None when an id exceeds 30 or a position 2^27 - 1."""
    c = np.asarray(s_chrom_id)
    p = np.asarray(s_pos)
    if len(c) and (int(c.max()) > 30 or int(p.min()) < 0 or int(p.max()) >= (1 << 27)):
        return None
    cc = np.where(c < 0, 31, c).astype(np.uint32)
    return np.ascontiguousarray((cc << np.uint32(27)) | p.astype(np.uint32))


def code_markers(offsets, s_chrom_id, s_pos, wei=None, codes=None, wtable=None):
    """CodedSamples from position-order markers and either f64 weights [n,3] (dictionary-coded here with index_weights: done
    once per sample at parse time) or ready-made codes + table (a VCF parser's integer PLs).  None when the samples do not
    qualify (more than 65536 distinct weight values, negative / non-finite weights, ids or positions that do not fit one
    word): score such samples in position order with the fp64 kernel."""
    offsets = as_c(offsets, np.int64)
    if codes is not None and wtable is not None and len(wtable) <= 1024:
        # ready-made codes of a small table (a VCF's integer PLs): both upload words in one native pass over the markers
        wtable = as_c(wtable, np.float64)
        if len(wtable) == 0:
            wtable = np.zeros(1)
        if not (np.all(np.isfinite(wtable)) and np.all(wtable >= 0.0)):
            return None
        cid, pp = as_c(s_chrom_id, np.int32), as_c(s_pos, np.int32)
        codes = as_c(codes, np.uint16).reshape(-1, 3)
        n = int(offsets[-1])
        assert len(codes) == len(cid) == len(pp) == n
        if n and int(codes.max()) >= len(wtable):
            return None
        cp, c32 = np.empty(n, np.uint32), np.empty(n, np.uint32)
        rc = load().snpm_pack_coded(n, ptr(cid), ptr(pp), ptr(codes), ptr(cp), ptr(c32))
        if rc == SNPM_E_RANGE:
            return None
        check(rc)
        return CodedSamples(offsets, cp, codes, wtable, codes32=c32)
    cp = pack_chrom_pos(s_chrom_id, s_pos)
    if cp is None:
        return None
    if codes is None:
        iw = index_weights(as_c(wei, np.float64).reshape(-1, 3))
        if iw is None:
            return None
        codes, wtable = iw
    wtable = as_c(wtable, np.float64)
    if len(wtable) == 0:
        wtable = np.zeros(1)
    if not (np.all(np.isfinite(wtable)) and np.all(wtable >= 0.0)):
        return None
    codes = as_c(codes, np.uint16).reshape(-1, 3)
    assert len(codes) == len(cp) == int(offsets[-1])
    return CodedSamples(offsets, cp, codes, wtable).pack()


class SnpmError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "libsnpmatch_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None

_p = C.c_void_p
_i32 = C.c_int32
_i64 = C.c_int64
_f64 = C.c_double

# name -> (restype, argtypes); every symbol include/snpmatch_b200.h declares
SIGNATURES = {
    "snpm_version": (C.c_int, []),
    "snpm_last_error": (C.c_char_p, []),
    "snpm_device_count": (C.c_int, []),
    "snpm_device_info": (C.c_int, [C.c_int, C.c_char_p, C.c_int, _p, _p, _p]),
    "snpm_db_create": (C.c_int, [C.c_int, _i64, _i32, _p, _p, _i32, _i64, _p]),
    "snpm_db_destroy": (C.c_int, [_p]),
    "snpm_db_load_int8": (C.c_int, [_p, _i64, _i64, _p]),
    "snpm_db_load_packed": (C.c_int, [_p, _i64, _i64, _p]),
    "snpm_db_fill_synthetic": (C.c_int, [_p, C.c_uint64]),
    "snpm_db_read_rows_int8": (C.c_int, [_p, _p, _i64, _p]),
    "snpm_db_read_packed": (C.c_int, [_p, _i64, _i64, _p]),
    "snpm_db_segregating_rows": (C.c_int, [_p, _p, _i32, _p]),
    "snpm_db_read_columns": (C.c_int, [_p, _p, _i32, _p]),
    "snpm_pair_match_counts": (C.c_int, [C.c_int, _p, _p, _i64, _p, _p, _i64, _p, _i64, _i32, _p, _p]),
    "snpm_pair_matrix": (C.c_int, [C.c_int, _i64, _p, _p, _p, _i32, _i64, _p, _i32, _i64, _p, _p, _p]),
    "snpm_db_acc_pairs": (C.c_int, [_p, _p, _i32, C.c_int, _i64, _i32, _p, _p, _p]),
    "snpm_cross_window_genotypes": (C.c_int, [C.c_int, _p, _p, _i64, _p, _i32, _p, _p, _i64, _p, _i64, _i32, _f64, _i32, _p, _p, _p]),
    "snpm_db_n_rows": (_i64, [_p]),
    "snpm_db_n_acc": (_i32, [_p]),
    "snpm_db_row_words": (_i32, [_p]),
    "snpm_db_packed_bytes": (_i64, [_p]),
    "snpm_db_set_stream": (C.c_int, [_p, _p]),
    "snpm_intersect": (C.c_int, [_p, _p, _p, _i64, C.c_int, _p, _p, _p]),
    "snpm_match_gts_accs": (C.c_int, [C.c_int, _p, _p, _i64, _i32, C.c_int, _p, _p]),
    "snpm_calculate_likelihoods": (C.c_int, [C.c_int, _p, _p, _i64, C.c_int, _f64, _p, _p, _p]),
    "snpm_calculate_likelihoods_many": (C.c_int, [C.c_int, _p, _p, _i64, _i64, C.c_int, _f64, _p, _p, _p]),
    "snpm_batch_create": (C.c_int, [_p, _i64, _p, _p, _p, _p, _p]),
    "snpm_batch_upload": (C.c_int, [_p, _i64, _p, _p, _p, _p]),
    "snpm_batch_upload_indexed": (C.c_int, [_p, _i64, _p, _p, _p, _p, _p, _i32]),
    "snpm_batch_destroy": (C.c_int, [_p]),
    "snpm_group_markers": (C.c_int, [_i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i32, _p]),
    "snpm_batch_upload_grouped": (C.c_int, [_p, _i64, _p, _p, _p, _p, _p, _i32]),
    "snpm_pack_markers": (C.c_int, [_i64, _p, _p, _p]),
    "snpm_pack_coded": (C.c_int, [_i64, _p, _p, _p, _p, _p]),
    "snpm_batch_upload_grouped_runs": (C.c_int, [_p, _i64, _p, _p, _p, _p, _i64, _p, _i32]),
    "snpm_batch_upload_grouped_packed": (C.c_int, [_p, _i64, _p, _p, _p, _p, _i32]),
    "snpm_batch_upload_coded": (C.c_int, [_p, _i64, _p, _p, _p, _p, _i32]),
    "snpm_batch_upload_coded32": (C.c_int, [_p, _i64, _p, _p, _p, _p, _i32]),
    "snpm_batch_coded_timings": (C.c_int, [_p, _p, C.c_int]),
    "snpm_batch_guard_counts": (C.c_int, [_p, _p]),
    "snpm_batch_set_group_chunk": (C.c_int, [_p, _i32]),
    "snpm_batch_set_chunk_rows": (C.c_int, [_p, _i32]),
    "snpm_batch_set_track_pairs": (C.c_int, [_p, C.c_int]),
    "snpm_batch_set_result_range": (C.c_int, [_p, _i64, _i64]),
    "snpm_batch_set_row_filter": (C.c_int, [_p, _p, _i64]),
    "snpm_batch_set_segregation_filter": (C.c_int, [_p, _p, _i64, _i32]),
    "snpm_batch_count_flagged_pairs": (C.c_int, [_p, _p, _p]),
    "snpm_batch_run": (C.c_int, [_p, C.c_int, C.c_int]),
    "snpm_batch_epilogue": (C.c_int, [_p]),
    "snpm_batch_wait": (C.c_int, [_p, _p]),
    "snpm_batch_reduce_buffer": (C.c_int, [_p, _p, _p]),
    "snpm_batch_ipc_export": (C.c_int, [_p, _p, _p]),
    "snpm_batch_ipc_open": (C.c_int, [_p, _p, _i32, _i32]),
    "snpm_batch_reduce_peers": (C.c_int, [_p]),
    "snpm_batch_ipc_close": (C.c_int, [_p]),
    "snpm_batch_fetch": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p]),
    "snpm_batch_fetch_async": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "snpm_batch_fetch_wait": (C.c_int, [_p]),
    "snpm_batch_fetch_pairs": (C.c_int, [_p, _i64, _p, _p, _i64, _p]),
    "snpm_batch_timings": (C.c_int, [_p, _p, C.c_int]),
    "snpm_score": (C.c_int, [_p, _p, _p, _p, _i64, C.c_int, _p, _i64, _p, _p, _p, _p, _p, _p, _p]),
    "snpm_batch_run_windows": (C.c_int, [_p, C.c_int, _i64, _p, _p, _i32, _p, _i64, _f64]),
    "snpm_batch_run_windows_begin": (C.c_int, [_p, C.c_int, _i64, _p, _p, _i32, _p, _i64, _f64, _p, _p]),
    "snpm_batch_run_windows_finish": (C.c_int, [_p]),
    "snpm_batch_fetch_windows": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p]),
    "snpm_batch_fetch_window_rows": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _p, _i64, _p]),
    "snpm_batch_f1_pairs": (C.c_int, [_p, _p, _i32, _p, _p]),
    "snpm_score_shared_panel": (C.c_int, [_p, _p, _i64, _p, _i64, C.c_int, _p, _p, _p, _p, _p, _p]),
    "snpm_panel_create": (C.c_int, [_p, _p, _i64, C.c_int, _p]),
    "snpm_panel_score": (C.c_int, [_p, _p, C.c_int, _i64, _p, _p, _p, _p, _p, _p]),
    "snpm_panel_destroy": (None, [_p]),
    "snpm_vcf_create": (C.c_int, [C.c_int, _i32, _i64, _p]),
    "snpm_vcf_parse": (C.c_int, [_p, C.c_char_p, _i64, _p, _p]),
    "snpm_vcf_fetch": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "snpm_vcf_parse_gt_packed": (C.c_int, [_p, C.c_char_p, _i64, _p, _p]),
    "snpm_vcf_fetch_gt_packed": (C.c_int, [_p, _p, _p, _p, _p, _p, _p]),
    "snpm_vcf_parse_gt_codes": (C.c_int, [_p, C.c_char_p, _i64, _p, _p]),
    "snpm_vcf_fetch_gt_codes": (C.c_int, [_p, _p, _p, _p, _p, _p, _p]),
    "snpm_vcf_destroy": (None, [_p]),
    "snpm_bgzf_scan": (C.c_int, [_p, _i64, _p, _p, _i64, _p]),
    "snpm_bgzf_create": (C.c_int, [C.c_int, _i64, _i64, _p]),
    "snpm_bgzf_inflate": (C.c_int, [_p, _p, _i64, _p, _i64, _p, _p, _p]),
    "snpm_bgzf_text": (_p, [_p]),
    "snpm_bgzf_destroy": (None, [_p]),
}


def load():
    """Load the shared library (once); raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError("%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a); snpmatch_b200 has no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != SNPM_OK:
        msg = load().snpm_last_error()
        msg = msg.decode("utf-8", "replace") if msg else ""
        if rc == SNPM_E_ASSERT:
            raise AssertionError(msg)
        raise SnpmError(rc, msg)


def ptr(a):
    """Pointer to a C-contiguous NumPy buffer (None -> NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def as_c(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def device_count():
    return load().snpm_device_count()


def device_info(device=0):
    name = C.create_string_buffer(256)
    sm, mem, n_sm = C.c_int(0), C.c_int64(0), C.c_int(0)
    check(load().snpm_device_info(device, name, 256, C.byref(sm), C.byref(mem), C.byref(n_sm)))
    return {"name": name.value.decode(), "sm": sm.value, "mem_bytes": mem.value, "n_sm": n_sm.value}


class Database(object):
    """HBM-resident 2-bit packed panel (A0).  One per GPU (or per SNP-row shard)."""

    def __init__(self, positions, chr_regions, n_acc, device=0, row0_global=0):
        lib = load()
        self.positions = as_c(positions, np.int32)
        self.chr_regions = as_c(chr_regions, np.int64).reshape(-1, 2)
        self.n_rows = int(len(self.positions))
        self.n_acc = int(n_acc)
        self.device = int(device)
        self.row0_global = int(row0_global)
        h = C.c_void_p()
        check(lib.snpm_db_create(self.device, self.n_rows, self.n_acc, ptr(self.positions), ptr(self.chr_regions),
                                 len(self.chr_regions), self.row0_global, C.byref(h)))
        self._h = h
        self._batches = weakref.WeakSet()          # closed before the database: a batch handle points into it
        self.row_words = lib.snpm_db_row_words(h)
        self.packed_bytes = lib.snpm_db_packed_bytes(h)

    def close(self):
        b = getattr(self, "_scratch", None)
        if b is not None:
            b._scratch = False
            b.close()
            self._scratch = None
        for b in list(getattr(self, "_batches", ())):
            b._scratch = False
            b.close()
        if getattr(self, "_h", None):
            load().snpm_db_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_int8(self, snps, row0=0):
        snps = as_c(snps, np.int8)
        assert snps.ndim == 2 and snps.shape[1] == self.n_acc
        check(load().snpm_db_load_int8(self._h, row0, snps.shape[0], ptr(snps)))

    def load_packed(self, packed, row0=0):
        packed = as_c(packed, np.uint64)
        assert packed.ndim == 2 and packed.shape[1] == self.row_words
        check(load().snpm_db_load_packed(self._h, row0, packed.shape[0], ptr(packed)))

    def fill_synthetic(self, seed):
        check(load().snpm_db_fill_synthetic(self._h, int(seed)))

    def read_rows(self, rows):
        rows = as_c(rows, np.int64).ravel()
        out = np.empty((len(rows), self.n_acc), dtype=np.int8)
        check(load().snpm_db_read_rows_int8(self._h, ptr(rows), len(rows), ptr(out)))
        return out

    def read_packed(self, row0, n):
        out = np.empty((n, self.row_words), dtype=np.uint64)
        check(load().snpm_db_read_packed(self._h, row0, n, ptr(out)))
        return out

    def read_columns(self, acc_idx):
        """Whole accession columns, int8 [len(acc_idx), n_rows] = g_acc.snps[:, acc_idx].T (simulate.py:15, genotype_cross.py:97-98)."""
        acc_idx = as_c(np.atleast_1d(acc_idx), np.int32)
        out = np.empty((len(acc_idx), self.n_rows), dtype=np.int8)
        check(load().snpm_db_read_columns(self._h, ptr(acc_idx), len(acc_idx), ptr(out)))
        return out

    def segregating_rows(self, acc_idx):
        """Local row indices on which the given accessions carry >= 2 different called genotypes (full-panel scan on the GPU)."""
        acc_idx = as_c(acc_idx, np.int32)
        flags = np.empty(max(self.n_rows, 1), dtype=np.uint8)
        check(load().snpm_db_segregating_rows(self._h, ptr(acc_idx), len(acc_idx), ptr(flags)))
        return np.flatnonzero(flags[:self.n_rows])

    def acc_pairs(self, acc_idx=None, skip_db_hets=False, chunk_rows=0, block_acc=0):
        """Every pair of the accessions acc_idx (default: all, in panel order) over the rows this handle holds
        (snpm_db_acc_pairs): returns (common int32 [n,n], same int32 [n,n], (expand_ms, gemm_ms, device_ms)).  common[i, j] =
        rows both accessions have called, same[i, j] = those with equal calls; skip_db_hets counts hets as missing.
        chunk_rows / block_acc: rows per operand chunk and accessions per output block (0 = the library's defaults)."""
        acc_idx = np.arange(self.n_acc, dtype=np.int32) if acc_idx is None else as_c(np.atleast_1d(acc_idx), np.int32)
        n = len(acc_idx)
        common, same = np.empty((n, n), np.int32), np.empty((n, n), np.int32)
        ms = (C.c_float * 3)()
        check(load().snpm_db_acc_pairs(self._h, ptr(acc_idx), n, int(bool(skip_db_hets)), int(chunk_rows), int(block_acc),
                                       ptr(common), ptr(same), ms))
        return common, same, (ms[0], ms[1], ms[2])

    def score_shared_panel(self, panel_rows, codes, skip_db_hets=False, likelihoods=True):
        """Batched tensor-core scoring (A9): codes uint8 [S,K] (0 ref, 1 alt, 2 het, 3 absent) of S called-genotype samples on
        the K shared markers `panel_rows` (global rows).  Returns dict(matches, ninfo[, prob, L, LR], gemm_ms)."""
        panel_rows = as_c(panel_rows, np.int64)
        codes = as_c(codes, np.uint8)
        S, K = codes.shape
        assert K == len(panel_rows)
        r = {"matches": np.empty((S, self.n_acc), np.int64), "ninfo": np.empty((S, self.n_acc), np.int64)}
        if likelihoods:
            for k in ("prob", "L", "LR"):
                r[k] = np.empty((S, self.n_acc), np.float64)
        ms = C.c_float(0)
        check(load().snpm_score_shared_panel(self._h, ptr(panel_rows), K, ptr(codes), S, int(bool(skip_db_hets)), ptr(r["matches"]),
                                             ptr(r["ninfo"]), ptr(r.get("prob")), ptr(r.get("L")), ptr(r.get("LR")), C.byref(ms)))
        r["gemm_ms"] = ms.value
        return r

    def shared_panel(self, panel_rows, skip_db_hets=False):
        """SharedPanel on the markers `panel_rows` (global rows): score batch after batch against it."""
        return SharedPanel(self, panel_rows, skip_db_hets)

    def set_stream(self, cuda_stream):
        check(load().snpm_db_set_stream(self._h, C.c_void_p(cuda_stream) if cuda_stream else None))

    def scratch_batch(self, offsets, s_chrom_id, s_pos, wei, chunk_rows=CHUNK_ROWS):
        """A Batch that lives with the database: the first call creates it, later calls re-upload into the same device
        buffers (creating a batch costs a few ms of cudaMalloc / stream / event setup).  Do not close it.
        chunk_rows: Genotyper's chunk_size (the order-exact kernel sums in chunks of that many rows)."""
        b = getattr(self, "_scratch", None)
        if b is None or b._h is None:
            b = Batch(self, offsets, s_chrom_id, s_pos, wei)
            b._scratch = True
            b._chunk_rows = CHUNK_ROWS
            self._scratch = b
            if chunk_rows == CHUNK_ROWS:
                return b
        b.set_row_filter(None)
        if getattr(b, "_chunk_rows", CHUNK_ROWS) != chunk_rows:
            b.set_chunk_rows(chunk_rows)
            b._chunk_rows = chunk_rows
        b.upload(offsets, s_chrom_id, s_pos, wei)
        return b

    def intersect(self, s_chrom_id, s_pos, algo=JOIN_AUTO):
        s_chrom_id = as_c(s_chrom_id, np.int32)
        s_pos = as_c(s_pos, np.int32)
        n = len(s_pos)
        db_idx = np.empty(max(n, 1), dtype=np.int64)
        s_idx = np.empty(max(n, 1), dtype=np.int64)
        m = C.c_int64(0)
        check(load().snpm_intersect(self._h, ptr(s_chrom_id), ptr(s_pos), n, algo, ptr(db_idx), ptr(s_idx), C.byref(m)))
        return db_idx[:m.value].copy(), s_idx[:m.value].copy()


def pack_codes2(codes):
    """uint8 codes [S,K] (0 ref, 1 alt, 2 het, 3 or more absent, as in the unpacked form) -> 2-bit packed rows uint8
    [S, ceil(K/4)] (marker k in bits 2(k&3) of byte k >> 2; the spare bits of the last byte read as absent)."""
    codes = np.asarray(codes, dtype=np.uint8)
    S, K = codes.shape
    pad = (-K) % 4
    if pad:
        codes = np.concatenate([codes, np.full((S, pad), 3, np.uint8)], axis=1)
    c = np.minimum(codes, 3).reshape(S, -1, 4)
    return np.ascontiguousarray(c[:, :, 0] | (c[:, :, 1] << 2) | (c[:, :, 2] << 4) | (c[:, :, 3] << 6))


class SharedPanel(object):
    """A9 as an object: the panel-side tensor-core operand of K shared markers is expanded once, every score() call re-uses it
    and the panel's device scratch (snpm_panel_*)."""

    def __init__(self, db, panel_rows, skip_db_hets=False):
        self.db = db
        self.panel_rows = as_c(panel_rows, np.int64)
        self.K = int(len(self.panel_rows))
        h = C.c_void_p()
        check(load().snpm_panel_create(db._h, ptr(self.panel_rows), self.K, int(bool(skip_db_hets)), C.byref(h)))
        self._h = h
        db._batches.add(self)                      # closed before the database

    def score(self, codes, packed=False, likelihoods=False, out=None):
        """codes: uint8 [S,K], or with packed=True the 2-bit rows of pack_codes2 ([S, ceil(K/4)]).  out: optional dict of
        preallocated (page-locked) arrays matches/ninfo int32 [S,A] (and prob/L/LR f64 when likelihoods).
        Returns dict(matches, ninfo[, prob, L, LR], expand_ms, gemm_ms, device_ms)."""
        codes = as_c(codes, np.uint8)
        S = int(codes.shape[0])
        assert codes.ndim == 2 and codes.shape[1] == ((self.K + 3) // 4 if packed else self.K)
        A = self.db.n_acc
        r = dict(out) if out is not None else {}
        for k in ("matches", "ninfo"):
            if k not in r:
                r[k] = np.empty((S, A), np.int32)
            assert r[k].dtype == np.int32 and r[k].shape == (S, A) and r[k].flags.c_contiguous
        if likelihoods:
            for k in ("prob", "L", "LR"):
                if k not in r:
                    r[k] = np.empty((S, A), np.float64)
                assert r[k].dtype == np.float64 and r[k].shape == (S, A) and r[k].flags.c_contiguous
        ms = (C.c_float * 3)()
        check(load().snpm_panel_score(self._h, ptr(codes), int(bool(packed)), S, ptr(r["matches"]), ptr(r["ninfo"]),
                                      ptr(r.get("prob")) if likelihoods else None, ptr(r.get("L")) if likelihoods else None,
                                      ptr(r.get("LR")) if likelihoods else None, ms))
        r["expand_ms"], r["gemm_ms"], r["device_ms"] = ms[0], ms[1], ms[2]
        return r

    _scratch = False

    def close(self):
        if getattr(self, "_h", None):
            load().snpm_panel_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class VcfParser(object):
    """The genotype columns of a multi-sample VCF parsed on the device (snpm_vcf_*), one chunk of whole lines at a time.
    parse(text) returns the chunk's per-line arrays and every sample's called cells (see snpm_vcf_fetch); core.parsers.read_vcf_many
    turns them into one ParseInputs per sample.  parse_gt_packed(text) returns the chunk's records as rows of the packed panel
    (snpm_vcf_fetch_gt_packed), which core.makedb.makeDB_from_vcf assembles.  parse_gt_codes(text) returns them as rows of int8
    window-call codes (snpm_vcf_fetch_gt_codes), which core.parsers.read_vcf_gt_codes assembles."""

    FLAG_RECORD, FLAG_FALLBACK, FLAG_HAS_PL, FLAG_NEW_CHROM = 1, 2, 4, 8
    N_ALLELE_CODES = 111

    def __init__(self, device, n_samples, chunk_bytes):
        self.device, self.n_samples, self.chunk_bytes = int(device), int(n_samples), int(chunk_bytes)
        h = C.c_void_p()
        check(load().snpm_vcf_create(self.device, self.n_samples, self.chunk_bytes, C.byref(h)))
        self._h = h

    def parse(self, text):
        """text: bytes of whole lines, ending in a line end.  Returns dict(n_lines, n_cells, non_ascii, info_dp_lines, h2d_ms,
        kernel_ms, and the arrays line_start, flags, nsf, pos, dp, chrom_len, sample_off, line, cls, pl)."""
        info = np.zeros(5, np.int64)
        ms = (C.c_float * 2)()
        check(load().snpm_vcf_parse(self._h, text, len(text), ptr(info), ms))
        n, k, S = int(info[0]), int(info[2]), self.n_samples
        r = dict(n_lines=n, n_cells=int(info[1]), non_ascii=bool(info[3]), info_dp_lines=int(info[4]), h2d_ms=ms[0], kernel_ms=ms[1],
                 line_start=np.empty(n + 1, np.int32), sample_off=np.empty(S + 1, np.int32), line=np.empty(k, np.int32),
                 cls=np.empty(k, np.uint16), pl=np.empty((k, 3), np.int32))
        for key in ("flags", "nsf", "pos", "dp", "chrom_len"):
            r[key] = np.empty(n, np.int32)
        check(load().snpm_vcf_fetch(self._h, *[ptr(r[key]) for key in ("line_start", "flags", "nsf", "pos", "dp", "chrom_len",
                                                                       "sample_off", "line", "cls", "pl")]))
        return r

    def parse_gt_packed(self, text):
        """`makedb --no_csv`: text as for parse(), read with makedb's rules (snpm_vcf_parse_gt_packed).  Returns dict(n_lines,
        n_rows, other_calls, non_ascii, h2d_ms, kernel_ms, and the arrays line_start, flags, nsf, pos, chrom_len and packed uint64
        [n_rows, row_words]: the panel rows of the records with n_samples sample fields, in line order)."""
        info = np.zeros(4, np.int64)
        ms = (C.c_float * 2)()
        check(load().snpm_vcf_parse_gt_packed(self._h, text, len(text), ptr(info), ms))
        n, rows = int(info[0]), int(info[1])
        r = dict(n_lines=n, n_rows=rows, other_calls=int(info[2]), non_ascii=bool(info[3]), h2d_ms=ms[0], kernel_ms=ms[1],
                 line_start=np.empty(n + 1, np.int32), packed=np.empty((rows, self.row_words), np.uint64))
        for key in ("flags", "nsf", "pos", "chrom_len"):
            r[key] = np.empty(n, np.int32)
        check(load().snpm_vcf_fetch_gt_packed(self._h, *[ptr(r[key]) for key in ("line_start", "flags", "nsf", "pos", "chrom_len",
                                                                                 "packed")]))
        return r

    def parse_gt_codes(self, text):
        """`genotype_cross --gpu_parse`: text as for parse(), every record read into a row of the codes parseGT gives the GT
        strings of read_vcf_samples (snpm_vcf_parse_gt_codes).  Returns dict(n_lines, n_rows, non_ascii, h2d_ms, kernel_ms, and
        the arrays line_start, flags, nsf, pos, chrom_len and codes int8 [n_rows, n_samples]: one row per record, in line order)."""
        info = np.zeros(3, np.int64)
        ms = (C.c_float * 2)()
        check(load().snpm_vcf_parse_gt_codes(self._h, text, len(text), ptr(info), ms))
        n, rows = int(info[0]), int(info[1])
        r = dict(n_lines=n, n_rows=rows, non_ascii=bool(info[2]), h2d_ms=ms[0], kernel_ms=ms[1],
                 line_start=np.empty(n + 1, np.int32), codes=np.empty((rows, self.n_samples), np.int8))
        for key in ("flags", "nsf", "pos", "chrom_len"):
            r[key] = np.empty(n, np.int32)
        check(load().snpm_vcf_fetch_gt_codes(self._h, *[ptr(r[key]) for key in ("line_start", "flags", "nsf", "pos", "chrom_len",
                                                                                "codes")]))
        return r

    @property
    def row_words(self):
        """Words per packed row: snpm_db_row_words of a panel of n_samples accessions."""
        return (((self.n_samples + 31) // 32) + 1) & ~1

    def close(self):
        if getattr(self, "_h", None):
            load().snpm_vcf_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bgzf_scan(data):
    """Member table of a BGZF file held in data (a buffer of uint8, e.g. an mmap viewed by NumPy): (member_off int64 [n+1],
    isize int64 [n]) when the file is all BGZF (snpm_bgzf_scan: every member a BGZF member with ISIZE <= 65536, the members
    tiling the data to its last byte), else None.  Host code; needs no device."""
    data = np.frombuffer(data, np.uint8) if not isinstance(data, np.ndarray) else data
    n_bytes = len(data)
    cap = n_bytes // 8192 + 16
    while True:
        off, isize, n = np.empty(cap + 1, np.int64), np.empty(cap, np.int32), C.c_int64(0)
        check(load().snpm_bgzf_scan(ptr(data) if n_bytes else None, n_bytes, ptr(off), ptr(isize), cap, C.byref(n)))
        if n.value < 0:
            return None
        if n.value <= cap:
            return off[:n.value + 1], isize[:n.value].astype(np.int64)
        cap = n.value


class BgzfInflater(object):
    """BGZF members inflated on CUDA device `device` (snpm_bgzf_*): up to max_in_bytes of members and max_out_bytes of text
    per call.  inflate() raises gzip.BadGzipFile naming the path, the refused member's byte offset in the file and the reason."""

    REASONS = {1: "invalid DEFLATE stream", 2: "text length differs from ISIZE", 3: "CRC-32 mismatch"}

    def __init__(self, device, max_in_bytes, max_out_bytes):
        self.max_in_bytes, self.max_out_bytes = int(max_in_bytes), int(max_out_bytes)
        h = C.c_void_p()
        check(load().snpm_bgzf_create(int(device), self.max_in_bytes, self.max_out_bytes, C.byref(h)))
        self._h = h
        self.ms = np.zeros(3)                   # device ms summed over the calls: copy up, kernel, copy down

    def inflate(self, comp, member_off, path="<bytes>", base=0, out=None):
        """comp: uint8 array holding the members, member_off int64 [n+1] their offsets in it; base = the byte offset of
        comp[0] in the file (for the error).  Returns the number of bytes of text.  The text goes to out (uint8 array) when
        given; it stays in the handle's pinned staging (text()) until the next call either way."""
        member_off = as_c(member_off, np.int64)
        info = np.zeros(3, np.int64)
        ms = (C.c_float * 3)()
        check(load().snpm_bgzf_inflate(self._h, ptr(comp), len(comp), ptr(member_off), len(member_off) - 1, ptr(out), ptr(info), ms))
        self.ms += np.array(ms[:3])
        if info[1] >= 0:
            import gzip
            raise gzip.BadGzipFile("%s: BGZF member at byte %d: %s" % (path, base + int(member_off[info[1]]),
                                                                       self.REASONS.get(int(info[2]), "reason %d" % info[2])))
        return int(info[0])

    def text(self, start, stop):
        """bytes start..stop of the last call's text, copied once out of the pinned staging."""
        return C.string_at(load().snpm_bgzf_text(self._h) + start, stop - start)

    def close(self):
        if getattr(self, "_h", None):
            load().snpm_bgzf_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Batch(object):
    """One or more samples resident on the device next to a Database, plus their results."""

    def __init__(self, db, offsets, s_chrom_id, s_pos, wei):
        self.db = db
        self._h = None
        args = self._prep(offsets, s_chrom_id, s_pos, wei)
        h = C.c_void_p()
        check(load().snpm_batch_create(db._h, self.n_samples, *[ptr(a) for a in args], C.byref(h)))
        self._h = h
        db._batches.add(self)

    def _prep(self, offsets, s_chrom_id, s_pos, wei):
        offsets = as_c(offsets, np.int64)
        s_chrom_id = as_c(s_chrom_id, np.int32)
        s_pos = as_c(s_pos, np.int32)
        wei = as_c(wei, np.float64).reshape(-1, 3)
        assert len(s_chrom_id) == len(s_pos) == len(wei) == int(offsets[-1])
        self.n_samples = len(offsets) - 1
        self.offsets = offsets
        self._keep = (offsets, s_chrom_id, s_pos, wei)
        return self._keep

    def upload(self, offsets, s_chrom_id, s_pos, wei):
        """Replace the batch's samples, reusing its device buffers (queued on the stream)."""
        args = self._prep(offsets, s_chrom_id, s_pos, wei)
        check(load().snpm_batch_upload(self._h, self.n_samples, *[ptr(a) for a in args]))

    def upload_indexed(self, offsets, s_chrom_id, s_pos, wei_idx, table):
        """upload() with dictionary-coded weights: wei_idx uint16 [n,3] into `table` (f64).  See index_weights()."""
        offsets = as_c(offsets, np.int64)
        s_chrom_id = as_c(s_chrom_id, np.int32)
        s_pos = as_c(s_pos, np.int32)
        wei_idx = as_c(wei_idx, np.uint16).reshape(-1, 3)
        table = as_c(table, np.float64)
        assert len(s_chrom_id) == len(s_pos) == len(wei_idx) == int(offsets[-1]) and 1 <= len(table) <= 65536
        self.n_samples = len(offsets) - 1
        self.offsets = offsets
        self._keep = (offsets, s_chrom_id, s_pos, wei_idx, table)
        check(load().snpm_batch_upload_indexed(self._h, self.n_samples, ptr(offsets), ptr(s_chrom_id), ptr(s_pos), ptr(wei_idx),
                                               ptr(table), len(table)))

    def upload_grouped(self, g):
        """Replace the batch's samples by grouped ones (GroupedSamples); score them with run(kernel_mode=KERNEL_GROUPED)."""
        self.n_samples = g.n_samples
        self.offsets = g.offsets
        self._keep = (g,)
        if g.packed is not None and g.run_gid is not None:
            check(load().snpm_batch_upload_grouped_runs(self._h, g.n_samples, ptr(g.offsets), ptr(g.packed), ptr(g.run_gid), ptr(g.run_end),
                                                        len(g.run_gid), ptr(g.table), len(g.table)))
        elif g.packed is not None:
            check(load().snpm_batch_upload_grouped_packed(self._h, g.n_samples, ptr(g.offsets), ptr(g.packed), ptr(g.gid),
                                                          ptr(g.table), len(g.table)))
        else:
            check(load().snpm_batch_upload_grouped(self._h, g.n_samples, ptr(g.offsets), ptr(g.chrom), ptr(g.pos), ptr(g.gid),
                                                   ptr(g.table), len(g.table)))

    def upload_coded(self, cs):
        """Replace the batch's samples by coded ones (CodedSamples: position order + weight codes; grouped on the device);
        score them with run(kernel_mode=KERNEL_GROUPED)."""
        self.n_samples = cs.n_samples
        self.offsets = cs.offsets
        self._keep = (cs,)
        if cs.codes32 is not None:
            check(load().snpm_batch_upload_coded32(self._h, cs.n_samples, ptr(cs.offsets), ptr(cs.chrom_pos), ptr(cs.codes32), ptr(cs.wtable),
                                                   len(cs.wtable)))
        else:
            check(load().snpm_batch_upload_coded(self._h, cs.n_samples, ptr(cs.offsets), ptr(cs.chrom_pos), ptr(cs.codes), ptr(cs.wtable),
                                                 len(cs.wtable)))

    def coded_timings(self):
        """Device times (ms) of the last coded run: join (expansion, search, compaction), group (key sort + change masks),
        score (k_score_grouped2), combine."""
        ms = np.zeros(4, dtype=np.float32)
        check(load().snpm_batch_coded_timings(self._h, ptr(ms), 4))
        return {"join_ms": float(ms[0]), "group_ms": float(ms[1]), "score_ms": float(ms[2]), "combine_ms": float(ms[3])}

    def set_result_range(self, first_sample=0, n_samples=-1):
        """Epilogue, fetches and guard counts work on samples [first_sample, first_sample + n_samples) only (-1: all)."""
        check(load().snpm_batch_set_result_range(self._h, int(first_sample), int(n_samples)))
        self._res = (int(first_sample), int(n_samples))

    def _n_results(self):
        r = getattr(self, "_res", (0, -1))
        return self.n_samples if r[1] < 0 else r[1]

    def set_chunk_rows(self, rows):
        """Genotyper chunk_size (snpmatch.py:173): rows per chunk of the order-exact kernel; applies from the next upload()."""
        check(load().snpm_batch_set_chunk_rows(self._h, int(rows)))

    def set_track_pairs(self, on):
        """Coded batches: keep the marker index of every matched pair (fetch_pairs) or not (one array less to move)."""
        check(load().snpm_batch_set_track_pairs(self._h, int(bool(on))))

    def set_group_chunk(self, rows):
        check(load().snpm_batch_set_group_chunk(self._h, int(rows)))

    def guard_counts(self):
        """Per sample: accessions whose int(score) depends on the reference's summation order (grouped batches; see
        snpm_batch_guard_counts).  Re-score those samples with the fp64 kernel."""
        out = np.zeros(self._n_results(), dtype=np.int32)
        check(load().snpm_batch_guard_counts(self._h, ptr(out)))
        return out

    def close(self):
        if getattr(self, "_scratch", False):
            return                                  # owned by the Database
        if getattr(self, "_h", None):
            load().snpm_batch_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_row_filter(self, rows):
        """rows=None clears the filter; an empty array keeps no pair at all (Genotyper.genotyper(filter_pos_ix=...) with nothing
        in it leaves no common SNP, snpmatch.py:211-216)."""
        if rows is None:
            check(load().snpm_batch_set_row_filter(self._h, None, 0))
            return
        rows = as_c(np.unique(np.asarray(rows, dtype=np.int64)), np.int64)
        self._filter_keep = rows if len(rows) else np.zeros(1, np.int64)      # a valid pointer for the empty list
        check(load().snpm_batch_set_row_filter(self._h, ptr(self._filter_keep), len(rows)))

    def set_segregation_filter(self, sel):
        """Per-sample `--refine` filter: sel uint32 [S, row_words] accession bit masks (selection_masks()), one row per sample of
        the next run; a sample keeps only the pairs whose row segregates among its selected accessions.  None clears it."""
        if sel is None:
            check(load().snpm_batch_set_segregation_filter(self._h, None, 0, 0))
            return
        sel = as_c(sel, np.uint32)
        assert sel.ndim == 2
        check(load().snpm_batch_set_segregation_filter(self._h, ptr(sel), sel.shape[0], sel.shape[1]))

    def count_flagged_pairs(self, flags):
        """After run(): per sample, the kept pairs whose marker is flagged (flags: one per uploaded marker, upload order)."""
        flags = as_c(np.asarray(flags, dtype=bool).view(np.uint8), np.uint8)
        assert len(flags) == int(self.offsets[-1])
        counts = np.zeros(self.n_samples, dtype=np.int64)
        check(load().snpm_batch_count_flagged_pairs(self._h, ptr(flags) if len(flags) else None, ptr(counts)))
        return counts

    def run(self, skip_db_hets=False, kernel_mode=0, join_algo=JOIN_AUTO):
        check(load().snpm_batch_run(self._h, int(bool(skip_db_hets)), int(kernel_mode) | (int(join_algo) << 8)))

    def epilogue(self):
        check(load().snpm_batch_epilogue(self._h))

    def wait(self):
        ms = C.c_float(0)
        check(load().snpm_batch_wait(self._h, C.byref(ms)))
        return ms.value

    def timings(self):
        ms = np.zeros(8, dtype=np.float32)
        check(load().snpm_batch_timings(self._h, ptr(ms), 8))
        t = {"join_ms": float(ms[0]), "score_ms": float(ms[1]), "combine_ms": float(ms[2]), "epilogue_ms": float(ms[3]),
             "total_ms": float(ms[4]), "launches": int(ms[5])}
        if ms[6] > 0:              # one-shot peer reduce: the kernel, and the part of it spent waiting for the slowest rank
            t["peer_reduce_ms"], t["peer_wait_ms"] = float(ms[6]), float(ms[7])
        return t

    def reduce_buffer(self):
        """(device pointer, number of f64) of the per-sample totals — the payload of the cross-GPU sum."""
        p, n = C.c_void_p(), C.c_int64(0)
        check(load().snpm_batch_reduce_buffer(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def ipc_export(self):
        """64-byte CUDA IPC handle of the reduce buffer (bytes) for the one-shot peer reduce."""
        h = C.create_string_buffer(64)
        n = C.c_int64(0)
        check(load().snpm_batch_ipc_export(self._h, h, C.byref(n)))
        return h.raw

    def ipc_open(self, handles, rank):
        """handles: list of every rank's ipc_export() bytes, in rank order."""
        blob = b"".join(handles)
        assert len(blob) == 64 * len(handles)
        check(load().snpm_batch_ipc_open(self._h, C.c_char_p(blob), len(handles), int(rank)))

    def reduce_peers(self):
        check(load().snpm_batch_reduce_peers(self._h))

    def ipc_close(self):
        check(load().snpm_batch_ipc_close(self._h))

    def fetch(self, epilogue=True, out=None):
        S, A = self._n_results(), self.db.n_acc
        r = out if out is not None else {}
        if "score" not in r:
            r["score"] = np.empty((S, A), dtype=np.float64)
            r["m"] = np.empty(S, dtype=np.int64)
            if epilogue:
                r["matches"] = np.empty((S, A), dtype=np.int64)
                r["ninfo"] = np.empty((S, A), dtype=np.int64)
                r["prob"] = np.empty((S, A), dtype=np.float64)
                r["L"] = np.empty((S, A), dtype=np.float64)
                r["LR"] = np.empty((S, A), dtype=np.float64)
        check(load().snpm_batch_fetch(self._h, ptr(r["score"]), ptr(r.get("matches")), ptr(r.get("ninfo")), ptr(r["m"]),
                                      ptr(r.get("prob")), ptr(r.get("L")), ptr(r.get("LR"))))
        return r

    def fetch_async(self, out):
        """Queue the read-back of the results into `out` (dict of PINNED arrays with the keys of fetch() plus an optional
        int32 "guard" [S]) behind the batch's kernels; fetch_wait() makes them valid.  Another batch may run in between."""
        self._pending = out
        check(load().snpm_batch_fetch_async(self._h, ptr(out.get("score")), ptr(out.get("matches")), ptr(out.get("ninfo")), ptr(out.get("m")),
                                            ptr(out.get("prob")), ptr(out.get("L")), ptr(out.get("LR")), ptr(out.get("guard"))))

    def fetch_wait(self):
        check(load().snpm_batch_fetch_wait(self._h))
        out, self._pending = self._pending, None
        return out

    def fetch_pairs(self, s=0):
        n = int(self.offsets[s + 1] - self.offsets[s])
        db_idx = np.empty(max(n, 1), dtype=np.int64)
        s_idx = np.empty(max(n, 1), dtype=np.int64)
        m = C.c_int64(0)
        check(load().snpm_batch_fetch_pairs(self._h, s, ptr(db_idx), ptr(s_idx), n, C.byref(m)))
        return db_idx[:m.value].copy(), s_idx[:m.value].copy()

    def run_windows(self, skip_db_hets, bin_len, win_count, win_off, n_windows, kmax, lr_thres=3.841):
        win_count = as_c(win_count, np.int32)
        win_off = as_c(win_off, np.int32)
        kmax = as_c(kmax, np.int32)
        self.n_windows = int(n_windows)
        check(load().snpm_batch_run_windows(self._h, int(bool(skip_db_hets)), int(bin_len), ptr(win_count), ptr(win_off),
                                            self.n_windows, ptr(kmax), len(kmax), float(lr_thres)))

    def run_windows_begin(self, skip_db_hets, bin_len, win_count, win_off, n_windows, kmax, lr_thres=3.841):
        """First half of run_windows on a SNP-row shard: returns (device pointer, number of f64) of the packed per-window
        partials (score | ninfo | rows) to be summed over the ranks in place; run_windows_finish() then completes the run."""
        win_count = as_c(win_count, np.int32)
        win_off = as_c(win_off, np.int32)
        kmax = as_c(kmax, np.int32)
        self.n_windows = int(n_windows)
        p, n = C.c_void_p(), C.c_int64(0)
        check(load().snpm_batch_run_windows_begin(self._h, int(bool(skip_db_hets)), int(bin_len), ptr(win_count), ptr(win_off),
                                                  self.n_windows, ptr(kmax), len(kmax), float(lr_thres), C.byref(p), C.byref(n)))
        return p.value, n.value

    def run_windows_finish(self):
        check(load().snpm_batch_run_windows_finish(self._h))

    def fetch_windows(self):
        """Every window's arrays: score, L, LR f64, ninfo int32, identical uint8 [W, A]; num_amb, nrows int32 [W]; matched_s_idx
        int64 (the sample's matched markers in window order).  A batch of S > 1 samples gets a leading sample axis ([S, W, A],
        [S, W]) and matched_s_idx as a list of S arrays (indices into the concatenated upload)."""
        S, W, A = self.n_samples, self.n_windows, self.db.n_acc
        SW = S * W
        n = int(self.offsets[-1])
        r = {"score": np.empty((SW, A), np.float64), "ninfo": np.empty((SW, A), np.int32), "L": np.empty((SW, A), np.float64),
             "LR": np.empty((SW, A), np.float64), "identical": np.empty((SW, A), np.uint8), "num_amb": np.empty(SW, np.int32),
             "nrows": np.empty(SW, np.int32)}
        tar = np.empty(max(n, 1), dtype=np.int64)
        m = C.c_int64(0)
        check(load().snpm_batch_fetch_windows(self._h, ptr(r["score"]), ptr(r["ninfo"]), ptr(r["L"]), ptr(r["LR"]),
                                              ptr(r["identical"]), ptr(r["num_amb"]), ptr(r["nrows"]), ptr(tar), n, C.byref(m)))
        tar = tar[:m.value].copy()
        if S == 1:
            r["matched_s_idx"] = tar
            return r
        for k in ("score", "ninfo", "L", "LR", "identical"):
            r[k] = r[k].reshape(S, W, A)
        r["num_amb"], r["nrows"] = r["num_amb"].reshape(S, W), r["nrows"].reshape(S, W)
        cut = np.concatenate([[0], np.cumsum(r["nrows"].sum(axis=1, dtype=np.int64))])
        r["matched_s_idx"] = [tar[cut[i]:cut[i + 1]] for i in range(S)]
        return r

    def fetch_window_rows(self):
        """The surviving rows of every window (csmatch.py:57-60), compacted on the device.  Returns dict(row_off int32 [W+1],
        num_amb, nrows int32 [W], acc int32 [R], score f64 [R], ninfo int32 [R], L f64 [R], identical uint8 [R],
        matched_s_idx).  A batch of S > 1 samples gets a list of S such dicts, one per sample (row_off starting at 0,
        matched_s_idx indexing the concatenated upload)."""
        S = self.n_samples
        W = S * self.n_windows
        n = int(self.offsets[-1])
        r = {"row_off": np.zeros(W + 1, np.int32), "num_amb": np.zeros(max(W, 1), np.int32), "nrows": np.zeros(max(W, 1), np.int32)}
        tar = np.empty(max(n, 1), dtype=np.int64)
        n_rows, m = C.c_int64(0), C.c_int64(0)
        lib_ = load()
        check(lib_.snpm_batch_fetch_window_rows(self._h, ptr(r["row_off"]), ptr(r["num_amb"]), ptr(r["nrows"]), None, None, None, None, None,
                                                0, C.byref(n_rows), ptr(tar), n, C.byref(m)))
        R = n_rows.value
        r.update(acc=np.empty(max(R, 1), np.int32), score=np.empty(max(R, 1), np.float64), ninfo=np.empty(max(R, 1), np.int32),
                 L=np.empty(max(R, 1), np.float64), identical=np.empty(max(R, 1), np.uint8))
        if R:
            check(lib_.snpm_batch_fetch_window_rows(self._h, None, None, None, ptr(r["acc"]), ptr(r["score"]), ptr(r["ninfo"]), ptr(r["L"]),
                                                    ptr(r["identical"]), R, C.byref(n_rows), None, 0, None))
        for k in ("acc", "score", "ninfo", "L", "identical"):
            r[k] = r[k][:R]
        r["num_amb"], r["nrows"] = r["num_amb"][:W], r["nrows"][:W]
        r["matched_s_idx"] = tar[:m.value].copy()
        if S == 1:
            return r
        Wn, out, at = self.n_windows, [], 0
        for i in range(S):
            lo, hi = i * Wn, (i + 1) * Wn
            r0, r1 = int(r["row_off"][lo]), int(r["row_off"][hi])
            nrows = r["nrows"][lo:hi]
            k = int(nrows.sum(dtype=np.int64))
            d = {"row_off": r["row_off"][lo:hi + 1] - r0, "num_amb": r["num_amb"][lo:hi], "nrows": nrows,
                 "matched_s_idx": r["matched_s_idx"][at:at + k]}
            for key in ("acc", "score", "ninfo", "L", "identical"):
                d[key] = r[key][r0:r1]
            out.append(d)
            at += k
        return out

    def f1_pairs(self, acc_idx):
        """Simulated F1 sums of the accession pairs (i < j in list order): acc_idx [k] -> (score f64, ninfo int64) [P]; on a batch
        of S samples acc_idx [S, k] (one list per sample) -> [S, P]."""
        acc_idx = as_c(acc_idx, np.int32)
        multi = acc_idx.ndim == 2
        assert (acc_idx.shape[0] == self.n_samples) if multi else self.n_samples == 1
        k = acc_idx.shape[-1]
        n_pairs = k * (k - 1) // 2
        score = np.empty((self.n_samples, n_pairs), dtype=np.float64)
        ninfo = np.empty((self.n_samples, n_pairs), dtype=np.int64)
        check(load().snpm_batch_f1_pairs(self._h, ptr(acc_idx), k, ptr(score), ptr(ninfo)))
        return (score, ninfo) if multi else (score[0], ninfo[0])


def match_gts_accs(wei, snps, skip_hets_db=False, device=0):
    wei = as_c(wei, np.float64)
    snps = as_c(snps, np.int8)
    k, n_acc = snps.shape
    score = np.empty(n_acc, dtype=np.float64)
    ninfo = np.empty(n_acc, dtype=np.int64)
    check(load().snpm_match_gts_accs(device, ptr(wei), ptr(snps), k, n_acc, int(bool(skip_hets_db)), ptr(score), ptr(ninfo)))
    return score, ninfo


def pair_match_counts(idx1, idx2, chrom1, gt1, gt2, n_chr, device=0):
    """Per-chromosome (common, matches) of pairwiseScore's counting loop (snpmatch.py:291-297) on the device."""
    idx1, idx2 = as_c(idx1, np.int64), as_c(idx2, np.int64)
    chrom1, gt1, gt2 = as_c(chrom1, np.int32), as_c(gt1, np.int32), as_c(gt2, np.int32)
    assert len(idx1) == len(idx2) and len(chrom1) == len(gt1)
    common = np.zeros(n_chr, dtype=np.int64)
    matches = np.zeros(n_chr, dtype=np.int64)
    check(load().snpm_pair_match_counts(device, ptr(idx1), ptr(idx2), len(idx1), ptr(chrom1), ptr(gt1), len(gt1), ptr(gt2), len(gt2),
                                        n_chr, ptr(common), ptr(matches)))
    return common, matches


def pair_matrix(offsets, col, cls, n_cls, K, chr_start, chunk_markers=0, device=0):
    """All-against-all counts of pairsnp on the device (snpm_pair_matrix): samples as CSR (offsets int64[S+1]; col int32 union
    column of each marker, strictly ascending inside a sample; cls uint8 GT-string class < n_cls <= 8), chr_start int64[C+1]
    column range of each chromosome.  Returns (common int32 [C,S,S], same int32 [C,S,S], (expand_ms, gemm_ms, device_ms))."""
    offsets, col, cls = as_c(offsets, np.int64), as_c(col, np.int32), as_c(cls, np.uint8)
    chr_start = as_c(chr_start, np.int64)
    S, C_ = len(offsets) - 1, len(chr_start) - 1
    assert S >= 0 and C_ >= 0 and len(col) == len(cls)
    shape = (C_, max(S, 0), max(S, 0)) if S <= PAIR_MAX_SAMPLES else (0, 0, 0)     # an S past the limit is refused by the library
    common, same = np.empty(shape, np.int32), np.empty(shape, np.int32)
    ms = (C.c_float * 3)()
    check(load().snpm_pair_matrix(device, S, ptr(offsets), ptr(col), ptr(cls), int(n_cls), int(K), ptr(chr_start), C_, int(chunk_markers),
                                  ptr(common), ptr(same), ms))
    return common, same, (ms[0], ms[1], ms[2])


def cross_window_genotypes(par_idx, vcf_idx, win_start, p1, p2, gt, lr_thres, n_marker_thres=5, device=0):
    """Window calls of genotype_cross (genotype_cross.py:210-241) on the device: returns (counts int32 [W,S,3], geno int8 [W,S]
    with -1 = NA, borderline uint8 [W,S])."""
    par_idx, vcf_idx = as_c(par_idx, np.int64), as_c(vcf_idx, np.int64)
    win_start = as_c(win_start, np.int32)
    p1, p2, gt = as_c(p1, np.int8), as_c(p2, np.int8), as_c(gt, np.int8)
    assert gt.ndim == 2 and len(p1) == len(p2) and len(par_idx) == len(vcf_idx)
    W, S = len(win_start) - 1, gt.shape[1]
    counts = np.zeros((W, S, 3), dtype=np.int32)
    geno = np.full((W, S), -1, dtype=np.int8)
    border = np.zeros((W, S), dtype=np.uint8)
    check(load().snpm_cross_window_genotypes(device, ptr(par_idx), ptr(vcf_idx), len(par_idx), ptr(win_start), W, ptr(p1), ptr(p2), len(p1),
                                             ptr(gt), gt.shape[0], S, float(lr_thres), int(n_marker_thres), ptr(counts), ptr(geno), ptr(border)))
    return counts, geno, border


def calculate_likelihoods(scores, ninfo, amin="calc", device=0):
    scores = as_c(scores, np.float64).ravel()
    ninfo = as_c(ninfo, np.float64).ravel()
    n = len(scores)
    prob = np.empty(n, dtype=np.float64)
    lik = np.empty(n, dtype=np.float64)
    lr = np.empty(n, dtype=np.float64)
    calc = amin == "calc"
    check(load().snpm_calculate_likelihoods(device, ptr(scores), ptr(ninfo), n, int(calc), 0.0 if calc else float(amin),
                                            ptr(prob), ptr(lik), ptr(lr)))
    return prob, lik, lr


def calculate_likelihoods_many(scores, ninfo, amin="calc", device=0):
    """calculate_likelihoods for every row of scores / ninfo [S, K] in one device call; pad short rows with ninfo = 0."""
    scores = as_c(scores, np.float64)
    ninfo = as_c(ninfo, np.float64)
    assert scores.ndim == 2 and scores.shape == ninfo.shape
    S, K = scores.shape
    prob, lik, lr = (np.empty((S, K), dtype=np.float64) for _ in range(3))
    calc = amin == "calc"
    check(load().snpm_calculate_likelihoods_many(device, ptr(scores), ptr(ninfo), S, K, int(calc), 0.0 if calc else float(amin),
                                                 ptr(prob), ptr(lik), ptr(lr)))
    return prob, lik, lr


def selection_masks(acc_lists, n_acc):
    """uint32 [len(acc_lists), row words] accession bit masks for Batch.set_segregation_filter: bit j of word w selects
    accession 32w + j, the layout of a packed row (rows padded to an even number of words)."""
    words = 2 * ((int(n_acc) + 63) // 64)
    sel = np.zeros((len(acc_lists), words), dtype=np.uint32)
    for s, acc in enumerate(acc_lists):
        acc = np.asarray(acc, dtype=np.int64)
        assert acc.size == 0 or (acc.min() >= 0 and acc.max() < n_acc), "accession index outside the panel"
        np.bitwise_or.at(sel[s], acc >> 5, (np.uint32(1) << (acc & 31).astype(np.uint32)))
    return sel


def score_grouped(db, offsets, s_chrom_id, s_pos, wei, skip_db_hets=False, grouped=None, batch=None):
    """Throughput scoring of many samples (Genotyper.genotyper per sample, snpmatch.py:207-233) with the grouped kernel:
    returns the dict of Batch.fetch().  Samples whose truncated score would depend on the reference's summation order
    (guard_counts > 0, ~1e-7 per accession) are re-scored with the order-exact fp64 kernel, so `matches` is always the
    reference's.  Falls back to the fp64 kernel for every sample when the weights do not qualify for grouping."""
    offsets = as_c(offsets, np.int64)
    s_chrom_id = as_c(s_chrom_id, np.int32)
    s_pos = as_c(s_pos, np.int32)
    wei = as_c(wei, np.float64).reshape(-1, 3)
    g = grouped if grouped is not None else group_markers(offsets, s_chrom_id, s_pos, wei)
    own = batch is None
    b = batch if batch is not None else Batch(db, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3)))
    try:
        if g is None:
            b.upload(offsets, s_chrom_id, s_pos, wei)
            b.run(skip_db_hets)
            b.epilogue()
            r = b.fetch()
            r["rescored"] = np.arange(len(offsets) - 1)
            return r
        b.upload_grouped(g)
        b.run(skip_db_hets, kernel_mode=KERNEL_GROUPED)
        b.epilogue()
        r = b.fetch()
        flagged = np.flatnonzero(b.guard_counts())
        r["rescored"] = flagged
        for s in flagged:
            lo, hi = int(offsets[s]), int(offsets[s + 1])
            b.upload([0, hi - lo], s_chrom_id[lo:hi], s_pos[lo:hi], wei[lo:hi])
            b.run(skip_db_hets)
            b.epilogue()
            one = b.fetch()
            for k in ("score", "matches", "ninfo", "prob", "L", "LR", "m"):
                r[k][s] = one[k][0]
        return r
    finally:
        if own:
            b.close()


def score_coded(db, cs, s_chrom_id=None, s_pos=None, wei=None, skip_db_hets=False, batch=None, flags=None):
    """Throughput scoring of many samples (Genotyper.genotyper per sample, snpmatch.py:207-233) from CodedSamples: join,
    grouping by weight triple and counting all on the device.  Returns the dict of Batch.fetch() plus "rescored".  Samples
    whose truncated score would depend on the reference's summation order (guard_counts > 0) are re-scored with the
    order-exact fp64 kernel when their position-order arrays (s_chrom_id, s_pos, wei of the whole batch) are given (else from
    the codes: table[codes] gives the weights back bit for bit).  Pass a `batch` to keep its device buffers between calls: a
    fresh batch costs 0.3 - 1 s of cudaMalloc / cudaFree per call on a loaded device (core.batch.genotype_many keeps one).
    flags (optional, one per marker of cs in upload order): r["flagged"] = Batch.count_flagged_pairs of the coded run."""
    own = batch is None
    b = batch if batch is not None else Batch(db, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3)))
    try:
        b.set_track_pairs(False)                    # scores only: the marker indices of the pairs are not read back
        b.upload_coded(cs)
        b.run(skip_db_hets, kernel_mode=KERNEL_GROUPED)
        b.epilogue()
        r = b.fetch()
        if flags is not None:                       # before the re-scores below replace the run's pairs
            r["flagged"] = b.count_flagged_pairs(flags)
        flagged = np.flatnonzero(b.guard_counts())
        r["rescored"] = flagged
        offsets = cs.offsets
        for s in flagged:
            lo, hi = int(offsets[s]), int(offsets[s + 1])
            if wei is None:
                w = cs.wtable[cs.codes[lo:hi].astype(np.int64)]
                cid = (cs.chrom_pos[lo:hi] >> np.uint32(27)).astype(np.int32)
                cid[cid == 31] = -1
                pp = (cs.chrom_pos[lo:hi] & np.uint32((1 << 27) - 1)).astype(np.int32)
            else:
                w, cid, pp = np.asarray(wei)[lo:hi], np.asarray(s_chrom_id)[lo:hi], np.asarray(s_pos)[lo:hi]
            b.upload([0, hi - lo], cid, pp, w)
            b.run(skip_db_hets)
            b.epilogue()
            one = b.fetch()
            for k in ("score", "matches", "ninfo", "prob", "L", "LR", "m"):
                r[k][s] = one[k][0]
        return r
    finally:
        if own:
            b.close()
