"""
Database wrapper for the matching path.

Mirrors `snpmatch/core/snp_genotype.py`: `Genotype.__init__` (snp_genotype.py:26-41),
`get_positions_idxs` (:43-44) and `get_common_positions` (:46-68) — the (chrom, pos) join — with
the genotype matrix resident in HBM as 2-bit packed calls (lib.Database) instead of two HDF5
files.  `Genotype.g` keeps the attribute surface of `pygwas.genotype.HDF5Genotype`
(pygwas/genotype.py:534-673) that the matching path touches: `positions`, `chrs`, `chr_regions`,
`accessions`, `chromosomes`, and `snps[rows, :]` / `snps[:, col]` reads (served from the device).

Sources of a database:
  * `Genotype(hdf5_file, hdf5_acc_file)` — the reference's constructor; needs h5py (absent in the
    build container, so this branch is only exercised where h5py exists);
  * `Genotype.from_arrays(...)` — in-memory arrays;
  * `Genotype.synthetic(...)` — the deterministic panel of SURVEY 8d, generated in HBM;
  * `Genotype.load_packed(path)` / `save_packed(path)` — native 2-bit file (npz of packed words).
"""
import logging
import os.path
import re

import numpy as np

from .. import lib
from . import labels
from . import parsers  # noqa: F401  (the reference module exposes snp_genotype.parsers)

log = logging.getLogger(__name__)

chunk_size = 1000
_CHR_RE = re.compile("chr", re.IGNORECASE)


def normalize_chr_names(chrs):
    """parsers.py:161 — delete every 'chr' (any case).  Computed on the distinct names only (labels.map_labels)."""
    return labels.map_labels(chrs, lambda c: _CHR_RE.sub("", c))[0]


def load_genotype_files(h5file, hdf5_acc_file=None):
    return Genotype(h5file, hdf5_acc_file)


def order_markers(cid, sample_pos):
    """(order, chrom_id int32, pos int32) for the device join from per-marker database chromosome ids (-1 = not in the
    database): markers grouped by chromosome id (unknown last), inside a chromosome in the caller's order."""
    cid = np.asarray(cid)
    sample_pos = np.asarray(sample_pos)
    n = len(cid)
    if n and int(sample_pos.min()) >= -2**31 and int(sample_pos.max()) < 2**31 - 1 and int(cid.min()) >= 0:
        # the common case in two cheap passes: every position fits, every chromosome is known
        in_range = np.ones(n, dtype=bool)
        cid = cid.astype(np.int32, copy=False)
        sort_key = cid
    else:
        in_range = (sample_pos >= -2**31) & (sample_pos < 2**31 - 1)
        cid = np.where(in_range, cid, -1).astype(np.int32)
        sort_key = np.where(cid < 0, np.int64(2**31), cid.astype(np.int64))
    if len(sort_key) < 2 or bool(np.all(sort_key[1:] >= sort_key[:-1])):      # already grouped by chromosome in database order: nothing moves
        order = np.arange(len(cid), dtype=np.int64)
        cid_o = cid
        pos_o = sample_pos.astype(np.int32) if sort_key is cid else np.where(in_range, sample_pos, 0).astype(np.int32)
    else:
        order = np.argsort(sort_key, kind="stable")
        cid_o = cid[order]
        pos_o = np.where(in_range, sample_pos, 0)[order].astype(np.int32)
    # the join needs strictly ascending positions inside a chromosome (the reference's implicit
    # precondition, SURVEY A.1); sort a chromosome that is not
    bad = (cid_o[1:] == cid_o[:-1]) & (cid_o[1:] >= 0) & (pos_o[1:] <= pos_o[:-1])
    if bad.any():
        log.warning("sample positions are not sorted inside a chromosome; sorting them for the join")
        k = np.lexsort((pos_o, np.where(cid_o < 0, np.int64(2**31), cid_o.astype(np.int64))))
        order, cid_o, pos_o = order[k], cid_o[k], pos_o[k]
        dup = (cid_o[1:] == cid_o[:-1]) & (cid_o[1:] >= 0) & (pos_o[1:] == pos_o[:-1])
        if dup.any():                      # a repeated marker cannot be paired one-to-one: keep the first
            cid_o = cid_o.copy()
            cid_o[1:][dup] = -1
            k2 = np.argsort(np.where(cid_o < 0, np.int64(2**31), cid_o.astype(np.int64)), kind="stable")
            order, cid_o, pos_o = order[k2], cid_o[k2], pos_o[k2]
    return order, np.ascontiguousarray(cid_o), np.ascontiguousarray(pos_o)


def join_coded(c1, p1, c2, p2, n_chr, device=0):
    """Inner join of two marker lists on (chromosome code, position) on the device: side 1 is indexed as a one-accession
    panel.  Codes are integers in [0, n_chr) (side 2: anything else = no partner).  Returns (i1, i2), paired, ordered by
    (code, position)."""
    c1, p1 = np.asarray(c1, dtype=np.int64), np.asarray(p1, dtype=np.int64)
    if len(c1) == 0 or len(c2) == 0:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    if np.all((c1[1:] > c1[:-1]) | ((c1[1:] == c1[:-1]) & (p1[1:] > p1[:-1]))):
        o1 = np.arange(len(p1))                    # already grouped by chromosome with ascending positions
    else:
        o1 = np.lexsort((p1, c1))
    counts = np.bincount(c1, minlength=n_chr)
    ends = np.cumsum(counts)
    regions = np.stack([ends - counts, ends], axis=1)
    c2 = np.asarray(c2, dtype=np.int64)
    cid2 = np.where((c2 >= 0) & (c2 < n_chr), c2, -1)
    order2, cid2_o, pos2_o = order_markers(cid2, p2)
    db = lib.Database(p1[o1].astype(np.int32), regions, 1, device=device)
    try:
        db_idx, s_idx = db.intersect(cid2_o, pos2_o, lib.JOIN_AUTO)
    finally:
        db.close()
    return o1[db_idx], order2[s_idx]


class _SnpsView(object):
    """`g.snps[rows, :]` (snpmatch.py:222) and `g_acc.snps[:, col]` (csmatch.py:116) served by
    unpacking the HBM-resident rows."""

    def __init__(self, panel):
        self._panel = panel
        self.shape = (panel.num_snps, panel.num_accessions)
        self.dtype = np.dtype("int8")

    def __getitem__(self, key):
        n_rows, n_acc = self.shape
        if not isinstance(key, tuple):
            key = (key, slice(None))
        rows, cols = key
        if isinstance(rows, slice) and rows == slice(None) and not isinstance(cols, slice):
            # whole columns (g_acc.snps[:, ix], csmatch.py:116, simulate.py:15): a column kernel on the resident rows,
            # one sector per row instead of unpacking the panel
            scalar_col = np.isscalar(cols)
            ix = np.atleast_1d(np.asarray(cols, dtype=np.int64))
            ix = np.where(ix < 0, ix + n_acc, ix)
            out = self._panel.db.read_columns(ix)
            return out[0] if scalar_col else np.ascontiguousarray(out.T)
        if isinstance(rows, slice):
            rows = np.arange(*rows.indices(n_rows))
            scalar_row = False
        else:
            scalar_row = np.isscalar(rows)
            rows = np.atleast_1d(np.asarray(rows, dtype=np.int64))
        out = np.empty((len(rows), n_acc), dtype=np.int8)
        step = max(1, (64 << 20) // max(n_acc, 1))
        for i in range(0, len(rows), step):
            out[i:i + step] = self._panel.db.read_rows(rows[i:i + step] - 0)
        out = out[:, cols]
        return out[0] if scalar_row else out


class Panel(object):
    """What `Genotype.g` / `Genotype.g_acc` expose (HDF5Genotype attribute surface)."""

    def __init__(self, db, positions, chrs, chr_regions, accessions):
        self.db = db
        self.positions = np.asarray(positions, dtype=np.int32)
        self.chrs = np.asarray(chrs)
        self.chr_regions = np.asarray(chr_regions, dtype=np.int64).reshape(-1, 2)
        self.accessions = np.asarray(accessions)
        self.num_snps = len(self.positions)
        self.num_accessions = len(self.accessions)
        self.snps = _SnpsView(self)

    @property
    def chromosomes(self):
        """One label per row (pygwas/genotype.py:156-161) — built lazily, never on the hot path."""
        reps = (self.chr_regions[:, 1] - self.chr_regions[:, 0]).astype(int)
        return np.repeat(self.chrs.astype("U"), reps).tolist()


class Genotype(object):

    def __init__(self, hdf5_file, hdf5_acc_file=None, device=0):
        assert hdf5_file is not None or hdf5_acc_file is not None, "Provide atleast one hdf5 genotype file"
        path = hdf5_file if hdf5_file is not None else hdf5_acc_file
        assert os.path.isfile(path), "Path to %s seems to be broken" % path
        if path.endswith(".npz"):
            self._init_from_packed(path, device)
            return
        try:
            import h5py
        except ImportError:
            raise ImportError("reading %s needs h5py; convert the database once with Genotype.save_packed "
                              "where h5py is available, or use Genotype.from_arrays" % path)
        with h5py.File(path, "r") as h5:          # schema: pygwas/genotype.py:310-328
            positions = h5["positions"][:]
            accessions = h5["accessions"][:]
            chrs = h5["positions"].attrs["chrs"]
            chr_regions = h5["positions"].attrs["chr_regions"]
            db = lib.Database(positions, chr_regions, len(accessions), device=device)
            snps = h5["snps"]
            step = max(1, (256 << 20) // max(len(accessions), 1))
            for r in range(0, len(positions), step):
                db.load_int8(snps[r:r + step, :], row0=r)
        self._finish(db, positions, chrs, chr_regions, accessions)

    # ---- alternative constructors ------------------------------------------------------------------
    @classmethod
    def from_arrays(cls, snps, positions, chrs, chr_regions, accessions, device=0):
        self = object.__new__(cls)
        snps = np.asarray(snps)
        db = lib.Database(positions, chr_regions, snps.shape[1], device=device)
        db.load_int8(snps)
        self._finish(db, positions, chrs, chr_regions, accessions)
        return self

    @classmethod
    def synthetic(cls, n_rows, n_acc, seed=None, device=0, row_range=None):
        """The deterministic panel of synth.py generated in HBM.  row_range=(r0, r1) keeps only
        that SNP-row shard on this device (multi-GPU); indices returned by the join stay global."""
        from .. import sharding, synth
        seed = synth.SEED_PANEL if seed is None else seed
        positions, regions = synth.panel_positions(n_rows, seed=seed)
        r0, r1 = (0, n_rows) if row_range is None else row_range
        local_regions = sharding.local_regions(regions, r0, r1)
        self = object.__new__(cls)
        db = lib.Database(positions[r0:r1], local_regions, n_acc, device=device, row0_global=r0)
        db.fill_synthetic(seed)
        self._finish(db, positions[r0:r1], np.array(synth.TAIR10_CHRS, dtype="str"), local_regions, synth.accession_ids(n_acc))
        self.global_chr_regions = regions
        return self

    @classmethod
    def load_packed(cls, path, device=0):
        self = object.__new__(cls)
        self._init_from_packed(path, device)
        return self

    def _init_from_packed(self, path, device):
        with np.load(path, allow_pickle=False) as z:
            positions, chrs, chr_regions, accessions = z["positions"], z["chrs"], z["chr_regions"], z["accessions"]
            db = lib.Database(positions, chr_regions, len(accessions), device=device)
            db.load_packed(z["packed"])
        self._finish(db, positions, chrs, chr_regions, accessions)

    def save_packed(self, path):
        """Native 2-bit file: the packed words as they sit in HBM plus the index arrays."""
        g = self.g
        np.savez(path, packed=g.db.read_packed(0, g.num_snps), positions=g.positions, chrs=g.chrs.astype("U"),
                 chr_regions=g.chr_regions, accessions=g.accessions.astype("S"))

    def _finish(self, db, positions, chrs, chr_regions, accessions):
        self.db = db
        self.g = Panel(db, positions, chrs, chr_regions, accessions)
        self.g_acc = self.g                       # one resident copy serves row and column reads
        self.accessions = self.g.accessions.astype("U")
        self.chrs = self.g.chrs.astype("U")
        self._db_chr_norm = normalize_chr_names(self.chrs)

    # ---- sample preparation for the device -----------------------------------------------------------
    def prepare_markers(self, sample_chrs, sample_pos, style="join"):
        """Map sample markers to what crosses the C ABI: (order, chrom_id int32, pos int32) where
        `order` lists the sample's marker indices grouped by database chromosome (database order,
        markers of unknown chromosomes last) and inside a chromosome in the sample's own order —
        the order in which the reference's per-chromosome loop emits them (snp_genotype.py:60-67).

        style='join' normalises names like the join (every 'chr', any case, removed, parsers.py:161);
        style='genome' like the window iterators (lower-case then 'chr' removed, genomes.py:75,95)."""
        from . import genomes
        sample_chrs = np.asarray(sample_chrs)
        sample_pos = np.asarray(sample_pos)
        norm = (lambda c: _CHR_RE.sub("", c)) if style == "join" else (lambda c: c.lower().replace("chr", ""))
        db_norm = self._db_chr_norm if style == "join" else genomes.genome_style_ids(self.chrs)
        first = {}
        for i, name in enumerate(db_norm):
            first.setdefault(name, i)
        # per-marker names -> codes + the few distinct names; the database index is looked up per distinct name
        _, codes, uniq_norm = labels.map_labels(sample_chrs, norm, per_label=False)
        table = np.array([first.get(u, -1) for u in uniq_norm], dtype=np.int32)
        cid = table[codes] if len(codes) else np.zeros(0, dtype=np.int32)
        return order_markers(cid, sample_pos)

    # ---- A1 -------------------------------------------------------------------------------------------
    def get_positions_idxs(self, commonSNPsCHR, commonSNPsPOS, algo=lib.JOIN_AUTO):
        """Join of the sample markers with the resident database -> (db_idx, sample_idx), paired,
        ordered by (database chromosome order, position) (snp_genotype.py:43-68).  Runs on the GPU."""
        order, cid, pos = self.prepare_markers(commonSNPsCHR, commonSNPsPOS)
        db_idx, s_idx = self.db.intersect(cid, pos, algo)
        return db_idx, order[s_idx]

    @staticmethod
    def get_common_positions(input_1_chr, input_1_pos, input_2_chr, input_2_pos, device=0):
        """Join of two arbitrary marker lists (snp_genotype.py:46-68): side 1 plays the database.
        Side 1 is indexed on the device as a one-accession panel; results are mapped back to the
        callers' own orders."""
        assert len(input_1_chr) == len(input_1_pos), "Both chromosome and position array provided should be of same length"
        assert len(input_2_chr) == len(input_2_pos), "Both chromosome and position array provided should be of same length"
        p1 = np.asarray(input_1_pos).astype(np.int64)
        if len(input_1_chr) == 0 or len(input_2_chr) == 0:
            return np.zeros(0, dtype=int), np.zeros(0, dtype=int)
        # side-1 chromosomes in first-appearance order of their normalised names (parsers.py:161-163)
        _, codes1, uniq_norm = labels.map_labels(input_1_chr, lambda c: _CHR_RE.sub("", c))
        rank_of_uniq, ids = labels.factorize(uniq_norm)              # raw names that normalise to the same id share a rank
        r1 = rank_of_uniq[codes1]
        # side 2: the rank of its normalised chromosome names among side 1's
        _, codes2, uniq2 = labels.map_labels(input_2_chr, lambda c: _CHR_RE.sub("", c))
        rank = {name: i for i, name in enumerate(ids)}
        r2 = np.array([rank.get(u, -1) for u in uniq2], dtype=np.int64)[codes2]
        idx1, idx2 = join_coded(r1, p1, r2, input_2_pos, len(ids), device=device)
        # reference order: per chromosome (side-1 order) each side in its own order
        k1 = np.lexsort((idx1, r1[idx1]))
        k2 = np.lexsort((idx2, r1[idx1]))
        return idx1[k1], idx2[k2]

    def close(self):
        if getattr(self, "_many_batch", None) is not None:      # the batch of core.batch.genotype_many
            self._many_batch.close()
            self._many_batch = None
        if getattr(self, "_inbred_batch", None) is not None:    # the batch of core.snpmatch.inbred_identify_many
            self._inbred_batch.close()
            self._inbred_batch = None
        if getattr(self, "_cross_batch", None) is not None:     # the batch of core.csmatch.cross_identify_many
            self._cross_batch.close()
            self._cross_batch = None
        if getattr(self, "db", None) is not None:
            self.db.close()
            self.db = None
