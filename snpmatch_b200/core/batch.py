"""
Batched many-sample mode (north-star item (d), SURVEY.md section 8a row A9).

The reference has no batched entry point: many samples are genotyped as one `snpmatch inbred` process per sample
(README.md:9).  When the samples are CALLED genotypes (BED files, VCFs without PL: one-hot weights,
parsers.py:132-139) they can instead be scored together: their matched database rows are merged into one shared marker
panel, every sample becomes a row of 2-bit calls on that panel, and scores and informative-site counts of all samples
against all accessions come out of ONE one-hot int8 GEMM on the tensor cores (csrc/gemm_onehot.cuh).  Results equal
those of `Genotyper.genotyper` run sample by sample (integers, exactly).
"""
import numpy as np

from .. import lib
from . import parsers
from . import snpmatch


def shared_panel(g, samples):
    """Join every sample with the database (GPU) and merge the matched rows.
    Returns (panel_rows int64[K] global rows ascending, codes uint8 [S,K] with 3 = sample lacks the marker,
    matched list of (db_idx, sample_idx) per sample)."""
    matched = []
    for inp in samples:
        matched.append(g.get_positions_idxs(inp.chrs, inp.pos))
    rows = np.unique(np.concatenate([m[0] for m in matched])) if matched else np.zeros(0, dtype=np.int64)
    codes = np.full((len(samples), len(rows)), 3, dtype=np.uint8)
    for i, (inp, (db_idx, s_idx)) in enumerate(zip(samples, matched)):
        c = parsers.parseGT(np.asarray(inp.gt)[s_idx])            # 0 ref, 1 alt, 2 het, -1 no call
        col = np.searchsorted(rows, db_idx)
        codes[i, col] = np.where(c < 0, 3, c).astype(np.uint8)
    return rows.astype(np.int64), codes, matched


def genotype_batch(g, samples, skip_db_hets=False):
    """Score S called-genotype samples in one tensor-core pass; returns (list of GenotyperOutput, info dict).
    Every sample's weights must be one-hot (use Genotyper for likelihood-weighted samples)."""
    for inp in samples:
        assert lib.weights_are_one_hot(inp.wei), "genotype_batch scores called genotypes; use Genotyper for PL-weighted samples"
    rows, codes, matched = shared_panel(g, samples)
    local_rows = rows                                             # score_shared_panel takes global rows
    r = g.db.score_shared_panel(local_rows, codes, skip_db_hets=skip_db_hets)
    out = []
    for i, (inp, (db_idx, _)) in enumerate(zip(samples, matched)):
        m = len(db_idx)
        res = snpmatch.GenotyperOutput(g.g.accessions, r["matches"][i], r["ninfo"][i], snpmatch.get_fraction(m, len(inp.pos)), m, inp.dp)
        res._attach_fused(r["prob"][i], r["L"][i], r["LR"][i])
        out.append(res)
    return out, {"panel_markers": len(rows), "gemm_ms": r["gemm_ms"]}


def _is_identity(order):
    n = len(order)
    return n == 0 or (order[0] == 0 and order[-1] == n - 1 and bool(np.all(order[1:] > order[:-1])))


def coded_batch(g, samples, with_weights=True, prepared=None):
    """lib.CodedSamples of a list of ParseInputs: every sample's markers in the order the join wants (database chromosome
    order, position), chromosome id + position in one word, weights as dictionary codes (ParseInputs.coded_weights: the
    integer PLs of a VCF, or a one-off np.unique for other inputs) into ONE table for the batch.  Returns (CodedSamples or
    None, offsets, chrom ids, positions, weights) — the last three in upload order, for re-scoring flagged samples (weights:
    None unless `with_weights` or the samples cannot be coded; table[codes] gives them back bit for bit).  `prepared`: the
    samples' g.prepare_markers results when the caller has them already.
    Per-marker work is skipped wherever the input allows it: a file that is already in the join's order is not permuted, and
    samples whose tables are prefixes of one table (VCFs: code = PL, table = exp(-PL/10)) keep their codes as they are."""
    if prepared is None:
        prepared = [g.prepare_markers(inp.chrs, inp.pos) for inp in samples]
    ident = [_is_identity(p[0]) for p in prepared]
    offs = np.concatenate([[0], np.cumsum([len(p[2]) for p in prepared])]).astype(np.int64)
    cid = np.concatenate([p[1] for p in prepared]) if samples else np.zeros(0, np.int32)
    pos = np.concatenate([p[2] for p in prepared]) if samples else np.zeros(0, np.int32)

    def weights():
        if not samples:
            return np.zeros((0, 3))
        return np.concatenate([np.asarray(inp.wei, dtype=np.float64) if same else np.asarray(inp.wei, dtype=np.float64)[p[0]]
                               for inp, p, same in zip(samples, prepared, ident)])

    coded = [inp.coded_weights() for inp in samples]
    cs = None
    if all(c is not None for c in coded) and samples:
        # one table for the batch: the longest table when every other one is a prefix of it (bit patterns), else the union of
        # the tables with every sample's codes remapped into it
        tables = [np.ascontiguousarray(c[1], dtype=np.float64).view(np.uint64) for c in coded]
        longest = max(tables, key=len)
        if all(np.array_equal(t, longest[:len(t)]) for t in tables):
            union, remaps = longest, [None] * len(tables)
        else:
            union, inv = np.unique(np.concatenate(tables), return_inverse=True)
            remaps, at = [], 0
            for t in tables:
                remaps.append(inv[at:at + len(t)].astype(np.uint16))
                at += len(t)
        if len(union) <= 65536:
            codes = []
            for (c, _), p, same, remap in zip(coded, prepared, ident, remaps):
                c = np.asarray(c, dtype=np.uint16)
                if not same:
                    c = c[p[0]]
                codes.append(c if remap is None else remap[c])
            cs = lib.code_markers(offs, cid, pos, codes=np.concatenate(codes), wtable=union.view(np.float64))
    return cs, offs, cid, pos, (weights() if with_weights or cs is None else None)


def genotype_many(g, samples, skip_db_hets=False):
    """Genotyper.genotyper (snpmatch.py:207-233) for MANY samples with any weights (PL likelihoods or called genotypes) in
    one device pass: markers go up in position order with their weights as dictionary codes (`coded_batch`), the device
    joins them with the panel, groups the matched pairs by weight triple (csrc/group_sort.cuh) and scores them with the
    counting kernel (csrc/grouped2.cuh).  Returns the list of GenotyperOutput, one per sample, with matches / ninfo / overlap
    identical to Genotyper run sample by sample and likelihoods within 1e-9; samples whose int(score) would depend on the
    reference's summation order are re-scored by the order-exact kernel inside `lib.score_coded`.  Inputs that cannot be
    coded (more than 65536 distinct weight values, negative weights) take the order-exact kernel for every sample."""
    cs, offs, cid, pos, wei = coded_batch(g, samples, with_weights=False)     # flagged samples get their weights back from the codes
    if cs is not None:
        # one batch object lives with the panel: its device buffers (key tables, partial sums, results: ~150 MB for 64 samples)
        # are allocated once, not per call (cudaMalloc / cudaFree of a fresh batch cost 0.3 - 1 s per call on a loaded device)
        if getattr(g, "_many_batch", None) is None:
            g._many_batch = lib.Batch(g.db, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3)))
        r = lib.score_coded(g.db, cs, cid, pos, wei, skip_db_hets=skip_db_hets, batch=g._many_batch)
    else:
        r = lib.score_grouped(g.db, offs, cid, pos, wei, skip_db_hets=skip_db_hets)
    out = []
    for i, inp in enumerate(samples):
        m = int(r["m"][i])
        res = snpmatch.GenotyperOutput(g.g.accessions, r["score"][i], r["ninfo"][i], snpmatch.get_fraction(m, len(inp.pos)), m, inp.dp)
        res._attach_fused(r["prob"][i], r["L"][i], r["LR"][i])
        out.append(res)
    return out
