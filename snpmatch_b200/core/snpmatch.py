"""
`snpmatch inbred` — host side of the B200 matching path.

Mirrors the public surface of the reference's `snpmatch/core/snpmatch.py`: module constants
(:17-19), `get_fraction` (:25-28), `likeliTest` (:40-55), `np_test_identity` (:57-72),
`matchGTsAccs` (:74-89), `GenotyperOutput` (:91-168), `Genotyper` (:170-241), `getHeterozygosity`
(:244-253), `potatoGenotyper` (:256-268), `pairwiseScore` (:270-309).  All array arithmetic of the path — the join, the
per-accession reduction, truncation, probabilities, likelihoods and ratios — runs in
libsnpmatch_b200 on the GPU (snpmatch_b200/csrc); this file only prepares buffers and writes the
reference's output files (`scores.txt`, `matches.json`).
"""
import json
import logging
import os
import sys

import numpy as np
import pandas as pd

from .. import lib
from . import labels
from . import parsers
from . import snp_genotype

log = logging.getLogger(__name__)
lr_thres = 3.841
snp_thres = 4000
prob_thres = 0.98


def die(msg):
    sys.stderr.write('Error: ' + msg + '\n')
    sys.exit(1)


def get_fraction(x, y, y_min=0):
    if y <= y_min:
        return np.nan
    return float(x) / y


np_get_fraction = np.vectorize(get_fraction, excluded="y_min")


def likeliTest(n, y):
    """Likelihood of y matches out of n informative sites (snpmatch.py:40-55), evaluated by the
    device epilogue (csrc/score.cuh: likeli_test) so that scalars and arrays agree bit for bit."""
    assert y <= n, "provided y is greater than n"
    _, lik, _ = lib.calculate_likelihoods(np.array([y], dtype=np.float64), np.array([n], dtype=np.float64))
    return float(lik[0])


_KMAX_CACHE = {}


def identity_kmax_table(n_max, error_rate=0.02, pthres=0.05):
    """kmax[n] = largest k with binom.sf(k - 1, n, error_rate) >= pthres, for n = 0..n_max.

    np_test_identity (snpmatch.py:57-72) is `binom.sf((n - x) - 1, n, e) >= pthres`; SciPy floors
    the first argument and sf is non-increasing in it, so identical <=> floor(n - x - 1) + 1 <=
    kmax[n].  The table is built with the same SciPy function the reference calls, which makes the
    device's identity calls bit-exact by construction."""
    from scipy import stats
    key = (float(error_rate), float(pthres))
    have = _KMAX_CACHE.get(key)
    if have is not None and len(have) > n_max:
        return have
    n_max = max(int(n_max), 64)
    n = np.arange(n_max + 1)
    # candidate from the inverse survival function, then fix up with sf itself
    k = np.clip(stats.binom.isf(pthres, n, error_rate).astype(np.int64) + 1, 0, n + 1)
    for _ in range(64):
        ok_here = stats.binom.sf(k - 1, n, error_rate) >= pthres
        ok_next = stats.binom.sf(k, n, error_rate) >= pthres
        up = ok_here & ok_next & (k < n + 1)
        down = ~ok_here & (k > 0)
        if not (up.any() or down.any()):
            break
        k = np.where(up, k + 1, np.where(down, k - 1, k))
    table = k.astype(np.int32)
    _KMAX_CACHE[key] = table
    return table


def np_test_identity(x, n, error_rate=0.0005, pthres=0.05):
    """snpmatch.py:70-72 through the kmax table (host integers; the windowed path evaluates the same
    comparison on the device)."""
    x = np.asarray(x, dtype=np.float64)
    n = np.asarray(n)
    table = identity_kmax_table(int(np.max(n)) if n.size else 0, error_rate, pthres)
    return np.array(np.floor(n - x - 1) + 1 <= table[n.astype(np.int64)]).astype(int)


def matchGTsAccs(sampleWei, t1001snps, skip_hets_db=False):
    """Weighted genotype match of k markers against every accession (snpmatch.py:74-89) on the GPU:
    returns (score f64[A], ninfo int[A]) in the reference's summation order."""
    sampleWei = np.asarray(sampleWei)
    t1001snps = np.asarray(t1001snps)
    assert sampleWei.shape[0] == t1001snps.shape[0], "please provide same number of positions for both sample and db"
    assert sampleWei.ndim == 2 and sampleWei.shape[1] == 3, "SNP weights should be a np.array with  shape == n,3"
    return lib.match_gts_accs(sampleWei, t1001snps, skip_hets_db)


class GenotyperOutput(object):
    """Result table of a run (snpmatch.py:91-168)."""

    def __init__(self, AccList, ScoreList, NumInfoSites, overlap, NumMatSNPs, DPmean):
        self._fused = None
        self.overlap, self.num_snps, self.dp = overlap, NumMatSNPs, DPmean
        self.accs = np.asarray(AccList).astype("str")
        self.ninfo = np.asarray(NumInfoSites).astype("int")
        self.scores = np.asarray(ScoreList).astype("int")     # truncation toward zero (snpmatch.py:96)

    def _attach_fused(self, prob, lik, lrt):
        """Results of the epilogue that ran fused behind the scoring kernels."""
        self._fused = (len(self.accs), np.array(prob), np.array(lik), np.array(lrt))

    def _fused_ok(self):
        return self._fused is not None and self._fused[0] == len(self.scores)

    def get_probabilities(self):
        if self._fused_ok():
            self.probabilies = self._fused[1]
        else:
            self.probabilies, _, _ = lib.calculate_likelihoods(self.scores, self.ninfo)

    @staticmethod
    def calculate_likelihoods(scores, ninfo, amin="calc"):
        """(L, LR) of snpmatch.py:106-117, computed by the device epilogue."""
        _, lik, lrt = lib.calculate_likelihoods(scores, ninfo, amin)
        return lik, lrt

    def get_likelihoods(self, amin="calc"):
        if amin == "calc" and self._fused_ok():
            self.likelis, self.lrts = self._fused[2], self._fused[3]
        else:
            self.likelis, self.lrts = self.calculate_likelihoods(self.scores, self.ninfo, amin)

    def print_out_table(self, outFile):
        """`scores.txt`: acc, matches, ninfo, probability, likelihood, lrt, num_snps, dp; tab-separated,
        no header (snpmatch.py:122-138).  BED inputs carry dp = "NA": the mean is nan (SURVEY A.8 Q5)."""
        self.get_likelihoods()
        self.get_probabilities()
        columns = (('accs', self.accs), ('matches', self.scores), ('ninfo', self.ninfo), ('probabilities', self.probabilies),
                   ('likelihood', self.likelis), ('lrt', self.lrts), ('num_snps', self.num_snps), ('dp', parsers.mean_depth(self.dp)))
        n_rows = len(self.accs)
        table = pd.DataFrame({name: (col if np.ndim(col) else np.repeat(col, n_rows)) for name, col in columns},
                             columns=[name for name, _ in columns])
        if outFile:
            table.to_csv(outFile, sep="\t", header=False, index=False)
        return table

    def print_json_output(self, outFile):
        """`matches.json` (snpmatch.py:140-150)."""
        self.get_likelihoods()
        self.get_probabilities()
        with np.errstate(invalid="ignore"):
            topHits = np.where(self.lrts < lr_thres)[0]
        by_probability = topHits[np.argsort(-self.probabilies[topHits])]
        case, note = self.case_interpreter(topHits)
        rows = []
        for i in by_probability:            # accession, probability, informative sites, informative sites / matched markers
            rows.append((str(self.accs[i]), float(self.probabilies[i]), int(self.ninfo[i]), float(get_fraction(self.ninfo[i], self.num_snps))))
        report = {'interpretation': {'case': case, 'text': note}, 'matches': rows, 'overlap': [self.overlap, self.num_snps]}
        with open(outFile, "w") as fh:
            json.dump(report, fh, sort_keys=True, indent=4)

    def case_interpreter(self, topHits):
        """snpmatch.py:152-168."""
        overlap_thres = 0.5
        case, note = 1, "Ambiguous sample"
        if len(topHits) == 1:
            case, note = 0, "Unique hit"
        elif np.nanmean(self.probabilies[topHits]) > prob_thres:
            case, note = 2, "Ambiguous sample: Accessions in top hits can be really close"
        elif self.overlap > overlap_thres:
            case, note = 3, "Ambiguous sample: Sample might contain mixture of DNA or contamination"
        elif self.overlap < overlap_thres:
            case, note = 4, "Ambiguous sample: Many input SNP positions are missing in db positions. Maybe sample  not one in database"
        return case, note


class Genotyper(object):
    """`snpmatch inbred` for one sample against the resident database (snpmatch.py:170-241)."""

    def __init__(self, inputs, g, outFile, run_genotyper=True, skip_db_hets=False, chunk_size=1000):
        assert type(g) is snp_genotype.Genotype, "provide a snp_genotype.Genotype class for genotypes"
        assert int(chunk_size) >= 1, "chunk_size must be a positive number of SNPs"
        self.g, self.inputs, self.outFile = g, inputs, outFile
        self.chunk_size, self._skip_db_hets = chunk_size, skip_db_hets
        self.num_lines = len(g.g.accessions)
        self.inputs.filter_chr_names()
        if run_genotyper:
            self.result = self.genotyper()
            self.write_genotyper_output(self.result)

    def get_common_positions(self):
        self.commonSNPs = self.g.get_positions_idxs(self.inputs.chrs, self.inputs.pos)

    def filter_tophits(self):
        """`--refine` (snpmatch.py:189-205): rescoring over the SNPs that segregate among the
        indistinguishable accessions."""
        self.result = self.genotyper()
        self.write_genotyper_output(self.result)
        topHits = refine_tophits(self.result, self.num_lines)
        if topHits is None:
            return None
        seg_ix = identify_segregating_snps(self.g, topHits)
        self.result_fine = self.genotyper(filter_pos_ix=seg_ix, mask_acc_ix=refine_mask(self.result))
        self.result_fine.print_out_table(self.outFile + ".refined.scores.txt")

    def genotyper(self, filter_pos_ix=None, mask_acc_ix=None):
        """Join + chunked scoring + epilogue in one device pass (snpmatch.py:207-233)."""
        g = self.g
        order, cid, pos = g.prepare_markers(self.inputs.chrs, self.inputs.pos)
        wei = np.ascontiguousarray(np.asarray(self.inputs.wei, dtype=np.float64)[order])
        # called genotypes (BED, VCF without PL) take the popcount kernel; likelihood-weighted samples the fp64 one, which
        # sums in the reference's chunks of `chunk_size` rows (snpmatch.py:173,218: the chunking is part of its rounding)
        mode = lib.KERNEL_POPCOUNT if lib.weights_are_one_hot(wei) else lib.KERNEL_FP64
        batch = g.db.scratch_batch([0, len(pos)], cid, pos, wei,
                                   chunk_rows=int(self.chunk_size) if mode == lib.KERNEL_FP64 else lib.CHUNK_ROWS)
        try:
            if filter_pos_ix is not None:
                assert type(filter_pos_ix) is np.ndarray, "provide np array for indices to be considered"
                batch.set_row_filter(filter_pos_ix)
            batch.run(self._skip_db_hets, kernel_mode=mode)
            batch.epilogue()
            r = batch.fetch()
            db_idx, s_idx = batch.fetch_pairs(0)
            self.timings = batch.timings()
        finally:
            batch.close()
        if filter_pos_ix is not None and len(db_idx) < 100:
            log.info("#positions in segregating sites are are too little: %s" % len(db_idx))
        self.commonSNPs = (db_idx, order[s_idx])
        out = genotyper_output(g.g.accessions, r["score"][0], r["ninfo"][0], len(self.inputs.pos), int(r["m"][0]), self.inputs.dp,
                               mask_acc_ix)
        if mask_acc_ix is None:
            out._attach_fused(r["prob"][0], r["L"][0], r["LR"][0])
        return out

    def write_genotyper_output(self, result):
        write_scores_and_matches(result, self.outFile)
        getHeterozygosity(self.inputs.gt[self.commonSNPs[1]], self.outFile + ".matches.json")
        return result


# ---- host steps of `inbred` shared by Genotyper and inbred_identify_many --------------------------------------------------
def genotyper_output(accs, score, ninfo, n_markers, NumMatSNPs, dp, mask_acc_ix=None):
    """GenotyperOutput of one sample's totals (snpmatch.py:228-233); mask_acc_ix drops those accessions (the refined table)."""
    overlap = get_fraction(NumMatSNPs, n_markers)
    if mask_acc_ix is not None:
        assert type(mask_acc_ix) is np.ndarray, "provide a numpy array of accessions indices to mask"
        keep = np.setdiff1d(np.arange(len(accs)), mask_acc_ix)
        return GenotyperOutput(accs[keep], score[keep], ninfo[keep], overlap, NumMatSNPs, dp)
    return GenotyperOutput(accs, score, ninfo, overlap, NumMatSNPs, dp)


def write_scores_and_matches(result, outFile):
    """<outFile>.scores.txt and <outFile>.matches.json without the heterozygosity (snpmatch.py:235-241)."""
    log.info("writing %s.scores.txt and %s.matches.json", outFile, outFile)
    result.get_likelihoods()
    result.print_out_table(outFile + '.scores.txt')
    result.print_json_output(outFile + ".matches.json")


def refine_tophits(result, num_lines):
    """The accessions `--refine` re-scores (snpmatch.py:193-202), or None when there is nothing to refine: a single top hit, or
    more than half of the panel's `num_lines` accessions.  An empty array means no top hit at all (every ratio nan)."""
    result.get_likelihoods()
    with np.errstate(invalid="ignore"):
        topHits = np.where(result.lrts < lr_thres)[0]
    if len(topHits) == 1:
        log.info("a single accession is left: perfect hit, nothing to refine")
        return None
    log.info("%s accessions cannot be told apart at LR < %s", len(topHits), lr_thres)
    if len(topHits) > (num_lines / 2):
        log.info("more than half of the panel is indistinguishable: not refining")
        return None
    return topHits


def refine_mask(result):
    """Accessions the refined table leaves out (snpmatch.py:203): LR >= lr_thres; nan ratios stay in."""
    with np.errstate(invalid="ignore"):
        return np.where(result.lrts >= lr_thres)[0]


def identify_segregating_snps(g, accs_ix):
    """Rows where the given accessions carry more than one distinct called genotype (snp_genotype.py:188-211 with
    segregting_snps :378-383).  One scan of the resident panel on the GPU.  Like the reference, returns None when more
    than half of the accessions are selected."""
    assert type(accs_ix) is np.ndarray, "provide an np array for list of indices to be considered"
    assert len(accs_ix) > 1, "polymorphism happens in more than 1 line"
    if len(accs_ix) > (len(g.accessions) / 2):
        return None
    return g.db.segregating_rows(accs_ix) + g.db.row0_global


def getHeterozygosity(snpGT, outFile='default'):
    """Fraction of heterozygous calls among the matched markers; added to the JSON (snpmatch.py:244-253)."""
    snpBinary = parsers.parseGT(snpGT)
    return write_heterozygosity(int(np.count_nonzero(snpBinary == 2)), len(snpGT), outFile)


def write_heterozygosity(numHets, numSNPs, outFile='default'):
    """percent_heterozygosity = numHets / numSNPs, added to the JSON `outFile` (snpmatch.py:249-253)."""
    frac = get_fraction(numHets, numSNPs)
    if outFile != 'default':
        with open(outFile) as fh:
            report = json.load(fh)
        report['percent_heterozygosity'] = frac
        with open(outFile, "w") as fh:
            json.dump(report, fh, sort_keys=True, indent=4)
    return frac


def potatoGenotyper(args):
    inputs = parsers.ParseInputs(inFile=args['inFile'], logDebug=args['logDebug'])
    log.info("packing the database into HBM")
    g = snp_genotype.Genotype(args['hdf5File'], args['hdf5accFile'])
    log.info("matching the sample against %s accessions", len(g.accessions))
    genotyper = Genotyper(inputs, g, args['outFile'], run_genotyper=not args['refine'], skip_db_hets=args['skip_db_hets'])
    if args['refine']:                       # --refine: score, then re-score the indistinguishable accessions on their segregating SNPs
        genotyper.filter_tophits()
    log.info("finished!")


# Device memory one launch of inbred_identify_many may take, and what a sample takes of it: per marker the join, key, pair and
# weight arrays of both passes (~128 bytes), per segment of the counting kernel (320 markers) and of the order-exact kernel
# (chunk_size markers) the partial sums over the padded panel row (16 and 12 bytes per column), and per sample the key and group
# tables of the device grouping (~192 KB), the reduce buffer and the result arrays.  ~10 MB per 50 k-marker sample at 1135
# accessions, ~7x that at 20 000.
INBRED_BUDGET_BYTES = 8 << 30


def inbred_bytes_per_sample(n_markers, n_acc, row_words, chunk_size=1000):
    n, a_pad = int(n_markers), 32 * int(row_words)
    segs = -(-n // 320) * 16 + -(-n // int(chunk_size)) * 12
    return n * 128 + segs * a_pad + (192 << 10) + (8 * int(n_acc) + 2) * 8


def _het_flags(gt):
    """parseGT(gt) == 2 per marker, or None when the calls mix formats: parseGT sniffs its format from the first call it is
    given, so the heterozygous count of a subset (the matched markers) equals the flags' count only when every call has the
    format of the first."""
    gt = np.asarray(gt)
    if len(gt) == 0:
        return np.zeros(0, dtype=bool)
    first = str(gt[0])
    text = gt.astype("str")
    if "|" in first:
        same = np.char.find(text, "|") >= 0
    elif "/" in first:
        same = (np.char.find(text, "/") >= 0) & (np.char.find(text, "|") < 0)
    elif first.isdigit():
        same = np.char.isdigit(text)
    else:
        return None
    return parsers.parseGT(gt) == 2 if bool(np.all(same)) else None


def holds_whole_panel(g):
    """False when the Genotype holds a row shard of its panel (the many-sample paths need every row on one device)."""
    return g.db.row0_global == 0 and g.db.n_rows == int(np.max(getattr(g, "global_chr_regions", [[0, g.db.n_rows]])))


def inbred_identify_many(inputs_list, g, output_ids, refine=False, skip_db_hets=False, chunk_size=1000, samples_per_launch=None):
    """`inbred` (and `inbred --refine`) for many samples: every sample's files (<id>.scores.txt, <id>.matches.json and, when it
    refines, <id>.refined.scores.txt) are byte for byte the ones Genotyper (+ filter_tophits) writes for it alone.
    Per launch of samples: one coded counting pass for all of them (core.batch.coded_batch, lib.score_coded) with their
    heterozygous counts from the same run; the refine decisions on the host; one order-exact pass of every refining sample
    with a per-sample segregation filter on the device (Batch.set_segregation_filter) instead of a full-panel scan each; and
    the likelihoods of all refined tables in one call.  The host waits a fixed number of times per launch (plus one re-score
    per sample whose truncated score depends on the summation order, as in genotype_many).  Launches hold as many samples
    as fit INBRED_BUDGET_BYTES (`samples_per_launch` overrides).
    Returns one Genotyper per sample with `result`, `num_matched`, `num_hets` and, when it refined, `result_fine`.  A sample
    without any top hit (every ratio nan, e.g. no marker in the panel) cannot refine: the single path stops there with an
    assertion; here its `no_top_hits` is set, its scores and matches files are written, and the other samples go on."""
    from . import batch as batch_mod
    inputs_list, output_ids = list(inputs_list), list(output_ids)
    assert len(inputs_list) == len(output_ids), "one output prefix per sample"
    assert len(set(output_ids)) == len(output_ids), "output prefixes must differ"
    assert int(chunk_size) >= 1, "chunk_size must be a positive number of SNPs"
    if not holds_whole_panel(g):
        raise ValueError("inbred_identify_many needs the whole panel on one device; this one holds a shard of its rows")
    # every sample's chromosome names are mapped to the panel's before any device work; a bad sample is named
    gts, prepared = [], []
    for i, (inp, out) in enumerate(zip(inputs_list, output_ids)):
        try:
            assert len(inp.chrs) == len(inp.pos), "%d chromosome names for %d positions" % (len(inp.chrs), len(inp.pos))
            gts.append(Genotyper(inp, g, out, run_genotyper=False, skip_db_hets=skip_db_hets, chunk_size=chunk_size))
            prepared.append(g.prepare_markers(inp.chrs, inp.pos))
        except Exception as e:
            raise ValueError("sample %d (%s): %s" % (i, out, e)) from e
    if not gts:
        return gts
    per = samples_per_launch
    if per is None:
        biggest = max(inbred_bytes_per_sample(len(inp.pos), g.db.n_acc, g.db.row_words, chunk_size) for inp in inputs_list)
        per = max(1, INBRED_BUDGET_BYTES // biggest)
    assert int(per) >= 1, "samples_per_launch must be at least 1"
    # one batch lives with the panel: its device buffers are allocated once, not per call
    if getattr(g, "_inbred_batch", None) is None:
        g._inbred_batch = lib.Batch(g.db, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3)))
    g._inbred_batch.set_chunk_rows(int(chunk_size))         # the order-exact passes sum in Genotyper's chunks
    for c0 in range(0, len(gts), int(per)):
        _inbred_launch(gts[c0:c0 + int(per)], prepared[c0:c0 + int(per)], g._inbred_batch, batch_mod, refine)
    skipped = [gt.outFile for gt in gts if gt.no_top_hits]
    if skipped:
        log.error("no top hits, not refined: %s", ", ".join(skipped))
    return gts


def _inbred_launch(gts, prepared, batch, batch_mod, refine):
    g, skip = gts[0].g, gts[0]._skip_db_hets
    accs = g.g.accessions
    samples = [gt.inputs for gt in gts]
    flags = [_het_flags(inp.gt) for inp in samples]
    up_flags = np.concatenate([f[p[0]] if f is not None else np.zeros(len(p[0]), bool) for f, p in zip(flags, prepared)])
    # first pass: the coded counting path of genotype_many (position-order f64 weights when the weights cannot be coded)
    cs, offs, cid, pos, _ = batch_mod.coded_batch(g, samples, with_weights=False, prepared=prepared)
    if cs is not None:
        r = lib.score_coded(g.db, cs, cid, pos, None, skip_db_hets=skip, batch=batch, flags=up_flags)
    else:
        batch.upload(offs, cid, pos, _ordered_weights(samples, prepared))
        batch.run(skip, kernel_mode=lib.KERNEL_FP64)
        batch.epilogue()
        r = batch.fetch()
        r["flagged"] = batch.count_flagged_pairs(up_flags)
    for i, gt in enumerate(gts):
        m = int(r["m"][i])
        gt.result = genotyper_output(accs, r["score"][i], r["ninfo"][i], len(gt.inputs.pos), m, gt.inputs.dp)
        gt.result._attach_fused(r["prob"][i], r["L"][i], r["LR"][i])
        gt.num_matched, gt.num_hets, gt.no_top_hits = m, int(r["flagged"][i]), False
        write_scores_and_matches(gt.result, gt.outFile)
        if flags[i] is None:                                # calls in mixed formats: the single path's own count
            gt.get_common_positions()
            getHeterozygosity(gt.inputs.gt[gt.commonSNPs[1]], gt.outFile + ".matches.json")
        else:
            write_heterozygosity(gt.num_hets, m, gt.outFile + ".matches.json")
    if not refine:
        return
    todo = []
    for i, gt in enumerate(gts):
        top = refine_tophits(gt.result, gt.num_lines)
        if top is not None and len(top) == 0:
            gt.no_top_hits = True
        elif top is not None:
            todo.append((i, top))
    if todo:
        _refine_launch([gts[i] for i, _ in todo], [prepared[i] for i, _ in todo], [top for _, top in todo], batch)


def _ordered_weights(samples, prepared):
    return np.concatenate([np.asarray(inp.wei, dtype=np.float64).reshape(-1, 3)[p[0]] for inp, p in zip(samples, prepared)])


def _refine_launch(gts, prepared, tops, batch):
    """The refine pass of the samples of one launch that refine: one order-exact run with the segregation filter of every
    sample's top hits (the pairs and the summation order of Genotyper.genotyper(filter_pos_ix=...)), one fetch, one likelihood
    call for all refined tables."""
    g = gts[0].g
    accs = g.g.accessions
    r = _refine_scores(g, batch, [gt.inputs for gt in gts], prepared, tops, gts[0]._skip_db_hets)
    fine = []
    for i, gt in enumerate(gts):
        m = int(r["m"][i])
        if m < 100:
            log.info("#positions in segregating sites are are too little: %s" % m)
        fine.append(genotyper_output(accs, r["score"][i], r["ninfo"][i], len(gt.inputs.pos), m, gt.inputs.dp, refine_mask(gt.result)))
    K = max(len(f.accs) for f in fine)
    sc, ni = np.zeros((len(fine), K)), np.zeros((len(fine), K))
    for i, f in enumerate(fine):
        sc[i, :len(f.accs)], ni[i, :len(f.accs)] = f.scores, f.ninfo
    prob, lik, lrt = lib.calculate_likelihoods_many(sc, ni)
    for i, (gt, f) in enumerate(zip(gts, fine)):
        k = len(f.accs)
        f._attach_fused(prob[i, :k], lik[i, :k], lrt[i, :k])
        gt.result_fine = f
        f.print_out_table(gt.outFile + ".refined.scores.txt")


def _refine_scores(g, batch, samples, prepared, tops, skip_db_hets):
    """Device part of the refine pass: the samples in position order with f64 weights, each scored over the pairs whose row
    segregates among its top hits `tops[i]`.  Returns Batch.fetch()."""
    offs = np.concatenate([[0], np.cumsum([len(p[2]) for p in prepared])]).astype(np.int64)
    batch.upload(offs, np.concatenate([p[1] for p in prepared]), np.concatenate([p[2] for p in prepared]),
                 _ordered_weights(samples, prepared))
    batch.set_segregation_filter(lib.selection_masks(tops, g.db.n_acc))
    try:
        # on one-hot weights the order-exact kernel gives the popcount kernel's integers: one launch serves every sample
        batch.run(skip_db_hets, kernel_mode=lib.KERNEL_FP64)
        batch.epilogue()
        return batch.fetch()
    finally:
        batch.set_segregation_filter(None)


def potatoGenotyperMany(args, samples):
    """`inbred --samples`: samples = [(input file, output prefix)].  Exits with status 1, after every other sample is written,
    when a sample had no top hit to refine."""
    inputs = [parsers.ParseInputs(inFile=path, logDebug=args['logDebug']) for path, _ in samples]
    log.info("packing the database into HBM")
    g = snp_genotype.Genotype(args['hdf5File'], args['hdf5accFile'])
    try:
        log.info("matching %d samples against %s accessions", len(samples), len(g.accessions))
        gts = inbred_identify_many(inputs, g, [prefix for _, prefix in samples], refine=args['refine'], skip_db_hets=args['skip_db_hets'])
    finally:
        g.close()
    skipped = [path for (path, _), gt in zip(samples, gts) if gt.no_top_hits]
    if skipped:
        die("no top hits to refine (no marker shared with the panel?): " + ", ".join(skipped))
    log.info("finished!")


def potatoGenotyperVcf(args, prefixes):
    """`inbred --samples_vcf`: every sample column of one VCF, parsed on the device (parsers.read_vcf_many), sample i written
    under prefixes[i].  Exits with status 1 on a sharded panel or a VCF the parser refuses, and, after every other sample is
    written, when a sample had no top hit to refine."""
    log.info("packing the database into HBM")
    g = snp_genotype.Genotype(args['hdf5File'], args['hdf5accFile'])
    try:
        if not holds_whole_panel(g):
            die("--samples_vcf needs the whole panel on one device; this one holds a shard of its rows")
        try:
            parsed = parsers.read_vcf_many(args['samples_vcf'], device=g.db.device)
        except ValueError as e:
            die(str(e))
        log.info("matching %d samples against %s accessions", len(parsed), len(g.accessions))
        gts = inbred_identify_many([inp for _, inp in parsed], g, prefixes, refine=args['refine'], skip_db_hets=args['skip_db_hets'])
    finally:
        g.close()
    skipped = [name for (name, _), gt in zip(parsed, gts) if gt.no_top_hits]
    if skipped:
        die("no top hits to refine (no marker shared with the panel?): " + ", ".join(skipped))
    log.info("finished!")


def pairwiseScore(inFile_1, inFile_2, logDebug, outFile=None, hdf5File=None, device=0):
    """`snpmatch pairsnp` (snpmatch.py:270-309): fraction of identical genotype strings among the markers two samples
    share, per chromosome and overall, optionally restricted to the positions of a database.  Both joins and the counting
    loop (snpmatch.py:291-297) run on the GPU; the returned dict has the reference's keys and values.  Unlike the reference
    under Python 3 (its json.dumps trips over numpy integers, snpmatch.py:307) the output file is written."""
    snpmatch_stats = {}
    log.info("parsing %s and %s", inFile_1, inFile_2)
    inputs_1 = parsers.ParseInputs(inFile=inFile_1, logDebug=logDebug)
    inputs_2 = parsers.ParseInputs(inFile=inFile_2, logDebug=logDebug)
    if hdf5File is not None:
        log.info("restricting sample 1 to the positions of the database")
        g = hdf5File if isinstance(hdf5File, snp_genotype.Genotype) else snp_genotype.Genotype(hdf5File, None, device=device)
        snpmatch_stats['hdf5'] = hdf5File if not isinstance(hdf5File, snp_genotype.Genotype) else "resident"
        commonSNPs_1 = g.get_positions_idxs(inputs_1.chrs, inputs_1.pos)
        common_inds = snp_genotype.Genotype.get_common_positions(inputs_1.chrs[commonSNPs_1[1]], inputs_1.pos[commonSNPs_1[1]],
                                                                 inputs_2.chrs, inputs_2.pos, device=device)
        common_inds = (commonSNPs_1[1][common_inds[0]], common_inds[1])
    else:
        log.info("joining the two samples on (chromosome, position)")
        common_inds = snp_genotype.Genotype.get_common_positions(inputs_1.chrs, inputs_1.pos, inputs_2.chrs, inputs_2.pos, device=device)
    log.info("done!")
    n1, n2 = len(inputs_1.chrs), len(inputs_2.chrs)
    unique_1 = n1 - len(common_inds[0])
    unique_2 = n2 - len(common_inds[0])
    inputs_1.filter_chr_names()
    inputs_2.filter_chr_names()
    common_chrs = np.intersect1d(inputs_1.g_chrs_ids, inputs_2.g_chrs_ids)
    # what crosses the C ABI: chromosome id (index into common_chrs, -1 elsewhere) of every marker of sample 1 and the ids
    # of the genotype strings in one table for both samples
    codes1, uniq1 = labels.factorize(inputs_1.g_chrs)
    in_common = {c: k for k, c in enumerate(common_chrs)}
    chrom1 = np.array([in_common.get(u, -1) for u in uniq1], dtype=np.int32)[codes1] if n1 else np.zeros(0, dtype=np.int32)
    gt_ids = labels.factorize(np.concatenate([inputs_1.gt.astype("U"), inputs_2.gt.astype("U")]))[0]
    common, scores = lib.pair_match_counts(common_inds[0], common_inds[1], chrom1, gt_ids[:n1], gt_ids[n1:], len(common_chrs), device=device)
    for k, i in enumerate(common_chrs):
        log.debug("chromosome %s: %s common markers, %s identical calls", i, int(common[k]), int(scores[k]))
        snpmatch_stats[str(i)] = [get_fraction(int(scores[k]), int(common[k])), int(common[k])]
    snpmatch_stats['matches'] = [get_fraction(int(np.sum(scores)), int(np.sum(common))), int(np.sum(common))]
    snpmatch_stats['unique'] = {"%s" % os.path.basename(inFile_1): [get_fraction(unique_1, n1), n1],
                                "%s" % os.path.basename(inFile_2): [get_fraction(unique_2, n2), n2]}
    if outFile:
        log.info("writing %s.matches.json", outFile)
        with open(outFile + ".matches.json", "w") as fh:
            json.dump(snpmatch_stats, fh, sort_keys=True, indent=4)
    return snpmatch_stats


# ---- pairsnp for many samples ----------------------------------------------------------------------------------------------
def _chromosome_codes(inp):
    """(raw names, codes into them, normalised names) of a sample's markers: every 'chr' deleted, any case (parsers.py:161)."""
    codes, raw = labels.factorize(np.asarray(inp.chrs))
    norm = np.array([snp_genotype._CHR_RE.sub("", str(u)) for u in raw], dtype="str") if len(raw) else np.zeros(0, dtype="U1")
    return raw, codes, norm


def _no_repeats(cid, pos, n_names):
    """True when no (chromosome, position) repeats: the common case (one run per chromosome, ascending positions) in O(n)."""
    if len(cid) < 2:
        return True
    run = cid[1:] == cid[:-1]
    if np.count_nonzero(~run) + 1 == n_names and bool(np.all(pos[1:][run] > pos[:-1][run])):
        return True
    key = np.sort((cid.astype(np.int64) << 32) | (pos + 2**31))
    return not bool(np.any(key[1:] == key[:-1]))


def gt_classes(gts):
    """Class of every GT string (equal strings, equal classes) and the distinct strings, for the concatenated calls of all
    samples.  Strings of up to three characters are compared as one integer each (21 bits per character)."""
    gts = np.asarray(gts)
    if gts.dtype.kind != "U":
        gts = gts.astype("U")
    if len(gts) and gts.dtype.itemsize <= 12:
        v = np.ascontiguousarray(gts).view(np.uint32).reshape(len(gts), -1)
        key = v[:, 0].astype(np.uint64)
        for k in range(1, v.shape[1]):
            key |= v[:, k].astype(np.uint64) << np.uint64(21 * k)
        codes, uniq = pd.factorize(key)
        first = np.full(len(uniq), len(gts), np.int64)
        np.minimum.at(first, codes, np.arange(len(gts)))
        return codes.astype(np.int64), gts[first]
    return labels.factorize(gts)


def build_pair_columns(keys, counts, cls, device, restrict=None):
    """The union of all samples' markers and each marker's column in it, sorted on `device` (a torch device).
    keys int64[n] = chromosome index << 32 | (position + 2^31), sample after sample (counts[s] markers each, no key twice in a
    sample); cls uint8[n] the marker's GT-string class.  restrict(union keys) -> bool mask keeps only those columns (the
    positions of a database).  Returns (offsets int64[S+1], col int32[m], cls uint8[m], union keys int64[K]) with every
    sample's markers in column order; columns are ordered by (chromosome, position)."""
    import torch
    counts = np.asarray(counts, dtype=np.int64)
    kt = torch.as_tensor(np.ascontiguousarray(keys, dtype=np.int64)).to(device)
    ct = torch.as_tensor(np.ascontiguousarray(cls, dtype=np.uint8)).to(device)
    sample = torch.repeat_interleave(torch.arange(len(counts), device=device), torch.as_tensor(counts).to(device))
    uniq, inv = torch.unique(kt, sorted=True, return_inverse=True)
    if restrict is not None:
        keep_col = torch.as_tensor(np.ascontiguousarray(restrict(uniq.cpu().numpy()), dtype=bool)).to(device)
        keep = keep_col[inv]
        inv = (torch.cumsum(keep_col.to(torch.int64), 0) - 1)[inv[keep]]
        sample, ct, uniq = sample[keep], ct[keep], uniq[keep_col]
    K = len(uniq)
    order = torch.argsort(sample * max(K, 1) + inv)
    col = inv[order].to(torch.int32)
    offsets = np.zeros(len(counts) + 1, np.int64)
    offsets[1:] = np.cumsum(torch.bincount(sample, minlength=len(counts)).cpu().numpy())
    return offsets, col.cpu().numpy(), ct[order].cpu().numpy(), uniq.cpu().numpy()


class PairMatrix(object):
    """Result of pairwise_score_many: common / same int64 [C,S,S] = per normalised chromosome (`chromosomes`) the markers
    samples i and j share and how many of those carry identical GT strings."""

    def __init__(self, common, same, chromosomes, chr_ids, n_markers, names, hdf5=None):
        self.common, self.same = common, same
        self.chromosomes = chromosomes
        self._chr_ids = chr_ids              # per sample: sorted indices into `chromosomes` of its g_chrs_ids
        self.n_markers = n_markers
        self.names = names
        self.hdf5 = hdf5
        self.timings = {}

    def identity(self):
        """[S,S] same / common over all chromosomes, nan where the pair shares no marker."""
        c, s = self.common.sum(axis=0), self.same.sum(axis=0)
        with np.errstate(invalid="ignore", divide="ignore"):
            return np.where(c > 0, s / np.maximum(c, 1), np.nan)

    def stats(self, i, j):
        """The dict pairwiseScore(names[i], names[j], ..., hdf5File) returns."""
        d = {}
        if self.hdf5 is not None:
            d['hdf5'] = self.hdf5
        for c in np.intersect1d(self._chr_ids[i], self._chr_ids[j]):
            n = int(self.common[c, i, j])
            d[str(self.chromosomes[c])] = [get_fraction(int(self.same[c, i, j]), n), n]
        tc, ts = int(self.common[:, i, j].sum()), int(self.same[:, i, j].sum())
        d['matches'] = [get_fraction(ts, tc), tc]
        ni, nj = int(self.n_markers[i]), int(self.n_markers[j])
        d['unique'] = {"%s" % os.path.basename(self.names[i]): [get_fraction(ni - tc, ni), ni],
                       "%s" % os.path.basename(self.names[j]): [get_fraction(nj - tc, nj), nj]}
        return d

    def write(self, prefix, pairs_json=False, labels=None):
        """<prefix>.identity.tsv and <prefix>.common.tsv (S x S, the sample labels as header row and first column; labels
        default to the names' basenames) and, with pairs_json, <prefix>.pairs.jsonl: one line per pair i < j,
        {"sample_1", "sample_2", "stats": stats(i, j)}."""
        import time
        t0 = time.perf_counter()
        labels = [os.path.basename(n) for n in self.names] if labels is None else [str(x) for x in labels]
        check_labels(labels, len(self.names))
        write_matrix_tsv(prefix + ".identity.tsv", labels, self.identity())
        write_matrix_tsv(prefix + ".common.tsv", labels, self.common.sum(axis=0))
        if pairs_json:
            with open(prefix + ".pairs.jsonl", "w") as fh:
                S = len(self.names)
                for i in range(S):
                    for j in range(i + 1, S):
                        fh.write(json.dumps({"sample_1": self.names[i], "sample_2": self.names[j], "stats": self.stats(i, j)},
                                            sort_keys=True) + "\n")
        self.timings["write"] = time.perf_counter() - t0


def check_labels(labels, n):
    """Labels of the TSV header: one per sample, distinct, without tabs or line breaks."""
    if len(labels) != n:
        raise ValueError("%d labels for %d samples" % (len(labels), n))
    seen = {}
    for i, lab in enumerate(labels):
        if "\t" in lab or "\n" in lab or "\r" in lab or not lab:
            raise ValueError("sample %d: label %r is empty or holds a tab or line break" % (i, lab))
        if lab in seen:
            raise ValueError("samples %d and %d have the same label %s" % (seen[lab], i, lab))
        seen[lab] = i


def write_matrix_tsv(path, labels, matrix):
    """S x S matrix as TSV: header 'sample' + labels, then per row its label and the values (floats round-trip, nan as nan)."""
    with open(path, "w") as fh:
        fh.write("\t".join(["sample"] + list(labels)) + "\n")
        for lab, row in zip(labels, matrix):
            fh.write(lab + "\t" + "\t".join(map(str, row.tolist())) + "\n")


def pairwise_score_many(samples, hdf5File=None, device=0, names=None, chunk_markers=0, logDebug=False):
    """`pairsnp` for every pair of many samples in one device pass.  samples: sample files (VCF/BED/npz) or ParseInputs;
    names: what stands for each sample in stats() (default: its path, or sample<i> for a ParseInputs).  For every pair,
    PairMatrix.stats(i, j) is the dict pairwiseScore(names[i], names[j], ..., hdf5File) returns.
    Markers join on (normalised chromosome, position); with a database (path or Genotype, loaded once) only its positions
    count.  The columns are the union of all samples' markers, built by a device sort; the counts of all pairs come from
    lib.pair_matrix (one-hot tensor-core GEMMs over that union).  Refused before any device work: an empty list, more than
    lib.PAIR_MAX_SAMPLES samples, a sample with a repeated (chromosome, position), a position outside int32, and more than 8
    distinct GT strings.  `timings` of the result holds the host seconds of every stage and the library's device times."""
    import time
    t0 = time.perf_counter()
    samples = list(samples)
    if not samples:
        raise ValueError("pairwise_score_many: the sample list is empty")
    if len(samples) > lib.PAIR_MAX_SAMPLES:
        raise ValueError("pairwise_score_many: %d samples; one call takes at most %d" % (len(samples), lib.PAIR_MAX_SAMPLES))
    names = [s if isinstance(s, str) else "sample%d" % i for i, s in enumerate(samples)] if names is None else [str(n) for n in names]
    assert len(names) == len(samples), "one name per sample"
    inputs = [parsers.ParseInputs(inFile=s, logDebug=logDebug) if isinstance(s, str) else s for s in samples]
    t1 = time.perf_counter()
    # chromosomes: every normalised name any sample has, sorted (the order of np.intersect1d in pairwiseScore)
    chr_codes = [_chromosome_codes(inp) for inp in inputs]
    chromosomes = np.unique(np.concatenate([n for _, _, n in chr_codes])) if any(len(n) for _, _, n in chr_codes) else np.zeros(0, "U1")
    rep = np.empty(len(chromosomes), dtype=object)           # one raw name per chromosome, for the database join
    keys, chr_ids = [], []
    for i, ((raw, codes, norm), inp) in enumerate(zip(chr_codes, inputs)):
        gid = np.searchsorted(chromosomes, norm).astype(np.int64)
        rep[gid] = raw
        chr_ids.append(np.unique(gid))
        cid = gid[codes] if len(codes) else np.zeros(0, np.int64)
        pos = np.asarray(inp.pos, dtype=np.int64)
        if len(cid) != len(pos):
            raise ValueError("sample %d (%s): %d chromosome names for %d positions" % (i, names[i], len(cid), len(pos)))
        bad = pos[(pos < -2**31) | (pos >= 2**31 - 1)]
        if len(bad):
            raise ValueError("sample %d (%s): position %d is outside the int32 range of the join" % (i, names[i], int(bad[0])))
        if not _no_repeats(cid, pos, len(chr_ids[-1])):
            key = np.sort((cid << 32) | (pos + 2**31))
            k = key[1:][key[1:] == key[:-1]][0]
            raise ValueError("sample %d (%s): marker %s:%d appears more than once; compare such a sample with `pairsnp -i -j`"
                             % (i, names[i], chromosomes[k >> 32], (k & 0xFFFFFFFF) - 2**31))
        keys.append((cid << 32) | (pos + 2**31))
    counts = np.array([len(k) for k in keys], dtype=np.int64)
    cls, strings = gt_classes(np.concatenate([np.asarray(inp.gt).astype("U") for inp in inputs]))
    if len(strings) > 8:
        raise ValueError("the samples hold %d distinct GT strings (%s); at most 8 are compared in one call"
                         % (len(strings), ", ".join(map(str, strings[:9]))))
    t2 = time.perf_counter()
    g, hdf5 = None, None
    if hdf5File is not None:
        g = hdf5File if isinstance(hdf5File, snp_genotype.Genotype) else snp_genotype.Genotype(hdf5File, None, device=device)
        hdf5 = hdf5File if not isinstance(hdf5File, snp_genotype.Genotype) else "resident"
    try:
        restrict = None
        if g is not None:
            def restrict(u):
                in_db = np.zeros(len(u), dtype=bool)
                if len(u):
                    in_db[g.get_positions_idxs(rep[u >> 32].astype("U"), (u & 0xFFFFFFFF) - 2**31)[1]] = True
                return in_db
        offsets, col, mcls, union = build_pair_columns(np.concatenate(keys), counts, cls.astype(np.uint8), "cuda:%d" % device, restrict)
    finally:
        if g is not None and g is not hdf5File:
            g.close()
    chr_start = np.searchsorted(union >> 32, np.arange(len(chromosomes) + 1)).astype(np.int64)
    t3 = time.perf_counter()
    common, same, ms = lib.pair_matrix(offsets, col, mcls, max(len(strings), 1), len(union), chr_start, chunk_markers, device=device)
    t4 = time.perf_counter()
    pm = PairMatrix(common.astype(np.int64), same.astype(np.int64), chromosomes, chr_ids, counts, names, hdf5)
    pm.n_columns, pm.n_classes = len(union), len(strings)
    pm.timings = {"parse": t1 - t0, "prepare": t2 - t1, "union": t3 - t2, "device": t4 - t3, "build": time.perf_counter() - t4,
                  "expand_ms": ms[0], "gemm_ms": ms[1], "device_ms": ms[2]}
    return pm


def pairwiseScoreMany(args, samples):
    """`pairsnp --samples`: samples = [(file, label)]; writes <-o>.identity.tsv, <-o>.common.tsv and, with --pairs_json,
    <-o>.pairs.jsonl."""
    paths = [p for p, _ in samples]
    log.info("comparing %d samples, %d pairs", len(paths), len(paths) * (len(paths) - 1) // 2)
    pm = pairwise_score_many(paths, hdf5File=args['hdf5File'], names=paths, logDebug=args['logDebug'])
    log.info("writing %s.identity.tsv and %s.common.tsv", args['outFile'], args['outFile'])
    pm.write(args['outFile'], pairs_json=args.get('pairs_json', False), labels=[lab for _, lab in samples])
    return pm


# ---- accession against accession ------------------------------------------------------------------------------------------
class PanelIdentity(object):
    """Result of panel_identity: common / same int32 [n,n] over the selected accessions `accessions` (ids, in output order):
    the panel rows both accessions have called, and those of them with equal calls.  Symmetric; common[i, i] is the number
    of called rows of accession i."""

    def __init__(self, common, same, accessions, skip_db_hets=False):
        self.common, self.same = common, same
        self.accessions = accessions
        self.skip_db_hets = skip_db_hets
        self.timings = {}

    def identity(self):
        """[n,n] same / common, nan where the pair has no row both have called."""
        with np.errstate(invalid="ignore", divide="ignore"):
            return np.where(self.common > 0, self.same / np.maximum(self.common, 1), np.nan)

    def close_pairs(self, min_identity):
        """Pairs i < j with common > 0 and identity >= min_identity, most identical first (ties in (i, j) order):
        a list of (acc_1, acc_2, identity, common, same)."""
        n = len(self.accessions)
        ii, jj, idents = [], [], []
        step = max(1, (8 << 20) // max(n, 1))                   # rows at a time: the float matrix is never built whole
        for r0 in range(0, n, step):
            c = self.common[r0:r0 + step]
            with np.errstate(invalid="ignore", divide="ignore"):
                ident = self.same[r0:r0 + step] / np.maximum(c, 1)
            i, j = np.nonzero((c > 0) & (ident >= min_identity) & (np.arange(n)[None, :] > np.arange(r0, r0 + len(c))[:, None]))
            ii.append(i + r0)
            jj.append(j)
            idents.append(ident[i, j])
        ii, jj, idents = np.concatenate(ii), np.concatenate(jj), np.concatenate(idents)
        order = np.lexsort((jj, ii, -idents))
        return [(str(self.accessions[i]), str(self.accessions[j]), float(v), int(self.common[i, j]), int(self.same[i, j]))
                for i, j, v in zip(ii[order], jj[order], idents[order])]

    def write(self, prefix, min_identity=None):
        """<prefix>.identity.tsv and <prefix>.common.tsv (n x n, the accession ids as header row and first column, the layout
        of `pairsnp --samples`) and, with min_identity, <prefix>.close_pairs.tsv: acc_1, acc_2, identity, common, same of every
        close_pairs(min_identity) pair."""
        import time
        t0 = time.perf_counter()
        labels = [str(a) for a in self.accessions]
        check_labels(labels, len(labels))
        write_matrix_tsv(prefix + ".identity.tsv", labels, self.identity())
        write_matrix_tsv(prefix + ".common.tsv", labels, self.common)
        if min_identity is not None:
            with open(prefix + ".close_pairs.tsv", "w") as fh:
                fh.write("acc_1\tacc_2\tidentity\tcommon\tsame\n")
                for a, b, v, c, s in self.close_pairs(min_identity):
                    fh.write("%s\t%s\t%s\t%d\t%d\n" % (a, b, str(v), c, s))
        self.timings["write"] = time.perf_counter() - t0


def accession_indices(g, accessions):
    """Panel indices of the accession ids `accessions` (output order); None = every accession in panel order.  Raises
    ValueError naming an id the panel lacks or one listed twice."""
    ids = np.asarray(g.accessions).astype("U")
    if accessions is None:
        return np.arange(len(ids), dtype=np.int32)
    index = {a: k for k, a in enumerate(ids.tolist())}
    seen = {}
    out = np.empty(len(accessions), dtype=np.int32)
    for k, a in enumerate(str(x) for x in accessions):
        if a in seen:
            raise ValueError("accession %s is listed twice (entries %d and %d)" % (a, seen[a], k))
        if a not in index:
            raise ValueError("accession %s is not in the database" % a)
        seen[a] = k
        out[k] = index[a]
    if not len(out):
        raise ValueError("the accession list is empty")
    return out


def panel_identity(g, accessions=None, skip_db_hets=False, chunk_rows=0, block_acc=0):
    """Which accessions of a panel cannot be told apart: pairwiseScore's statistic for every pair of the accessions
    `accessions` (ids, in output order; default all) over every row of the resident panel g (a Genotype), in one tensor-core
    pass (lib.Database.acc_pairs).  "Called" is code 0, 1 or 2; skip_db_hets counts hets as missing; het equals het.
    Returns a PanelIdentity.  A Genotype holding a row shard is refused: its counts would cover part of the genome."""
    import time
    if g.db.row0_global != 0 or g.db.n_rows != int(np.max(getattr(g, "global_chr_regions", [[0, g.db.n_rows]]))):
        raise ValueError("panel_identity needs the whole panel on one device; this one holds a shard of its rows")
    idx = accession_indices(g, accessions)
    t0 = time.perf_counter()
    common, same, ms = g.db.acc_pairs(idx, skip_db_hets=skip_db_hets, chunk_rows=chunk_rows, block_acc=block_acc)
    res = PanelIdentity(common, same, np.asarray(g.accessions).astype("U")[idx], skip_db_hets=skip_db_hets)
    res.timings = {"device": time.perf_counter() - t0, "expand_ms": ms[0], "gemm_ms": ms[1], "device_ms": ms[2]}
    return res


def panelIdentity(args, accessions):
    """`pairsnp --accessions`: accessions = ids in output order or None (all); writes <-o>.identity.tsv, <-o>.common.tsv and,
    with --min_identity, <-o>.close_pairs.tsv.  Dies naming an id the database lacks."""
    g = snp_genotype.Genotype(args['hdf5File'], None)
    try:
        try:
            accession_indices(g, accessions)
        except ValueError as e:
            die(str(e))
        log.info("comparing %d accessions over %d rows", len(g.accessions) if accessions is None else len(accessions), g.g.num_snps)
        res = panel_identity(g, accessions, skip_db_hets=args.get('skip_db_hets', False))
    finally:
        g.close()
    log.info("writing %s.identity.tsv and %s.common.tsv", args['outFile'], args['outFile'])
    res.write(args['outFile'], min_identity=args.get('min_identity'))
    return res
