"""
`snpmatch cross` — host side of the windowed B200 matching path.

Mirrors `snpmatch/core/csmatch.py`: `CrossIdentifier` (csmatch.py:19-186) with `window_genotyper`
(:64-104), `get_window_data` (:44-61), `match_insilico_f1s` (:106-129), `cross_interpreter`
(:131-186) and `potatoCrossIdentifier` (:193-200).  The per-window join, scoring, likelihoods,
identity calls and the simulated-F1 reductions run on the GPU (csrc/windows.cuh, csrc/f1.cuh);
this file turns the device arrays into the reference's `windowscore.txt`, `scores.txt` and JSON
files.
"""
import itertools
import json
import logging

import numpy as np
import pandas as pd

from .. import lib
from . import genomes
from . import parsers
from . import snp_genotype
from . import snpmatch

log = logging.getLogger(__name__)
chunk_size = 1000

WINDOW_COLUMNS = ["acc", "snps_match", "snps_info", "score", "likelihood", "identical", "num_amb", "window_index"]


def _np_str(a):
    """Text NumPy gives a float column inside np.column_stack with a string column (csmatch.py:50)."""
    return np.asarray(a).astype("U32")


class CrossIdentifier(object):

    def __init__(self, inputs, g, genome_id, binLen, output_id="cross.identifier", run_identifier=True,
                 identity_error_rate=0.02, skip_db_hets=False):
        self.g = g
        assert type(inputs) is parsers.ParseInputs, "provide a parsers class"
        inputs.filter_chr_names()
        self.inputs = inputs
        self.genome = genomes.Genome(genome_id)
        self.binLen = binLen
        self.output_id = output_id
        self.error_rate = identity_error_rate
        self._skip_db_hets = skip_db_hets
        self._batch = None
        if run_identifier:
            self.cross_identifier()

    def cross_identifier(self):
        try:
            res = self.window_genotyper(self.output_id + '.windowscore.txt')
            self._write_scores_json(res)
            self.result = self.match_insilico_f1s(res, self.output_id + '.scores.txt')
            self.cross_interpreter(self.output_id + ".matches.json")
        finally:
            self._close_batch()

    def _write_scores_json(self, res):
        res.print_json_output(self.output_id + ".scores.txt.matches.json")
        snpmatch.getHeterozygosity(self.inputs.gt[res.matchedTarInd], self.output_id + ".scores.txt.matches.json")
        with open(self.output_id + ".scores.txt.matches.json") as json_out:
            self.cross_identfier_json = json.load(json_out)

    def _close_batch(self):
        if self._batch is not None:
            self._batch.close()
            self._batch = None

    @staticmethod
    def get_window_data(bin_inds, AccList, ScoreList, NumInfoSites, error_rate=0.02):
        """Rows of one window (csmatch.py:44-61) from host arrays — API-compatible entry point; the
        workflow itself gets the same quantities for all windows at once from the device."""
        AccList = np.asarray(AccList)
        ScoreList = np.asarray(ScoreList, dtype=np.float64)
        NumInfoSites = np.asarray(NumInfoSites)
        prob, lik, lrt = lib.calculate_likelihoods(ScoreList, NumInfoSites)
        identity = snpmatch.np_test_identity(ScoreList, NumInfoSites, error_rate=error_rate)
        with np.errstate(invalid="ignore"):
            amb = np.flatnonzero(lrt < snpmatch.lr_thres)
        return _window_frame(bin_inds, AccList, ScoreList, NumInfoSites, prob, lik, identity, len(amb), amb, len(AccList))

    def _check_genome(self):
        """The sample's chromosomes must name the genome's (the reference's assertions in get_bins_genome)."""
        uniq = np.unique(genomes.genome_style_ids(self.inputs.chrs))
        assert len(uniq) <= len(self.genome.chrs_ids), "Please change default --genome option"
        assert len(np.intersect1d(uniq, self.genome.chrs_ids)) > 0, "Please change default --genome option"

    def _window_markers(self):
        """The sample's markers as the windows upload wants them (genome-style chromosome ids, in window order) and the largest
        number of them one window can hold.  Records the marker order and whether the join orders them the same way."""
        g = self.g
        binLen = int(self.binLen)
        order, cid, pos = g.prepare_markers(self.inputs.chrs, self.inputs.pos, style="genome")
        wei = np.ascontiguousarray(np.asarray(self.inputs.wei, dtype=np.float64)[order])
        # identity table: a window cannot match more markers than the sample has in it
        n_max = int(np.bincount(np.maximum(cid, 0)).max()) if len(cid) else 0
        if len(pos):
            wkey = cid.astype(np.int64) * (1 << 32) + (np.maximum(pos.astype(np.int64), 1) - 1) // binLen
            n_max = int(np.unique(wkey, return_counts=True)[1].max())
        self._order = order
        self._join_style_same = np.array_equal(
            g.prepare_markers(self.inputs.chrs, self.inputs.pos, style="join")[1], cid)
        return cid, pos, wei, n_max

    def window_genotyper(self, out_file, mask_acc_ix=None):
        """All windows in one device pass (csmatch.py:64-104)."""
        g = self.g
        num_lines = len(g.accessions)
        if mask_acc_ix is not None:
            assert type(mask_acc_ix) is np.ndarray, "please provide numpy array of acc indices to be masked"
            keep = np.setdiff1d(np.arange(num_lines), mask_acc_ix)
        else:
            keep = np.arange(num_lines)
        binLen = int(self.binLen)
        win_count, win_off, n_windows, winds_chrs = self.genome.window_layout(g.g.chrs, binLen)
        self._check_genome()
        cid, pos, wei, n_max = self._window_markers()
        kmax = snpmatch.identity_kmax_table(n_max, self.error_rate)
        self._close_batch()
        batch = g.db.scratch_batch([0, len(pos)], cid, pos, wei)
        self._batch = batch
        batch.run_windows(self._skip_db_hets, binLen, win_count, win_off, n_windows, kmax, snpmatch.lr_thres)
        batch.epilogue()
        tot = batch.fetch()
        self.timings = batch.timings()
        masked = mask_acc_ix is not None
        if masked:                                       # likelihoods over the kept accessions only: from the full window arrays
            w = batch.fetch_windows()
        else:                                            # the surviving rows of all windows, compacted on the device
            w = batch.fetch_window_rows()
        return self._assemble_windows(out_file, {k: v[0] for k, v in tot.items()}, w, winds_chrs, keep if masked else None)

    def _assemble_windows(self, out_file, tot, w, winds_chrs, keep=None):
        """Host half of window_genotyper for one sample: windowscore rows, GenotyperOutput, matchedTarInd, winds_chrs.
        tot: the sample's row of Batch.fetch(); w: its Batch.fetch_window_rows() (or, with `keep`, the masked accessions'
        complement, its Batch.fetch_windows()); matched_s_idx of w indexes the sample's own upload."""
        accs = self.g.accessions
        frames = []
        masked = keep is not None
        if masked:
            for wi in np.flatnonzero(w["nrows"] > 0):
                sc, ni = w["score"][wi][keep], w["ninfo"][wi][keep]
                frames.append(self.get_window_data(wi + 1, accs[keep], sc, ni, self.error_rate))
        else:
            keep = np.arange(len(accs))
            frames.append(_window_rows_frame(w, accs))
        frames = [f for f in frames if len(f)]
        self.windows_data = pd.concat(frames, ignore_index=True) if frames else pd.DataFrame(columns=WINDOW_COLUMNS)
        NumMatSNPs = int(tot["m"])
        overlap = snpmatch.get_fraction(NumMatSNPs, len(self.inputs.pos))
        result = snpmatch.GenotyperOutput(accs[keep], tot["score"][keep], tot["ninfo"][keep], overlap, NumMatSNPs,
                                          self.inputs.dp)
        if not masked:
            result._attach_fused(tot["prob"], tot["L"], tot["LR"])
        result.matchedTarInd = self._order[w["matched_s_idx"]]
        result.winds_chrs = winds_chrs
        if out_file is not None:
            self.windows_data.to_csv(out_file, sep="\t", index=False)
            return result
        return [self.windows_data, result]

    @staticmethod
    def _top_hits(snpmatch_result):
        assert type(snpmatch_result) is snpmatch.GenotyperOutput, "Please provide GenotyperOutput class as input"
        if not hasattr(snpmatch_result, 'probabilies'):
            snpmatch_result.get_probabilities()
        return np.argsort(-snpmatch_result.probabilies)[0:10]

    def match_insilico_f1s(self, snpmatch_result, out_file):
        """Simulated F1s of the ten most probable accessions (csmatch.py:106-129)."""
        TopHitAccs = self._top_hits(snpmatch_result)
        log.info("simulating F1s for top 10 accessions")
        g = self.g
        batch = self._batch
        own = False
        if batch is None or not getattr(self, "_join_style_same", False):
            order, cid, pos = g.prepare_markers(self.inputs.chrs, self.inputs.pos)
            wei = np.ascontiguousarray(np.asarray(self.inputs.wei, dtype=np.float64)[order])
            batch = lib.Batch(g.db, [0, len(pos)], cid, pos, wei)
            batch.run(False)
            own = True
        try:
            if len(TopHitAccs) >= 2:
                f_score, f_ninfo = batch.f1_pairs(TopHitAccs)
            else:
                f_score, f_ninfo = np.zeros(0), np.zeros(0, dtype=np.int64)
        finally:
            if own:
                batch.close()
        return self._append_f1s(snpmatch_result, TopHitAccs, f_score, f_ninfo, out_file)

    def _append_f1s(self, snpmatch_result, TopHitAccs, f_score, f_ninfo, out_file):
        """The F1 rows after the accessions' rows, and scores.txt."""
        g = self.g
        names = [g.accessions[i] + "x" + g.accessions[j] for i, j in itertools.combinations(TopHitAccs, 2)]
        snpmatch_result.scores = np.append(snpmatch_result.scores, f_score)
        snpmatch_result.ninfo = np.append(snpmatch_result.ninfo, f_ninfo)
        snpmatch_result.accs = np.append(snpmatch_result.accs, np.array(names, dtype="str"))
        if out_file is not None:
            snpmatch_result.print_out_table(out_file)
        return snpmatch_result

    def cross_interpreter(self, out_file):
        """Verdict on the window table (csmatch.py:131-186); writes only for interpretation case >= 3."""
        assert 'cross_identfier_json' in dir(self), "run cross identifier first!"
        assert 'windows_data' in dir(self), "run window genotyper first!"
        log.info("running cross interpreter!")
        js = self.cross_identfier_json
        if js['interpretation']['case'] < 3:
            return
        wd = self.windows_data
        acc = wd["acc"].to_numpy().astype("str")
        widx = wd["window_index"].to_numpy().astype(int)
        ident = wd["identical"].to_numpy().astype(float)
        namb = wd["num_amb"].to_numpy().astype(int)
        windows = np.unique(widx)
        win_ident = np.array([ident[widx == k].max() for k in windows]) if len(windows) else np.zeros(0)
        identical_wind = np.flatnonzero(win_ident == 1)     # positions in the sorted window list, as in the reference
        num_winds = len(windows)
        js['identical_windows'] = [snpmatch.get_fraction(len(identical_wind), num_winds), num_winds]
        homo_wind = np.intersect1d(widx[namb < 20], identical_wind)
        in_homo = np.isin(widx, homo_wind)
        h_names, h_counts = np.unique(acc[in_homo], return_counts=True)
        js['matches'] = [(str(h_names[i]), int(h_counts[i])) for i in np.argsort(-h_counts)]
        res = self.result
        topMatch = np.argsort(res.likelis)[0]
        is_f1_row = ~np.isin(res.accs, self.g.accessions)
        if is_f1_row[topMatch]:
            mother, father = res.accs[topMatch].split("x")[0], res.accs[topMatch].split("x")[1]
            js['interpretation'] = {'text': "Sample may be a F1! or a contamination!", 'case': 5}
            js['parents'] = {'mother': [mother, 1], 'father': [father, 1]}
            js['genotype_windows'] = {'chr_bins': None, 'coordinates': {'x': None, 'y': None}}
        else:
            c_names, c_counts = np.unique(acc[namb == 1], return_counts=True)
            if len(c_names) > 0:
                top2 = np.argsort(-c_counts)[0:2]
                parents = c_names[top2].astype("str")
                counts = c_counts[top2].astype("int")
                xdict = np.array(windows, dtype="int")
                ydict = np.repeat("NA", len(xdict)).astype("S25")
                if len(parents) == 1:
                    js['interpretation'] = {'text': "Sample may be a F2! but only one parent found!", 'case': 6}
                    js['parents'] = {'mother': [parents[0], counts[0]], 'father': ["NA", "NA"]}
                    ydict[np.isin(xdict, widx[(acc == parents[0]) & in_homo])] = parents[0]
                    chr_bins = None
                else:
                    js['interpretation'] = {'text': "Sample may be a F2!", 'case': 6}
                    js['parents'] = {'mother': [parents[0], counts[0]], 'father': [parents[1], counts[1]]}
                    n_names, n_counts = np.unique(res.winds_chrs, return_counts=True)
                    chr_bins = dict((n_names[i], n_counts[i]) for i in range(len(n_names)))
                    ydict[np.isin(xdict, widx[(acc == parents[0]) & in_homo])] = parents[0]
                    ydict[np.isin(xdict, widx[(acc == parents[1]) & in_homo])] = parents[1]
                js['genotype_windows'] = {'chr_bins': chr_bins, 'coordinates': {'x': xdict.tolist(), 'y': ydict.tolist()}}
            else:
                js['interpretation'] = {'case': 7, 'text': "Sample may just be contamination!"}
                js['genotype_windows'] = {'chr_bins': None, 'coordinates': {'x': None, 'y': None}}
                js['parents'] = {'mother': [None, 0], 'father': [None, 1]}
        with open(out_file, "w") as out_stats:
            out_stats.write(json.dumps(js, sort_keys=True, indent=4, default=convert_int64))


# Device memory the window buffers of one launch may take.  Per sample, window and accession the buffers hold the partial score
# and informative sites over the padded panel row (12 bytes per padded column), the likelihood, ratio and identity call, and the
# compacted row arrays (42 bytes per accession): ~25 MB per sample at 1135 accessions x 399 windows, ~17x that at 20 000.
WINDOW_BUDGET_BYTES = 8 << 30


def window_bytes_per_sample(n_windows, n_acc, row_words):
    return int(n_windows) * (12 * 32 * int(row_words) + 42 * int(n_acc))


def cross_identify_many(inputs_list, g, genome_id, binLen, output_ids, skip_db_hets=False, identity_error_rate=0.02,
                        samples_per_launch=None):
    """`cross` for many samples: every sample's windows, totals and simulated F1s come out of one multi-sample batch per launch
    (one upload, one windows run, one F1 pass), and every sample's results and files (<output_ids[i]>.windowscore.txt,
    .scores.txt, .scores.txt.matches.json, .matches.json for case >= 3) are the ones CrossIdentifier gives for it alone.
    Launches hold as many samples as fit WINDOW_BUDGET_BYTES of window buffers (`samples_per_launch` overrides).  Every sample
    is checked against the genome before any device work.  Returns one CrossIdentifier per sample."""
    inputs_list, output_ids = list(inputs_list), list(output_ids)
    assert len(inputs_list) == len(output_ids), "one output prefix per sample"
    assert len(set(output_ids)) == len(output_ids), "output prefixes must differ"
    cis = [CrossIdentifier(inp, g, genome_id, binLen, out, run_identifier=False, identity_error_rate=identity_error_rate,
                           skip_db_hets=skip_db_hets) for inp, out in zip(inputs_list, output_ids)]
    for i, ci in enumerate(cis):
        try:
            ci._check_genome()
        except AssertionError as e:
            raise AssertionError("sample %d (%s): %s" % (i, output_ids[i], e))
    if not cis:
        return cis
    layout = cis[0].genome.window_layout(g.g.chrs, int(binLen))
    per = samples_per_launch
    if per is None:
        per = max(1, WINDOW_BUDGET_BYTES // max(window_bytes_per_sample(layout[2], g.db.n_acc, g.db.row_words), 1))
    assert int(per) >= 1, "samples_per_launch must be at least 1"
    # one batch lives with the panel: its device buffers are allocated once, not per call (cudaMalloc of a fresh batch costs
    # 0.3 - 1 s on a loaded device)
    if getattr(g, "_cross_batch", None) is None:
        g._cross_batch = lib.Batch(g.db, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3)))
    for c0 in range(0, len(cis), int(per)):
        _cross_launch(cis[c0:c0 + int(per)], g._cross_batch, layout)
    return cis


def _cross_launch(cis, batch, layout):
    """One multi-sample pass of `cross`: windows of all samples, then every sample's files from its slice."""
    g = cis[0].g
    binLen = int(cis[0].binLen)
    win_count, win_off, n_windows, winds_chrs = layout
    marks = [ci._window_markers() for ci in cis]
    offs = np.concatenate([[0], np.cumsum([len(m[1]) for m in marks])]).astype(np.int64)
    batch.upload(offs, np.concatenate([m[0] for m in marks]), np.concatenate([m[1] for m in marks]),
                 np.concatenate([m[2].reshape(-1, 3) for m in marks]))
    # kmax[n] does not depend on the table's length: one table for the largest window of the batch
    kmax = snpmatch.identity_kmax_table(max(m[3] for m in marks), cis[0].error_rate)
    batch.run_windows(cis[0]._skip_db_hets, binLen, win_count, win_off, n_windows, kmax, snpmatch.lr_thres)
    batch.epilogue()
    tot = batch.fetch()
    rows = batch.fetch_window_rows()
    if len(cis) == 1:
        rows = [rows]
    results = []
    for i, ci in enumerate(cis):
        w = dict(rows[i], matched_s_idx=rows[i]["matched_s_idx"] - offs[i])
        res = ci._assemble_windows(ci.output_id + '.windowscore.txt', {k: v[i] for k, v in tot.items()}, w, winds_chrs)
        ci._write_scores_json(res)
        results.append(res)
    log.info("simulating F1s for top 10 accessions")
    tops = np.stack([CrossIdentifier._top_hits(r) for r in results])
    k = tops.shape[1]
    f_score, f_ninfo = np.zeros((len(cis), k * (k - 1) // 2)), np.zeros((len(cis), k * (k - 1) // 2), dtype=np.int64)
    if k >= 2:
        f_score, f_ninfo = batch.f1_pairs(tops)
        # samples whose join order differs from their window order: the F1 pass runs on their markers in join order, as
        # CrossIdentifier.match_insilico_f1s does
        redo = [i for i, ci in enumerate(cis) if not ci._join_style_same]
        if redo:
            prep = [g.prepare_markers(cis[i].inputs.chrs, cis[i].inputs.pos) for i in redo]
            j_offs = np.concatenate([[0], np.cumsum([len(p[2]) for p in prep])]).astype(np.int64)
            j_wei = np.concatenate([np.asarray(cis[i].inputs.wei, dtype=np.float64).reshape(-1, 3)[p[0]] for i, p in zip(redo, prep)])
            jb = lib.Batch(g.db, j_offs, np.concatenate([p[1] for p in prep]), np.concatenate([p[2] for p in prep]), j_wei)
            try:
                jb.run(False)
                f_score[redo], f_ninfo[redo] = jb.f1_pairs(tops[redo])
            finally:
                jb.close()
    for i, ci in enumerate(cis):
        ci.result = ci._append_f1s(results[i], tops[i], f_score[i], f_ninfo[i], ci.output_id + '.scores.txt')
        ci.cross_interpreter(ci.output_id + ".matches.json")


def _window_frame(bin_inds, accs, score, ninfo, prob, lik, identity, num_amb, amb_rows, num_lines):
    """DataFrame rows of one window: only accessions with LR < lr_thres, and only when at least one
    but not all accessions pass (csmatch.py:57-60).  `score` and `likelihood` are text, as produced by
    the reference's np.column_stack with the accession names (csmatch.py:50)."""
    if not (1 <= num_amb < num_lines):
        return pd.DataFrame(columns=WINDOW_COLUMNS)
    k = np.asarray(amb_rows)
    sc = np.asarray(score, dtype=np.float64)[k]
    frame = pd.DataFrame({
        "acc": np.asarray(accs)[k].astype(str),
        "snps_match": np.array([int(float(s)) for s in _np_str(sc)], dtype=int),
        "snps_info": np.asarray(ninfo)[k].astype(int),
        "score": _np_str(np.asarray(prob, dtype=np.float64)[k]),
        "likelihood": _np_str(np.asarray(lik, dtype=np.float64)[k]),
        "identical": np.asarray(identity)[k].astype(float),
    })
    frame["num_amb"] = int(num_amb)
    frame["window_index"] = int(bin_inds)
    return frame[WINDOW_COLUMNS]


def _window_rows_frame(w, accs):
    """All rows of windowscore.txt at once from the device-compacted rows (Batch.fetch_window_rows): the same columns and
    the same text for `score` / `likelihood` as _window_frame builds window by window."""
    counts = np.diff(w["row_off"]).astype(np.int64)
    if counts.sum() == 0:
        return pd.DataFrame(columns=WINDOW_COLUMNS)
    sc = w["score"]
    ni = w["ninfo"]
    with np.errstate(invalid="ignore", divide="ignore"):
        prob = np.where(ni > 0, sc / ni, np.nan)
    frame = pd.DataFrame({
        "acc": np.asarray(accs)[w["acc"]].astype(str),
        "snps_match": np.array([int(float(x)) for x in _np_str(sc)], dtype=int),
        "snps_info": ni.astype(int),
        "score": _np_str(prob),
        "likelihood": _np_str(w["L"]),
        "identical": w["identical"].astype(float),
        "num_amb": np.repeat(w["num_amb"].astype(int), counts),
        "window_index": np.repeat(np.arange(1, len(counts) + 1, dtype=int), counts),
    })
    return frame[WINDOW_COLUMNS]


def convert_int64(o):
    """json `default` hook of the reference (csmatch.py:188-191): NumPy integers become ints; anything
    else it is asked about (the byte strings of `ydict`) falls through to None, i.e. JSON null."""
    if isinstance(o, np.integer):
        return int(o)


def potatoCrossIdentifier(args):
    inputs = parsers.ParseInputs(inFile=args['inFile'], logDebug=args['logDebug'])
    log.info("loading genotype files!")
    g = snp_genotype.Genotype(args['hdf5File'], args['hdf5accFile'])
    log.info("running cross identifier!")
    CrossIdentifier(inputs, g, args['genome'], args['binLen'], args['outFile'], run_identifier=True,
                    skip_db_hets=args['skip_db_hets'])
    log.info("finished!")


def potatoCrossIdentifierMany(args, samples):
    """`cross --samples`: samples = [(input file, output prefix)]."""
    inputs = [parsers.ParseInputs(inFile=path, logDebug=args['logDebug']) for path, _ in samples]
    log.info("loading genotype files!")
    g = snp_genotype.Genotype(args['hdf5File'], args['hdf5accFile'])
    try:
        log.info("running cross identifier on %d samples!" % len(samples))
        cross_identify_many(inputs, g, args['genome'], args['binLen'], [prefix for _, prefix in samples],
                            skip_db_hets=args['skip_db_hets'])
    finally:
        g.close()
    log.info("finished!")
