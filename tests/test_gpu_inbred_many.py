"""`inbred` for many samples (snpmatch.inbred_identify_many, `inbred --samples`) and the device pieces under it: the per-sample
segregation filter of a batch (Batch.set_segregation_filter, k_segregating_pairs), the heterozygous-pair count and the likelihoods
of many refined tables in one call.  Every sample's files equal the ones Genotyper (+ filter_tophits) writes for it alone, byte
for byte."""
import os

import numpy as np
import pytest

from oracle import snpmatch_oracle as orc
from snpmatch_b200 import synth

FILES = (".scores.txt", ".matches.json", ".refined.scores.txt")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


def _cluster_panel(n_rows=8000, n_acc=40, frac=0.004, seed=77):
    """A synthetic panel with clusters of near-duplicate accessions: 1 copies 0, 11-12 copy 10 and 21-24 copy 20, each with
    about 0.4 % of its calls flipped between ref and alt."""
    p = synth.small_panel(n_rows=n_rows, n_acc=n_acc)
    snps = p["snps"].copy()
    rng = np.random.default_rng(seed)
    for lead, size in ((0, 2), (10, 3), (20, 5)):
        for k in range(1, size):
            col = snps[:, lead].copy()
            d = rng.random(n_rows) < frac
            col[d] = np.where(col[d] == 0, 1, 0)
            snps[:, lead + k] = col
    p["snps"] = snps
    return p


@pytest.fixture(scope="module")
def cluster_panel():
    return _cluster_panel()


@pytest.fixture(scope="module")
def cluster_geno(lib, cluster_panel):
    from snpmatch_b200.core import snp_genotype
    p = cluster_panel
    g = snp_genotype.Genotype.from_arrays(p["snps"], p["positions"], p["chrs"], p["chr_regions"], p["accessions"])
    yield g
    g.close()


_PANELS = {}


def _synthetic(n_rows, n_acc):
    if (n_rows, n_acc) not in _PANELS:
        _PANELS[(n_rows, n_acc)] = synth.small_panel(n_rows=n_rows, n_acc=n_acc)
    return _PANELS[(n_rows, n_acc)]


def _db(lib, p):
    db = lib.Database(p["positions"], p["chr_regions"], p["snps"].shape[1])
    db.load_int8(p["snps"])
    return db


# ---- the segregation filter against a row filter of each sample's segregating rows ------------------------------------------
def _selections(n_acc, rng):
    """Selections that differ within a batch: none, one, two in different words, the last word's last accessions, a few
    spread over several words, and half of the panel."""
    return [rng.choice(n_acc, size=3, replace=False), np.array([], dtype=np.int64), np.array([n_acc // 2]),
            np.array([1, n_acc - 1]), np.array([n_acc - 2, n_acc - 1]), rng.choice(n_acc, size=min(7, n_acc), replace=False),
            rng.choice(n_acc, size=n_acc // 2, replace=False), np.array([0, 5])]


def _samples(p, n_acc, k, rng, hard=False):
    out = []
    for i in range(k):
        if i == 2:                     # an empty sample between two others
            out.append((np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3))))
            continue
        s = synth.make_sample_fast(p["positions"], p["chr_regions"], n_acc, true_acc=int(rng.integers(n_acc)),
                                   n_db=int(min(len(p["positions"]), 2500 + 700 * i)), n_extra=200, seed=300 + i)
        out.append((s["chr_ix"], s["pos"], synth.hard_weights(s["code"]) if hard else s["wei"]))
    return out


def _check_filter(lib, db, samples, sels, mode, row_filter=None):
    offs = np.concatenate([[0], np.cumsum([len(s[1]) for s in samples])]).astype(np.int64)
    b = lib.Batch(db, offs, np.concatenate([s[0] for s in samples]), np.concatenate([s[1] for s in samples]),
                  np.concatenate([s[2] for s in samples]))
    one = lib.Batch(db, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3)))
    try:
        if row_filter is not None:
            b.set_row_filter(row_filter)
        b.set_segregation_filter(lib.selection_masks(sels, db.n_acc))
        b.run(False, kernel_mode=mode)
        b.epilogue()
        r = b.fetch()
        kept = 0
        for s, (cid, pos, wei) in enumerate(samples):
            rows = db.segregating_rows(np.asarray(sels[s], dtype=np.int32))
            if row_filter is not None:
                rows = np.intersect1d(rows, row_filter)
            one.upload([0, len(pos)], cid, pos, wei)
            one.set_row_filter(rows)
            one.run(False, kernel_mode=mode)
            one.epilogue()
            o = one.fetch()
            got, want = b.fetch_pairs(s), one.fetch_pairs(0)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), s
            assert int(r["m"][s]) == int(o["m"][0]) == len(want[0])
            assert np.array_equal(r["score"][s], o["score"][0]), s          # mode 0: same pairs, same chunks, same bits
            assert np.array_equal(r["matches"][s], o["matches"][0]) and np.array_equal(r["ninfo"][s], o["ninfo"][0])
            if len(sels[s]) < 2:
                assert int(r["m"][s]) == 0
            kept += int(r["m"][s])
        assert kept > 0
    finally:
        b.close()
        one.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_acc,n_rows", [(40, None), (1135, 30000), (2100, 20000)])
@pytest.mark.parametrize("mode", [0, 1])
def test_segregation_filter_equals_row_filter(lib, small_panel, n_acc, n_rows, mode):
    rng = np.random.default_rng(n_acc + mode)
    p = small_panel if n_rows is None else _synthetic(n_rows, n_acc)
    db = _db(lib, p)
    try:
        assert db.row_words == 2 * ((n_acc + 63) // 64)
        sels = _selections(n_acc, rng)
        samples = _samples(p, n_acc, len(sels), rng, hard=mode == 1)
        _check_filter(lib, db, samples, sels, mode)
        # AND with a row filter
        _check_filter(lib, db, samples, sels, mode, row_filter=np.flatnonzero(rng.random(len(p["positions"])) < 0.6))
    finally:
        db.close()


@pytest.mark.gpu
def test_segregation_filter_errors_and_clearing(lib, small_panel, sample_inbred):
    p = small_panel
    db = _db(lib, p)
    s = synth.make_sample_fast(p["positions"], p["chr_regions"], 40, true_acc=7, n_db=3000, n_extra=100, seed=11)
    n = len(s["pos"])
    b = lib.Batch(db, [0, n, 2 * n], np.tile(s["chr_ix"], 2), np.tile(s["pos"], 2), np.tile(s["wei"], (2, 1)))
    try:
        b.run(False)
        b.epilogue()
        plain = b.fetch()
        sel = lib.selection_masks([[3, 7], [1, 2, 30]], 40)
        with pytest.raises(lib.SnpmError) as e:                       # rows of the wrong width
            b.set_segregation_filter(np.zeros((2, 4), np.uint32))
        assert e.value.code == lib.SNPM_E_ARG
        bad = sel.copy()
        bad[0, 1] |= np.uint32(1 << 8)                                 # accession 40 of a 40-accession panel
        with pytest.raises(lib.SnpmError) as e:
            b.set_segregation_filter(bad)
        assert e.value.code == lib.SNPM_E_ARG
        b.set_segregation_filter(sel[:1])                              # one selection for two samples: refused at run time
        with pytest.raises(lib.SnpmError) as e:
            b.run(False)
        assert e.value.code == lib.SNPM_E_ARG
        b.set_segregation_filter(sel)
        b.run(False)
        b.epilogue()
        filt = b.fetch()
        assert (filt["m"] < plain["m"]).all()
        # every other run form refuses a batch with the filter set
        from snpmatch_b200.core import snpmatch
        kmax = snpmatch.identity_kmax_table(5000, 0.02)
        cnt, off = np.array([40] * 5, np.int32), np.arange(0, 200, 40, dtype=np.int32)
        with pytest.raises(lib.SnpmError) as e:
            b.run_windows(False, 300000, cnt, off, 200, kmax)
        assert e.value.code == lib.SNPM_E_STATE
        b.set_segregation_filter(sel[:1])
        b.upload([0, n], s["chr_ix"], s["pos"], s["wei"])
        with pytest.raises(lib.SnpmError) as e:
            b.run_windows_begin(False, 300000, cnt, off, 200, kmax)
        assert e.value.code == lib.SNPM_E_STATE
        cs = lib.code_markers(np.array([0, n]), s["chr_ix"], s["pos"], s["wei"])
        b.upload_coded(cs)
        with pytest.raises(lib.SnpmError) as e:
            b.run(False, kernel_mode=lib.KERNEL_GROUPED)
        assert e.value.code == lib.SNPM_E_STATE
        # cleared: the plain results again
        b.set_segregation_filter(None)
        b.upload([0, n, 2 * n], np.tile(s["chr_ix"], 2), np.tile(s["pos"], 2), np.tile(s["wei"], (2, 1)))
        b.run(False)
        b.epilogue()
        again = b.fetch()
        assert np.array_equal(again["score"], plain["score"]) and np.array_equal(again["m"], plain["m"])
    finally:
        b.close()
        db.close()


@pytest.mark.gpu
def test_count_flagged_pairs(lib, small_panel):
    p = small_panel
    db = _db(lib, p)
    rng = np.random.default_rng(3)
    samples = _samples(p, 40, 5, rng)
    offs = np.concatenate([[0], np.cumsum([len(s[1]) for s in samples])]).astype(np.int64)
    cid, pos = np.concatenate([s[0] for s in samples]), np.concatenate([s[1] for s in samples])
    flags = rng.random(len(pos)) < 0.3
    b = lib.Batch(db, offs, cid, pos, np.concatenate([s[2] for s in samples]))
    try:
        b.run(False)
        got = b.count_flagged_pairs(flags)
        for s in range(len(samples)):
            _, s_idx = b.fetch_pairs(s)
            assert got[s] == int(flags[offs[s] + s_idx].sum()), s
    finally:
        b.close()
        db.close()


@pytest.mark.gpu
def test_calculate_likelihoods_many_equals_rows(lib):
    rng = np.random.default_rng(9)
    K = 300
    lens = [K, 1, 17, 250, K, 40, K]
    sc, ni = np.zeros((len(lens), K)), np.zeros((len(lens), K))
    for i, k in enumerate(lens):
        n = rng.integers(0, 4000, size=k).astype(np.float64)
        y = np.floor(n * rng.uniform(0.2, 1.0, size=k))
        if i == 4:
            n[:] = 0.0                                       # every likelihood nan
            y[:] = 0.0
        if i == 5:
            n[:3], y[:3] = 4000.0, 4000.0                    # perfect matches: L = 1 exactly
            n[3:6], y[3:6] = 4000.0, 0.0                     # no match: L = nan
        if i == 6:
            n[::5] = 0.0
            y[::5] = 0.0
        sc[i, :k], ni[i, :k] = y, n
    prob, lik, lrt = lib.calculate_likelihoods_many(sc, ni)
    for i, k in enumerate(lens):
        p1, l1, r1 = lib.calculate_likelihoods(sc[i, :k], ni[i, :k])
        assert np.array_equal(prob[i, :k], p1, equal_nan=True)
        assert np.array_equal(lik[i, :k], l1, equal_nan=True)
        assert np.array_equal(lrt[i, :k], r1, equal_nan=True)
        assert np.isnan(lik[i, k:]).all()
    assert (lik[5, :3] == 1.0).all() and np.isnan(lik[5, 3:6]).all() and np.isnan(lrt[4]).all()
    with pytest.raises(AssertionError):
        bad = sc.copy()
        bad[2, 0] = ni[2, 0] + 1
        lib.calculate_likelihoods_many(bad, ni)


# ---- files identical to single runs ---------------------------------------------------------------------------------------
def _inputs(s, wei_key="wei"):
    from snpmatch_b200.core import parsers
    inp = parsers.ParseInputs("")
    inp.load_snp_info(s["chrs"], s["pos"], s["gt"], s[wei_key], s["dp"])
    return inp


def _subset(s, keep):
    return {k: (v[keep] if isinstance(v, np.ndarray) and v.ndim >= 1 and len(v) == len(s["pos"]) else v) for k, v in s.items()}


def _batch_samples(p):
    """(name, sample, weight key): samples that refine with different top-hit sets (2, 3 and 5 accessions), one with a unique
    hit, one with more than half of the panel in its top hits, one whose refine keeps no pair, one with more than 100 refined
    pairs, one with its markers shuffled and one that shares no marker with the panel; PL and called-genotype weights."""
    def mk(acc, n_db, seed):
        return synth.make_sample(p["positions"], p["chr_regions"], p["chrs"], 40, true_acc=acc, n_db=n_db, n_extra=50, seed=seed)
    shuffled = mk(10, 3000, 12)
    shuffled = _subset(shuffled, np.random.default_rng(4).permutation(len(shuffled["pos"])))
    nomatch = mk(30, 500, 13)
    nomatch["pos"] = nomatch["pos"] + 1
    keep = np.ones(len(nomatch["pos"]), bool)
    for c, (lo, hi) in enumerate(p["chr_regions"]):
        on = np.char.endswith(nomatch["chrs"].astype(str), str(p["chrs"][c]))
        keep &= ~(on & np.isin(nomatch["pos"], p["positions"][lo:hi]))
    nomatch = _subset(nomatch, keep)
    return [("pair", mk(0, 3000, 1), "wei"), ("trio", mk(10, 3000, 2), "wei_hard"), ("five", mk(20, 3000, 3), "wei"),
            ("five_big", mk(20, 7900, 7), "wei_hard"), ("unique", mk(30, 3000, 4), "wei"), ("tiny", mk(0, 8, 5), "wei"),
            ("half", mk(21, 600, 6), "wei_hard"), ("shuffled", shuffled, "wei"), ("nomatch", nomatch, "wei")]


def _same_files(a, b):
    for ext in FILES:
        assert os.path.exists(a + ext) == os.path.exists(b + ext), b + ext
        if os.path.exists(b + ext):
            assert open(a + ext, "rb").read() == open(b + ext, "rb").read(), b + ext


@pytest.mark.gpu
@pytest.mark.parametrize("refine", [False, True])
@pytest.mark.parametrize("skip", [False, True])
def test_batched_files_equal_single(lib, cluster_geno, cluster_panel, tmp_path, refine, skip):
    from snpmatch_b200.core import snpmatch
    p = cluster_panel
    samples = _batch_samples(p)
    many = snpmatch.inbred_identify_many([_inputs(s, k) for _, s, k in samples], cluster_geno,
                                         [str(tmp_path / ("many_" + n)) for n, _, _ in samples], refine=refine, skip_db_hets=skip)
    refined = {}
    for (name, s, key), gm in zip(samples, many):
        one = snpmatch.Genotyper(_inputs(s, key), cluster_geno, str(tmp_path / ("one_" + name)), run_genotyper=not refine,
                                 skip_db_hets=skip)
        if refine and name == "nomatch":
            with pytest.raises(AssertionError):
                one.filter_tophits()
        elif refine:
            one.filter_tophits()
        _same_files(str(tmp_path / ("many_" + name)), str(tmp_path / ("one_" + name)))
        assert np.array_equal(gm.result.scores, one.result.scores) and gm.num_matched == one.result.num_snps
        assert gm.no_top_hits == (refine and name == "nomatch")
        if hasattr(gm, "result_fine"):
            refined[name] = gm
            fine = one.result_fine
            assert np.array_equal(gm.result_fine.accs, fine.accs) and np.array_equal(gm.result_fine.scores, fine.scores)
            # the refined integers against the reference's own filter_pos_ix path, on the markers in (chromosome, position)
            # order: the join sorts a sample that is not (snp_genotype.order_markers), the reference's join assumes it is
            top = np.flatnonzero(gm.result.lrts < snpmatch.lr_thres)
            so = _subset(s, np.lexsort((s["pos"], s["chr_ix"])))
            ref = orc.genotyper(p["snps"], p["chrs"], p["chr_regions"], p["positions"], so["chrs"], so["pos"], so[key], skip_db_hets=skip,
                                filter_pos_ix=orc.segregating_rows(p["snps"], top))
            keep = np.setdiff1d(np.arange(40), snpmatch.refine_mask(gm.result))
            assert np.array_equal(gm.result_fine.scores, ref.score_f64[keep].astype(int))
            assert np.array_equal(gm.result_fine.ninfo, ref.ninfo[keep]) and gm.result_fine.num_snps == ref.num_snps
    if refine:
        assert set(refined) == {"pair", "trio", "five", "five_big", "tiny", "shuffled"}
        tops = {n: tuple(np.flatnonzero(g.result.lrts < 3.841)) for n, g in refined.items()}
        assert len({tops["pair"], tops["trio"], tops["five"]}) == 3
        assert refined["tiny"].result_fine.num_snps < 100 <= refined["five_big"].result_fine.num_snps
    else:
        assert not any(hasattr(g, "result_fine") for g in many)


@pytest.mark.gpu
def test_launch_splitting_gives_the_same_files(lib, cluster_geno, cluster_panel, tmp_path):
    from snpmatch_b200.core import snpmatch
    samples = _batch_samples(cluster_panel)
    for tag, per in (("d", None), ("one", 1), ("three", 3)):
        snpmatch.inbred_identify_many([_inputs(s, k) for _, s, k in samples], cluster_geno,
                                      [str(tmp_path / ("%s_%s" % (tag, n))) for n, _, _ in samples], refine=True, samples_per_launch=per)
    for n, _, _ in samples:
        _same_files(str(tmp_path / ("one_" + n)), str(tmp_path / ("d_" + n)))
        _same_files(str(tmp_path / ("three_" + n)), str(tmp_path / ("d_" + n)))


@pytest.mark.gpu
def test_sharded_panel_and_bad_names_are_refused(lib, cluster_panel):
    from snpmatch_b200.core import snp_genotype, snpmatch
    s = _batch_samples(cluster_panel)[0][1]
    g = snp_genotype.Genotype.synthetic(4000, 40, row_range=(1000, 4000))
    try:
        with pytest.raises(ValueError, match="shard"):
            snpmatch.inbred_identify_many([_inputs(s)], g, ["x"])
    finally:
        g.close()
    g = snp_genotype.Genotype.from_arrays(cluster_panel["snps"], cluster_panel["positions"], cluster_panel["chrs"],
                                          cluster_panel["chr_regions"], cluster_panel["accessions"])
    try:
        bad = _inputs(s)
        bad.chrs = bad.chrs[:-3]                                      # fewer chromosome names than positions
        with pytest.raises(ValueError, match=r"sample 1 \(bad\)"):
            snpmatch.inbred_identify_many([_inputs(s), bad], g, ["good", "bad"])
    finally:
        g.close()


def _write_bed(path, s):
    with open(path, "w") as fh:
        for c, pos, gt in zip(s["chrs"], s["pos"], s["gt"]):
            fh.write("%s\t%d\t%s\n" % (c, pos, gt))


@pytest.mark.gpu
def test_command_line_samples(lib, cluster_geno, cluster_panel, tmp_path):
    import snpmatch_b200
    db_path = str(tmp_path / "panel.npz")
    cluster_geno.save_packed(db_path)
    samples = [(n, s) for n, s, _ in _batch_samples(cluster_panel) if n in ("pair", "unique", "five", "nomatch")]
    for name, s in samples:
        _write_bed(tmp_path / ("%s.sample.bed" % name), s)
    lst = tmp_path / "samples.txt"
    lst.write_text("".join("%s\n" % (tmp_path / ("%s.sample.bed" % n)) for n, _ in samples if n != "nomatch"))
    out = str(tmp_path / "many")
    assert snpmatch_b200.main(["inbred", "--samples", str(lst), "-d", db_path, "-o", out, "--refine"]) == 0
    for name, _ in samples:
        if name == "nomatch":
            continue
        assert snpmatch_b200.main(["inbred", "-i", str(tmp_path / ("%s.sample.bed" % name)), "-d", db_path, "-o",
                                   str(tmp_path / ("one_" + name)), "--refine"]) == 0
        _same_files(out + "." + name, str(tmp_path / ("one_" + name)))
    assert os.path.exists(out + ".pair.refined.scores.txt")
    # a sample without top hits: every other sample is written, then exit status 1 naming it
    lst.write_text("".join("%s\t%s\n" % (tmp_path / ("%s.sample.bed" % n), tmp_path / ("all_" + n)) for n, _ in samples))
    with pytest.raises(SystemExit) as e:
        snpmatch_b200.main(["inbred", "--samples", str(lst), "-d", db_path, "-o", out, "--refine"])
    assert e.value.code == 1
    for name, _ in samples:
        got = str(tmp_path / ("all_" + name))
        assert os.path.exists(got + ".scores.txt") and os.path.exists(got + ".matches.json")
        if name != "nomatch":
            _same_files(got, out + "." + name)
