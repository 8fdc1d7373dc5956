"""`cross` for many samples in one device pass (csmatch.cross_identify_many, `cross --samples`, the multi-sample forms of
Batch.run_windows / fetch_windows / fetch_window_rows / f1_pairs): every sample's arrays and files equal the ones the
single-sample path gives for it, bit for bit and byte for byte."""
import json
import os

import numpy as np
import pytest

from oracle import snpmatch_oracle as orc
from snpmatch_b200 import synth

RTOL = 1e-9
FILES = (".windowscore.txt", ".scores.txt", ".scores.txt.matches.json", ".matches.json")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


@pytest.fixture(scope="module")
def small_geno(lib, small_panel):
    from snpmatch_b200.core import snp_genotype
    p = small_panel
    g = snp_genotype.Genotype.from_arrays(p["snps"], p["positions"], p["chrs"], p["chr_regions"], p["accessions"])
    yield g
    g.close()


def _inputs(s, wei_key="wei"):
    from snpmatch_b200.core import parsers
    inp = parsers.ParseInputs("")
    inp.load_snp_info(s["chrs"], s["pos"], s["gt"], s[wei_key], s["dp"])
    return inp


def _subset(s, keep):
    return {k: (v[keep] if isinstance(v, np.ndarray) and v.ndim >= 1 and len(v) == len(s["pos"]) else v) for k, v in s.items()}


def _mosaics(p, n=4):
    out = []
    for i in range(n):
        p1, p2 = 3 + 5 * i, 8 + 5 * i
        out.append(synth.make_sample(p["positions"], p["chr_regions"], p["chrs"], 40, n_db=2500, n_extra=300, seed=900 + i,
                                     mosaic=(p1 % 40, p2 % 40, 2_000_000 + 500_000 * i)))
    return out


def _no_match_sample(p, s):
    """The markers of `s` moved one base off the panel's positions: nothing joins."""
    pos = s["pos"] + 1
    names = np.array([c.replace("Chr", "") for c in s["chrs"]])
    hit = np.zeros(len(pos), bool)
    for c, (lo, hi) in enumerate(p["chr_regions"]):
        sel = names == p["chrs"][c]
        hit[sel] = np.isin(pos[sel], p["positions"][lo:hi])
    t = _subset(s, ~hit)
    t["pos"] = pos[~hit]
    return t


def _samples(p, sample_cross, sample_inbred):
    """The batch of the equality tests (names in the order given)."""
    mos = _mosaics(p)
    one_chr = _subset(mos[0], np.char.endswith(mos[0]["chrs"].astype(str), "2"))
    # chromosome 5 ends at 20 Mb in the test genome: markers past it are matched but lie in no window (m counts window rows)
    beyond = _subset(mos[1], np.char.endswith(mos[1]["chrs"].astype(str), "5") | (np.arange(len(mos[1]["pos"])) % 7 == 0))
    assert (beyond["pos"][np.char.endswith(beyond["chrs"].astype(str), "5")] > 20_000_000).any()
    return [("cross", sample_cross), ("inbred", sample_inbred)] + [("mosaic%d" % i, m) for i, m in enumerate(mos)] + [
        ("nomatch", _no_match_sample(p, sample_cross)), ("onechr", one_chr), ("beyond", beyond)]


def _short_genome(tmp_path):
    path = str(tmp_path / "tair10_short5.json")
    with open(path, "w") as fh:
        json.dump({"ref_chrs": synth.TAIR10_CHRS, "ref_chrlen": synth.TAIR10_CHRLEN[:4] + [20_000_000]}, fh)
    return path


def _assert_same(ci_many, ci_one, prefix_many, prefix_one):
    a, b = ci_many.result, ci_one.result
    assert a.num_snps == b.num_snps and a.overlap == b.overlap
    assert np.array_equal(a.accs, b.accs)
    assert np.array_equal(a.scores, b.scores)
    assert np.array_equal(a.ninfo, b.ninfo)
    assert np.array_equal(a.likelis, b.likelis, equal_nan=True)
    assert np.array_equal(a.lrts, b.lrts, equal_nan=True)
    assert np.array_equal(a.matchedTarInd, b.matchedTarInd)
    assert np.array_equal(a.winds_chrs, b.winds_chrs)
    for ext in FILES:
        assert os.path.exists(prefix_many + ext) == os.path.exists(prefix_one + ext), ext
        if os.path.exists(prefix_one + ext):
            assert open(prefix_many + ext, "rb").read() == open(prefix_one + ext, "rb").read(), prefix_one + ext


@pytest.mark.gpu
@pytest.mark.parametrize("wei_key,skip,shuffle", [("wei", False, False), ("wei_hard", True, False), ("wei", False, True)])
def test_batched_equals_single(lib, small_geno, small_panel, sample_cross, sample_inbred, tmp_path, wei_key, skip, shuffle):
    from snpmatch_b200.core import csmatch
    genome = _short_genome(tmp_path)
    samples = _samples(small_panel, sample_cross, sample_inbred)
    if shuffle:
        samples = [samples[i] for i in np.random.default_rng(5).permutation(len(samples))]
    many = csmatch.cross_identify_many([_inputs(s, wei_key) for _, s in samples], small_geno, genome, 300000,
                                       [str(tmp_path / ("many_" + n)) for n, _ in samples], skip_db_hets=skip)
    ms = {}
    for (name, s), ci in zip(samples, many):
        one = csmatch.CrossIdentifier(_inputs(s, wei_key), small_geno, genome, 300000, str(tmp_path / ("one_" + name)),
                                      skip_db_hets=skip)
        _assert_same(ci, one, str(tmp_path / ("many_" + name)), str(tmp_path / ("one_" + name)))
        ms[name] = ci.result.num_snps
    assert ms["nomatch"] == 0 and ms["cross"] > 0
    # m counts the markers inside the sample's windows, not every matched marker
    s = dict(samples)["beyond"]
    assert 0 < ms["beyond"] < len(small_geno.get_positions_idxs(s["chrs"], s["pos"])[0])


@pytest.mark.gpu
def test_split_across_launches(lib, small_geno, small_panel, sample_cross, sample_inbred, tmp_path):
    from snpmatch_b200.core import csmatch
    samples = _samples(small_panel, sample_cross, sample_inbred)[:7]
    one = csmatch.cross_identify_many([_inputs(s) for _, s in samples], small_geno, "athaliana_tair10", 300000,
                                      [str(tmp_path / ("one_" + n)) for n, _ in samples])
    two = csmatch.cross_identify_many([_inputs(s) for _, s in samples], small_geno, "athaliana_tair10", 300000,
                                      [str(tmp_path / ("two_" + n)) for n, _ in samples], samples_per_launch=2)
    for (name, _), a, b in zip(samples, two, one):
        _assert_same(a, b, str(tmp_path / ("two_" + name)), str(tmp_path / ("one_" + name)))


@pytest.mark.gpu
def test_genome_check_names_the_sample(lib, small_geno, small_panel, sample_cross, tmp_path):
    from snpmatch_b200.core import csmatch
    bad = dict(sample_cross)
    bad["chrs"] = np.array(["scaffold%d" % (i % 9) for i in range(len(sample_cross["pos"]))])
    with pytest.raises(AssertionError, match=r"sample 1 .*Please change default --genome option"):
        csmatch.cross_identify_many([_inputs(sample_cross), _inputs(bad)], small_geno, "athaliana_tair10", 300000,
                                    [str(tmp_path / "a"), str(tmp_path / "b")])
    assert not os.listdir(tmp_path)


def _window_batch(lib, g, samples, kmax_n=500):
    from snpmatch_b200.core import genomes, snpmatch
    gen = genomes.Genome("athaliana_tair10")
    cnt, off, n_w, _ = gen.window_layout(g.g.chrs, 300000)
    prep = [g.prepare_markers(s["chrs"], s["pos"], style="genome") for s in samples]
    offs = np.concatenate([[0], np.cumsum([len(p[2]) for p in prep])])
    b = lib.Batch(g.db, offs, np.concatenate([p[1] for p in prep]), np.concatenate([p[2] for p in prep]),
                  np.concatenate([s["wei"][p[0]] for s, p in zip(samples, prep)]))
    b.run_windows(False, 300000, cnt, off, n_w, snpmatch.identity_kmax_table(kmax_n, 0.02))
    b.epilogue()
    return b, prep, offs, (cnt, off, n_w)


@pytest.mark.gpu
def test_window_arrays_vs_oracle_and_f1(lib, small_geno, small_panel, sample_cross, sample_inbred):
    """Each sample's windows of a multi-sample run against the oracle (bars of test_window_scores_bit_exact_vs_oracle), and
    the multi-sample F1 pass == the single-sample one, bit for bit."""
    from snpmatch_b200.core import snpmatch
    p = small_panel
    samples = [sample_cross, sample_inbred] + _mosaics(p)
    b, prep, offs, (cnt, off, n_w) = _window_batch(lib, small_geno, samples)
    tot = b.fetch()
    win = b.fetch_windows()
    rows = b.fetch_window_rows()
    S, n_acc = len(samples), p["snps"].shape[1]
    assert win["score"].shape == (S, n_w, n_acc) and len(rows) == S
    for i, s in enumerate(samples):
        w = orc.window_genotyper(p["snps"], p["chrs"], p["chr_regions"], p["positions"], s["chrs"], s["pos"], s["wei"],
                                 synth.TAIR10_CHRS, synth.TAIR10_CHRLEN, 300000, False)
        assert np.array_equal(tot["score"][i], w.tot_score) and np.array_equal(tot["ninfo"][i], w.tot_ninfo)
        assert int(tot["m"][i]) == w.num_snps
        seen = np.zeros(n_w, bool)
        for widx, sc, ni in w.windows:
            assert np.array_equal(win["score"][i, widx - 1], sc), "sample %d window %d" % (i, widx)
            assert np.array_equal(win["ninfo"][i, widx - 1], ni)
            lik, lr, ident, num_amb, keep = orc.window_epilogue(sc, ni, 0.02)
            np.testing.assert_allclose(win["L"][i, widx - 1], lik, rtol=RTOL, equal_nan=True)
            np.testing.assert_allclose(win["LR"][i, widx - 1], lr, rtol=RTOL, equal_nan=True)
            assert np.array_equal(win["identical"][i, widx - 1], ident)
            assert int(win["num_amb"][i, widx - 1]) == num_amb
            seen[widx - 1] = True
        assert np.array_equal(win["nrows"][i] > 0, seen)
        r = rows[i]
        assert np.array_equal(r["num_amb"], win["num_amb"][i]) and np.array_equal(r["nrows"], win["nrows"][i])
        assert np.array_equal(r["matched_s_idx"], win["matched_s_idx"][i])
        assert np.all((r["matched_s_idx"] >= offs[i]) & (r["matched_s_idx"] < offs[i + 1]))
        for widx in range(1, n_w + 1):
            amb = int(win["num_amb"][i, widx - 1])
            k = np.flatnonzero(win["LR"][i, widx - 1] < snpmatch.lr_thres) if (win["nrows"][i, widx - 1] > 0 and 1 <= amb < n_acc) else np.zeros(0, int)
            lo, hi = r["row_off"][widx - 1], r["row_off"][widx]
            assert np.array_equal(r["acc"][lo:hi], k)
            assert np.array_equal(r["score"][lo:hi], win["score"][i, widx - 1][k])
            assert np.array_equal(r["L"][lo:hi], win["L"][i, widx - 1][k])
            assert np.array_equal(r["identical"][lo:hi], win["identical"][i, widx - 1][k])
    tops = np.stack([np.argsort(-tot["prob"][i])[:10] for i in range(S)])
    f_score, f_ninfo = b.f1_pairs(tops)
    assert f_score.shape == (S, 45)
    for i, s in enumerate(samples):
        order, cid, pos = prep[i]
        one = lib.Batch(small_geno.db, [0, len(pos)], cid, pos, s["wei"][order])
        one.run_windows(False, 300000, cnt, off, n_w, snpmatch.identity_kmax_table(500, 0.02))
        sc1, ni1 = one.f1_pairs(tops[i])
        assert np.array_equal(f_score[i], sc1) and np.array_equal(f_ninfo[i], ni1), "sample %d" % i
        one.close()
    b.close()


@pytest.mark.gpu
def test_1135_accessions_batched_equals_single(lib):
    """64 samples on a 300 000-row panel of 1135 accessions: totals, compacted window rows and F1 sums of the multi-sample
    run == the single-sample runs."""
    from snpmatch_b200.core import genomes, snp_genotype, snpmatch
    g = snp_genotype.Genotype.synthetic(300_000, 1135)
    try:
        positions, regions = g.g.positions, g.g.chr_regions
        ss = [synth.make_sample_fast(positions, regions, 1135, (17 * i) % 1135, n_db=15000, n_extra=1000, seed=3000 + i)
              for i in range(64)]
        cnt, off, n_w, _ = genomes.Genome("athaliana_tair10").window_layout(g.g.chrs, 300000)
        kmax = snpmatch.identity_kmax_table(2000, 0.02)
        offs = np.concatenate([[0], np.cumsum([len(s["pos"]) for s in ss])])
        b = lib.Batch(g.db, offs, np.concatenate([s["chr_ix"] for s in ss]), np.concatenate([s["pos"] for s in ss]),
                      np.concatenate([s["wei"] for s in ss]))
        b.run_windows(False, 300000, cnt, off, n_w, kmax)
        b.epilogue()
        tot = b.fetch()
        rows = b.fetch_window_rows()
        tops = np.stack([np.argsort(-tot["prob"][i])[:10] for i in range(len(ss))])
        f_score, f_ninfo = b.f1_pairs(tops)
        one = lib.Batch(g.db, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3)))
        for i, s in enumerate(ss):
            one.upload([0, len(s["pos"])], s["chr_ix"], s["pos"], s["wei"])
            one.run_windows(False, 300000, cnt, off, n_w, kmax)
            one.epilogue()
            t1 = one.fetch()
            for k in ("score", "matches", "ninfo", "m", "prob", "L", "LR"):
                assert np.array_equal(tot[k][i], t1[k][0], equal_nan=(k in ("prob", "L", "LR"))), (i, k)
            r1 = one.fetch_window_rows()
            r1["matched_s_idx"] = r1["matched_s_idx"] + offs[i]
            for k, v in r1.items():
                assert np.array_equal(rows[i][k], v, equal_nan=(k == "L")), (i, k)
            sc1, ni1 = one.f1_pairs(tops[i])
            assert np.array_equal(f_score[i], sc1) and np.array_equal(f_ninfo[i], ni1), i
        one.close()
        b.close()
    finally:
        g.close()


@pytest.mark.gpu
def test_f1_in_join_order(lib, small_panel, tmp_path):
    """A database with chromosomes 'X' and 'x': the window (genome-style) ids fold the case, the join's do not, so a sample on
    'x' has its F1 pass in join order on a second batch, as the single path does; everything still equals the single path."""
    from snpmatch_b200.core import csmatch, snp_genotype
    p = small_panel
    chrs = np.array(["1", "2", "3", "X", "x"])
    g = snp_genotype.Genotype.from_arrays(p["snps"], p["positions"], chrs, p["chr_regions"], p["accessions"])
    genome = str(tmp_path / "case.json")
    with open(genome, "w") as fh:
        json.dump({"ref_chrs": chrs.tolist(), "ref_chrlen": synth.TAIR10_CHRLEN}, fh)
    try:
        samples = [synth.make_sample(p["positions"], p["chr_regions"], chrs, 40, n_db=2500, n_extra=200, seed=40 + i,
                                     chr_prefix="", mosaic=(2 + i, 20 + i, 3_000_000)) for i in range(3)]
        many = csmatch.cross_identify_many([_inputs(s) for s in samples], g, genome, 300000,
                                           [str(tmp_path / ("many%d" % i)) for i in range(3)])
        assert not all(ci._join_style_same for ci in many)
        for i, (s, ci) in enumerate(zip(samples, many)):
            one = csmatch.CrossIdentifier(_inputs(s), g, genome, 300000, str(tmp_path / ("one%d" % i)))
            _assert_same(ci, one, str(tmp_path / ("many%d" % i)), str(tmp_path / ("one%d" % i)))
    finally:
        g.close()


def _write_bed(path, s):
    with open(path, "w") as fh:
        for c, pos, gt in zip(s["chrs"], s["pos"], s["gt"]):
            fh.write("%s\t%d\t%s\n" % (c, pos, gt))


@pytest.mark.gpu
def test_command_line_samples(lib, small_geno, small_panel, sample_cross, sample_inbred, tmp_path):
    import snpmatch_b200
    db_path = str(tmp_path / "panel.npz")
    small_geno.save_packed(db_path)
    samples = [("inbred", sample_inbred), ("cross", sample_cross), ("mosaic", _mosaics(small_panel, 1)[0])]
    lst = tmp_path / "samples.txt"
    with open(lst, "w") as fh:
        for k, (name, s) in enumerate(samples):
            _write_bed(tmp_path / ("%s.sample.bed" % name), s)
            fh.write("%s\n" % (tmp_path / ("%s.sample.bed" % name)) if k != 1 else "%s\t%s\n" % (tmp_path / ("%s.sample.bed" % name), tmp_path / "own"))
    out = str(tmp_path / "many")
    assert snpmatch_b200.main(["cross", "--samples", str(lst), "-d", db_path, "-o", out, "-b", "300000"]) == 0
    for k, (name, _) in enumerate(samples):
        assert snpmatch_b200.main(["cross", "-i", str(tmp_path / ("%s.sample.bed" % name)), "-d", db_path, "-o", str(tmp_path / ("one_" + name)),
                                   "-b", "300000"]) == 0
        got = str(tmp_path / "own") if k == 1 else out + "." + name
        for ext in FILES:
            assert os.path.exists(got + ext) == os.path.exists(str(tmp_path / ("one_" + name)) + ext)
            if os.path.exists(got + ext):
                assert open(got + ext, "rb").read() == open(str(tmp_path / ("one_" + name)) + ext, "rb").read()


@pytest.mark.gpu
def test_sharded_windows_reject_many_samples(lib, small_geno, sample_cross):
    from snpmatch_b200.core import snpmatch
    s = sample_cross
    b, _, _, (cnt, off, n_w) = _window_batch(lib, small_geno, [s, s])
    with pytest.raises(lib.SnpmError, match="single-sample batch"):
        b.run_windows_begin(False, 300000, cnt, off, n_w, snpmatch.identity_kmax_table(500, 0.02))
    b.close()


# ---- `cross --samples` input checks: they fail before any device work, so they run without a GPU -------------------------
def _cli_fails(argv, tmp_path, before):
    import snpmatch_b200
    with pytest.raises(SystemExit) as e:
        snpmatch_b200.main(argv)
    assert e.value.code != 0
    assert sorted(os.listdir(tmp_path)) == before, "nothing may be written"


def _bed_files(tmp_path, sample_inbred, n=2):
    paths = []
    for i in range(n):
        paths.append(str(tmp_path / ("s%d.sample.bed" % i)))
        _write_bed(paths[-1], sample_inbred)
    return paths


def test_cli_samples_duplicate_prefixes(tmp_path, sample_inbred):
    a, b = _bed_files(tmp_path, sample_inbred)
    lst = tmp_path / "list.txt"
    lst.write_text("%s\tsame\n%s\tsame\n" % (a, b))
    _cli_fails(["cross", "--samples", str(lst), "-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "out")], tmp_path,
               sorted(os.listdir(tmp_path)))
    # two files whose names agree up to the first '.' get the same default prefix
    os.makedirs(tmp_path / "d")
    c = str(tmp_path / "d" / "s0.other.bed")
    _write_bed(c, sample_inbred)
    lst.write_text("%s\n%s\n" % (a, c))
    _cli_fails(["cross", "--samples", str(lst), "-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "out")], tmp_path,
               sorted(os.listdir(tmp_path)))


def test_cli_samples_missing_file_and_empty_list(tmp_path, sample_inbred):
    a, _ = _bed_files(tmp_path, sample_inbred)
    lst = tmp_path / "list.txt"
    lst.write_text("%s\n%s\n" % (a, tmp_path / "missing.bed"))
    _cli_fails(["cross", "--samples", str(lst), "-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "out")], tmp_path,
               sorted(os.listdir(tmp_path)))
    lst.write_text("\n  \n")
    _cli_fails(["cross", "--samples", str(lst), "-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "out")], tmp_path,
               sorted(os.listdir(tmp_path)))


def test_cli_input_and_samples_exclusive(tmp_path, sample_inbred):
    a, _ = _bed_files(tmp_path, sample_inbred)
    lst = tmp_path / "list.txt"
    lst.write_text("%s\n" % a)
    _cli_fails(["cross", "-i", a, "--samples", str(lst), "-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "out")], tmp_path,
               sorted(os.listdir(tmp_path)))


def test_read_sample_list_default_prefixes(tmp_path, sample_inbred):
    import snpmatch_b200
    a, b = _bed_files(tmp_path, sample_inbred)
    lst = tmp_path / "list.txt"
    lst.write_text("%s\n\n%s\tmine\n" % (a, b))
    assert snpmatch_b200.read_sample_list(str(lst), "run") == [(a, "run.s0"), (b, "mine")]
