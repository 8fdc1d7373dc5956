"""The position-order path behind `cross` at its launch-shape limits, against the CPU oracle:

1. windows (k_window_bounds -> k_score_segments in segment-table form -> k_combine -> k_window_epilogue -> k_window_row_offsets
   -> k_window_compact) at every slice shape of the segment kernel, on panels whose windows reach the epilogue's edges
   (tests/test_cross_limits_cpu.py builds them), also on three row shards summed by hand;
2. simulated F1s (k_f1_partial -> k_f1_final) against an exact reference with dyadic weights, over 1 to 4 row blocks, repeated
   and word-edge accessions and n_top up to 4096, and against orc.f1_pair_scores with likelihood weights;
3. the order-exact kernel (mode 0) and the popcount kernel (mode 1) of a genotyper run where the earlier sweeps stop.

Bars: integers, window scores, totals and every fp64 score of the order-exact kernel ==; likelihoods and ratios rtol 1e-9."""
import numpy as np
import pytest

from oracle import snpmatch_oracle as orc
from snpmatch_b200 import synth
from test_cross_limits_cpu import (BIN, CHR1_WINDOWS, dyadic_weights, f1_reference, pl_weights, random_codes, window_oracle,
                                   window_panel, window_rows_reference, window_samples)

RTOL = 1e-9


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


@pytest.fixture(scope="module")
def kmax():
    from snpmatch_b200.core import snpmatch
    return snpmatch.identity_kmax_table(1000, 0.02)


def _layout(bin_len):
    from snpmatch_b200.core import genomes
    return genomes.Genome("athaliana_tair10").window_layout(np.array(synth.TAIR10_CHRS), bin_len)[:3]


def _concat(samples):
    offs = np.concatenate([[0], np.cumsum([len(s[1]) for s in samples])])
    return offs, np.concatenate([s[0] for s in samples]), np.concatenate([s[1] for s in samples]), np.concatenate([s[3] for s in samples])


_PANELS = {}


def _panel(n_acc):
    if n_acc not in _PANELS:
        _PANELS.clear()
        pos, regions, codes = window_panel(n_acc)
        _PANELS[n_acc] = (pos, regions, codes, window_samples(pos, regions, codes))
    return _PANELS[n_acc]


def _check_windows(tot, win, rows, i, w, n_w, offs_i, boundary=()):
    """Sample i of a windows run against the oracle's windows `w`: scores == except in the `boundary` windows (0-based), and
    there and in the totals rtol 1e-12 when there are such windows."""
    assert int(tot["m"][i]) == w.num_snps
    assert np.array_equal(tot["ninfo"][i], w.tot_ninfo)
    if not boundary:
        assert np.array_equal(tot["score"][i], w.tot_score)
    else:
        np.testing.assert_allclose(tot["score"][i], w.tot_score, rtol=1e-12, atol=0)
    seen = np.zeros(n_w, bool)
    for widx, sc, ni in w.windows:
        k = widx - 1
        seen[k] = True
        assert np.array_equal(win["ninfo"][k], ni), "window %d" % widx
        if k not in boundary:
            assert np.array_equal(win["score"][k], sc), "window %d" % widx
        else:
            np.testing.assert_allclose(win["score"][k], sc, rtol=1e-12, atol=0)
        lik, lr, ident, num_amb, _ = orc.window_epilogue(sc, ni, 0.02)
        np.testing.assert_allclose(win["L"][k], lik, rtol=RTOL, equal_nan=True)
        np.testing.assert_allclose(win["LR"][k], lr, rtol=RTOL, equal_nan=True)
        assert np.array_equal(win["identical"][k], ident), "window %d" % widx
        assert int(win["num_amb"][k]) == num_amb, "window %d" % widx
    assert np.array_equal(win["nrows"] > 0, seen)
    assert np.array_equal(win["num_amb"][~seen], np.zeros(int((~seen).sum())))
    if offs_i is not None:
        assert np.array_equal(win["matched_s_idx"], w.matched_tar + offs_i)
    ref = window_rows_reference(w, n_w)
    assert np.array_equal(rows["num_amb"], ref["num_amb"])
    assert np.array_equal(rows["row_off"], ref["row_off"]), "row offsets"
    assert np.array_equal(rows["acc"], ref["acc"]) and np.array_equal(rows["ninfo"], ref["ninfo"])
    assert np.array_equal(rows["identical"], ref["identical"])
    inside = np.repeat(np.arange(n_w), np.diff(ref["row_off"]))
    plain = ~np.isin(inside, list(boundary))
    assert np.array_equal(rows["score"][plain], ref["score"][plain])
    np.testing.assert_allclose(rows["score"], ref["score"], rtol=1e-12, atol=0)
    np.testing.assert_allclose(rows["L"], ref["L"], rtol=RTOL)
    return ref


# ---- 1. windows at every slice shape of k_score_segments ----------------------------------------------------------------------
# A -> (words per row, consumer warps, slices): 1 keeps no row; 257 (10, 3, 1) and two passes of the epilogue / compaction loops;
# 700 (22, 6, 1); 960 (30, 8, 1) the <9,2> instantiation; 1135 (36, 9, 1) <10,2>; 1300 (42, 11, 1) and 1536 (48, 12, 1) generic;
# 1537 (50, 8, 2): slices of 32 + 18 words, warps 5-7 idle in the second; 2049 (66, 8, 3): the last slice 2 words
WINDOW_ACCS = [1, 257, 700, 960, 1135, 1300, 1536, 1537, 2049]


@pytest.mark.gpu
@pytest.mark.parametrize("skip", [False, True], ids=["hets", "skip_hets"])
@pytest.mark.parametrize("n_acc", WINDOW_ACCS)
def test_windows_vs_oracle(lib, kmax, n_acc, skip):
    pos, regions, codes, samples = _panel(n_acc)
    cnt, off, n_w = _layout(BIN)
    assert len(samples) * n_w == 1197                         # two passes of the 1024-thread offset scan
    db = lib.Database(pos, regions, n_acc)
    db.load_int8(codes)
    offs, cid, spos, wei = _concat(samples)
    b = lib.Batch(db, offs, cid, spos, wei)
    try:
        b.run_windows(skip, BIN, cnt, off, n_w, kmax)
        b.epilogue()
        tot = b.fetch()
        win = b.fetch_windows()
        rows = b.fetch_window_rows()
        for i, s in enumerate(samples):
            w = window_oracle(pos, regions, codes, s, skip)
            ref = _check_windows(tot, {k: v[i] for k, v in win.items()}, rows[i], i, w, n_w, offs[i])
            if i == 1:
                assert w.num_snps == 0 and rows[i]["row_off"][-1] == 0
            else:
                amb = ref["num_amb"]
                assert amb[CHR1_WINDOWS["all_equal"]] == n_acc and amb[CHR1_WINDOWS["all_missing"]] == 0
                assert int(win["nrows"][i, CHR1_WINDOWS["one_marker"]]) == 1
                assert int(win["nrows"][i, CHR1_WINDOWS["dense"]]) >= 257
                assert (ref["row_off"][-1] > 0) == (n_acc > 1)
        assert int(np.nanargmin(tot["L"][0])) == n_acc - 1
    finally:
        b.close()
        db.close()


@pytest.mark.gpu
def test_windows_vs_oracle_50kb_bins(lib, kmax):
    """About 7 000 window slots: the single-CTA offset scan takes seven passes."""
    n_acc = 1135
    pos, regions, codes, samples = _panel(n_acc)
    cnt, off, n_w = _layout(50_000)
    assert 3 * n_w > 7000
    db = lib.Database(pos, regions, n_acc)
    db.load_int8(codes)
    offs, cid, spos, wei = _concat(samples)
    b = lib.Batch(db, offs, cid, spos, wei)
    try:
        b.run_windows(False, 50_000, cnt, off, n_w, kmax)
        b.epilogue()
        tot, win, rows = b.fetch(), b.fetch_windows(), b.fetch_window_rows()
        for i, (c, p, _, wt) in enumerate(samples):
            w = orc.window_genotyper(codes, np.array(synth.TAIR10_CHRS), regions, pos, np.array(synth.TAIR10_CHRS)[c], p, wt,
                                     synth.TAIR10_CHRS, synth.TAIR10_CHRLEN, 50_000, False)
            _check_windows(tot, {k: v[i] for k, v in win.items()}, rows[i], i, w, n_w, offs[i])
    finally:
        b.close()
        db.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_acc", [1135, 2049])
def test_windows_on_three_row_shards(lib, kmax, n_acc):
    """Three SNP-row shards on one GPU, cut inside windows (one inside the 300-row window); the packed partials of
    snpm_batch_run_windows_begin summed by hand, then the second half on every shard: integers ==, scores == except in the
    windows that straddle a cut (rtol 1e-12), against the oracle."""
    import torch
    from snpmatch_b200 import sharding
    pos, regions, codes, samples = _panel(n_acc)
    cnt, off, n_w = _layout(BIN)
    cid, spos, _, wei = samples[0]
    chr1 = np.arange(regions[0][0], regions[0][1])
    dense = chr1[(pos[chr1].astype(np.int64) - 1) // BIN == CHR1_WINDOWS["dense"]]
    c3 = int(regions[2][0]) + (int(regions[2][1]) - int(regions[2][0])) // 2
    cuts = [int(dense[150]), c3]
    gwin = _global_windows(pos, regions)
    boundary = {int(gwin[c - 1]) for c in cuts if gwin[c - 1] == gwin[c]}
    assert len(boundary) == 2
    w = window_oracle(pos, regions, codes, samples[0], False)
    edges = [0] + cuts + [len(pos)]
    shards = []
    try:
        for r0, r1 in zip(edges[:-1], edges[1:]):
            d = lib.Database(pos[r0:r1], sharding.local_regions(regions, r0, r1), n_acc, row0_global=r0)
            d.load_int8(codes[r0:r1])
            i0, i1 = sharding.shard_marker_range(cid, spos, regions, pos, r0, r1)
            shards.append((d, lib.Batch(d, [0, i1 - i0], cid[i0:i1], spos[i0:i1], wei[i0:i1]), i0))
        views = []
        for _, bb, _ in shards:
            ptr, n = bb.run_windows_begin(False, BIN, cnt, off, n_w, kmax)
            views.append(sharding.device_view(ptr, n, torch.device("cuda", 0)))
        torch.cuda.synchronize()
        total = views[0].clone() + views[1] + views[2]
        for v in views:
            v.copy_(total)
        torch.cuda.synchronize()
        matched = []
        for _, bb, i0 in shards:
            bb.run_windows_finish()
            bb.epilogue()
            tot, win, rows = bb.fetch(), bb.fetch_windows(), bb.fetch_window_rows()
            matched.append(win["matched_s_idx"] + i0)        # a shard lists its own markers: all of them, in order, below
            _check_windows(tot, win, rows, 0, w, n_w, None, boundary=boundary)
        assert np.array_equal(np.concatenate(matched), w.matched_tar)
    finally:
        for d, bb, _ in shards:
            bb.close()
            d.close()


def _global_windows(pos, regions):
    counts = np.array([orc.num_windows(l, BIN) for l in synth.TAIR10_CHRLEN])
    chrom = np.repeat(np.arange(len(regions)), regions[:, 1] - regions[:, 0])
    return np.concatenate([[0], np.cumsum(counts)])[:-1][chrom] + (pos.astype(np.int64) - 1) // BIN


# ---- 2. simulated F1s ----------------------------------------------------------------------------------------------------------
F1_PAIRS = [1, 4095, 4096, 4097, 12_289, 0]           # matched pairs per sample: 1 to 4 row blocks of 4096, and none
F1_ROWS = 16_000


def _f1_setup(lib, n_acc, weights, pairs=F1_PAIRS, seed=5):
    """A panel of F1_ROWS random rows (10 % hets) and one sample per entry of `pairs`, each matching that many rows (the empty one
    carries 7 markers between panel rows); a batch of all of them after run().  A sample is (chrom, pos, matched rows, wei)."""
    rng = np.random.default_rng(seed + n_acc)
    pos, regions = synth.panel_positions(F1_ROWS)
    codes = random_codes(rng, F1_ROWS, n_acc, het=0.1)
    chrom = np.repeat(np.arange(len(regions), dtype=np.int32), regions[:, 1] - regions[:, 0])
    samples = []
    for n in pairs:
        rows = np.sort(rng.choice(F1_ROWS, size=n, replace=False)) if n else np.arange(7) * 1000
        p = pos[rows] + (0 if n else 1)
        call = rng.integers(0, 3, size=len(rows))
        wei = dyadic_weights(rng, len(rows)) if weights == "dyadic" else pl_weights(rng, call)
        samples.append((chrom[rows], p.astype(np.int32), rows[:n], wei))
    db = lib.Database(pos, regions, n_acc)
    db.load_int8(codes)
    offs, cid, spos, wei = _concat(samples)
    b = lib.Batch(db, offs, cid, spos, wei)
    b.run()
    for i, (_, _, rows, _) in enumerate(samples):
        db_idx, s_idx = b.fetch_pairs(i)
        assert len(db_idx) == pairs[i]
        if pairs[i]:
            assert np.array_equal(db_idx, rows)
    return db, b, codes, samples


def _lists(rng, n_acc, n_top, S):
    """One accession list per sample: it holds 0, 31, 32 and A-1 (those below A) and repeats one accession; the rest is drawn
    from at most 160 distinct accessions, which keeps the reference's products small at n_top = 4096."""
    edge = [a for a in (0, 31, 32, n_acc - 1) if a < n_acc]
    pool = rng.permutation(n_acc)[:160]
    out = []
    for _ in range(S):
        lst = np.concatenate([edge, [edge[0]], rng.choice(pool, size=max(0, n_top - len(edge) - 1))])[:n_top]
        out.append(rng.permutation(lst))
    return np.stack(out).astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("n_acc", [40, 1135, 2049])
def test_f1_dyadic_weights_equal_the_reference(lib, n_acc):
    """Weights k/64: every partial sum is exact, so the device must equal the reference whatever its summation order.
    n_top 363 and up gives more than 65 535 pairs, past the grid-y limit where the pairs used to sit."""
    db, b, codes, samples = _f1_setup(lib, n_acc, "dyadic")
    rng = np.random.default_rng(n_acc)
    try:
        for n_top in (2, 10, 64, 362, 363):
            acc = _lists(rng, n_acc, n_top, len(samples))
            score, ninfo = b.f1_pairs(acc)
            P = n_top * (n_top - 1) // 2
            assert score.shape == (len(samples), P)
            for i, (_, _, rows, wei) in enumerate(samples):
                ref_s, ref_n = f1_reference(codes[rows], wei[:len(rows)], acc[i])
                assert np.array_equal(ninfo[i], ref_n), (n_top, i)
                assert np.array_equal(score[i], ref_s), (n_top, i)
    finally:
        b.close()
        db.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_acc", [40, 1135, 2049])
def test_f1_n_top_4096(lib, n_acc):
    """n_top = 4096: 8 386 560 pairs per sample, on samples of 4096 and 1 matched pairs."""
    db, b, codes, samples = _f1_setup(lib, n_acc, "dyadic", pairs=[4096, 1])
    rng = np.random.default_rng(7 + n_acc)
    try:
        acc = _lists(rng, n_acc, 4096, 2)
        score, ninfo = b.f1_pairs(acc)
        assert score.shape == (2, 4096 * 4095 // 2)
        for i, (_, _, rows, wei) in enumerate(samples):
            ref_s, ref_n = f1_reference(codes[rows], wei, acc[i])
            assert np.array_equal(ninfo[i], ref_n) and np.array_equal(score[i], ref_s), i
    finally:
        b.close()
        db.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_acc", [40, 1135, 2049])
def test_f1_likelihood_weights_vs_oracle(lib, n_acc):
    """Likelihood weights: counts == orc.f1_pair_scores, scores rtol 1e-12 (the oracle sums each class with np.sum)."""
    db, b, codes, samples = _f1_setup(lib, n_acc, "pl")
    rng = np.random.default_rng(3 + n_acc)
    try:
        acc = _lists(rng, n_acc, 10, len(samples))
        score, ninfo = b.f1_pairs(acc)
        for i, (_, _, rows, wei) in enumerate(samples):
            common = (rows, np.arange(len(rows)))
            _, o_score, o_ninfo = orc.f1_pair_scores(codes, common, wei[:len(rows)], acc[i])
            assert np.array_equal(ninfo[i], o_ninfo), i
            np.testing.assert_allclose(score[i], o_score, rtol=1e-12, atol=0)
    finally:
        b.close()
        db.close()


@pytest.mark.gpu
def test_f1_refusals(lib):
    import ctypes
    db, b, codes, samples = _f1_setup(lib, 40, "dyadic", pairs=[100, 5])
    try:
        for n_top in (1, 4097):
            with pytest.raises(lib.SnpmError, match="n_top %d" % n_top):
                b.f1_pairs(np.zeros((2, n_top), np.int32))
        bad = np.zeros((2, 10), np.int32)
        bad[1, 3] = 40
        with pytest.raises(lib.SnpmError, match="accession index 40 of sample 1"):
            b.f1_pairs(bad)
        good = np.tile(np.arange(10, dtype=np.int32), (2, 1))
        s1, n1 = b.f1_pairs(good)                                 # the batch still works after a refusal
        ref_s, ref_n = f1_reference(codes[samples[0][2]], samples[0][3], good[0])
        assert np.array_equal(s1[0], ref_s) and np.array_equal(n1[0], ref_n)
    finally:
        b.close()
        db.close()
    # 257 samples x 8 386 560 pairs is more pair slots than k_f1_final numbers with an int: refused before any allocation
    pos, regions = synth.panel_positions(1000)
    db = lib.Database(pos, regions, 40)
    db.load_int8(np.zeros((1000, 40), np.int8))
    S = 257
    b = lib.Batch(db, np.arange(S + 1), np.zeros(S, np.int32), pos[:S].astype(np.int32), np.full((S, 3), 0.5))
    try:
        b.run()
        acc = np.zeros((S, 4096), np.int32)
        out_s, out_n = np.zeros(1), np.zeros(1, np.int64)
        p = (lambda a: a.ctypes.data_as(ctypes.c_void_p))
        rc = lib.load().snpm_batch_f1_pairs(b._h, p(acc), 4096, p(out_s), p(out_n))
        assert rc != 0
        assert "257 samples x 8386560 pairs" in lib.load().snpm_last_error().decode()
    finally:
        b.close()
        db.close()


# ---- 3. order-exact and popcount kernels of a genotyper run ------------------------------------------------------------------
# 960 / 1300 / 1537: shapes of k_score_segments (above); k_score_hard: 2700 (86 words, 2 segments per CTA), 4129 (130 words:
# one segment, 130 of 256 threads), 8192 (one full 256-word slice), 8193 (slices of 256 + 2 words)
GENO_ACCS = [960, 1300, 1537, 2700, 4129, 8192, 8193]
GENO_PAIRS = [2500, 0, 1001]


def _geno_setup(lib, n_acc, seed=9):
    rng = np.random.default_rng(seed + n_acc)
    n_rows = 6000
    pos, regions = synth.panel_positions(n_rows)
    codes = random_codes(rng, n_rows, n_acc)
    chrom = np.repeat(np.arange(len(regions), dtype=np.int32), regions[:, 1] - regions[:, 0])
    samples = []
    for n in GENO_PAIRS:
        rows = np.sort(rng.choice(n_rows, size=n, replace=False)) if n else np.arange(5) * 1000
        call = rng.integers(0, 3, size=len(rows))
        hard = np.zeros((len(rows), 3))
        hard[np.arange(len(rows)), call] = 1.0
        samples.append((chrom[rows], (pos[rows] + (0 if n else 1)).astype(np.int32), rows, pl_weights(rng, call), hard))
    db = lib.Database(pos, regions, n_acc)
    db.load_int8(codes)
    return db, codes, samples


def _geno_oracle(codes, rows, wei, skip, chunk):
    n_acc = codes.shape[1]
    score, ninfo = np.zeros(n_acc), np.zeros(n_acc, dtype=np.int64)
    for j in range(0, len(rows), chunk):
        t_s, t_n = orc.match_gts_accs(wei[j:j + chunk], codes[rows[j:j + chunk]], skip)
        score, ninfo = score + t_s, ninfo + t_n
    return score, ninfo


def _geno_run(b, offs, samples, key, skip, mode):
    b.upload(offs, np.concatenate([s[0] for s in samples]), np.concatenate([s[1] for s in samples]),
             np.concatenate([s[key] for s in samples]))
    b.run(skip_db_hets=skip, kernel_mode=mode)
    b.epilogue()
    return {k: v.copy() for k, v in b.fetch().items()}


def _check_geno(r, i, ref_s, ref_n, m):
    assert int(r["m"][i]) == m
    assert np.array_equal(r["score"][i], ref_s) and np.array_equal(r["ninfo"][i], ref_n)
    assert np.array_equal(r["matches"][i], ref_s.astype(np.int64))
    lik, lr = orc.calculate_likelihoods(ref_s.astype(np.int64), ref_n)
    np.testing.assert_allclose(r["L"][i], lik, rtol=RTOL, equal_nan=True)
    np.testing.assert_allclose(r["LR"][i], lr, rtol=RTOL, equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("skip", [False, True], ids=["hets", "skip_hets"])
@pytest.mark.parametrize("n_acc", GENO_ACCS)
def test_genotyper_kernels_vs_oracle(lib, n_acc, skip):
    db, codes, samples = _geno_setup(lib, n_acc)
    offs = np.concatenate([[0], np.cumsum([len(s[1]) for s in samples])])
    b = lib.Batch(db, offs, np.concatenate([s[0] for s in samples]), np.concatenate([s[1] for s in samples]),
                  np.concatenate([s[3] for s in samples]))
    try:
        r_pl = _geno_run(b, offs, samples, 3, skip, lib.KERNEL_FP64)
        r_h0 = _geno_run(b, offs, samples, 4, skip, lib.KERNEL_FP64)
        r_h1 = _geno_run(b, offs, samples, 4, skip, lib.KERNEL_POPCOUNT)
        for k in ("score", "matches", "ninfo", "m", "prob", "L", "LR"):
            assert np.array_equal(r_h0[k], r_h1[k], equal_nan=True), k
        for i, (_, _, rows, pl, hard) in enumerate(samples):
            m = len(rows) if GENO_PAIRS[i] else 0
            rows = rows if m else rows[:0]
            _check_geno(r_pl, i, *_geno_oracle(codes, rows, pl[:m], skip, 1000), m)
            _check_geno(r_h1, i, *_geno_oracle(codes, rows, hard[:m], skip, 1000), m)
    finally:
        b.close()
        db.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_acc", [1537, 2049])
def test_genotyper_chunk_rows_vs_oracle(lib, n_acc):
    """Chunks of 1, 63, 65 and 257 rows (less than one 64-row tile, just past one, past the 4-stage ring) == the oracle's
    chunk loop with the same chunk size."""
    db, codes, samples = _geno_setup(lib, n_acc)
    offs = np.concatenate([[0], np.cumsum([len(s[1]) for s in samples])])
    b = lib.Batch(db, offs, np.concatenate([s[0] for s in samples]), np.concatenate([s[1] for s in samples]),
                  np.concatenate([s[3] for s in samples]))
    try:
        for chunk in (1, 63, 65, 257):
            b.set_chunk_rows(chunk)
            for skip in (False, True):
                r = _geno_run(b, offs, samples, 3, skip, lib.KERNEL_FP64)
                for i, (_, _, rows, pl, _) in enumerate(samples):
                    m = len(rows) if GENO_PAIRS[i] else 0
                    _check_geno(r, i, *_geno_oracle(codes, rows[:m], pl[:m], skip, chunk), m)
    finally:
        b.close()
        db.close()
