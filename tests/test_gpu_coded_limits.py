"""The coded path (snpm_batch_upload_coded -> join -> device grouping, csrc/group_sort.cuh -> k_score_grouped2 ->
k_combine_grouped -> k_grouped_finalize + k_epilogue) where it changes behaviour: the capacity of the per-sample group table
(GH_MAX_GROUPS dense ids, GH_SLOTS hash slots), the 16-bit counters of the one-CTA-per-sample grouping (GP_MAX_PAIRS), row
shards whose totals are summed by hand (all-reduce and reduce-scatter), a second epilogue on the same run, and the panel widths
at which the scoring kernel's slice shape or the epilogue's cluster size changes.

Every case is compared with the order-exact fp64 kernel (mode 0) on the same batch and, for at least one sample, with the
CPU oracle.  Bars as in tests/test_gpu_coded.py: matches, ninfo, m and prob ==; fp64 scores rtol 1e-12 (== for re-scored
samples); likelihoods and ratios rtol 1e-9."""
import numpy as np
import pytest

from oracle import snpmatch_oracle as orc
from snpmatch_b200 import sharding, synth

RTOL = 1e-9
SCORE_RTOL = 1e-12
GH_MAX_GROUPS = 2048                 # csrc/group_sort.cuh
GP_MAX_PAIRS = 65535


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


def _concat(samples, wei_key="wei"):
    offs = np.concatenate([[0], np.cumsum([len(s["pos"]) for s in samples])])
    return (offs, np.concatenate([s["chr_ix"] for s in samples]).astype(np.int32), np.concatenate([s["pos"] for s in samples]).astype(np.int32),
            np.concatenate([s[wei_key] for s in samples]))


def _oracle_sample(db_idx, s_idx, wei, n_acc, skip=False):
    """Genotyper.genotyper's chunk loop (snpmatch.py:218-225) on the panel rows of the matched pairs."""
    codes = synth.panel_codes(synth.SEED_PANEL, db_idx, n_acc)
    score, ninfo = np.zeros(n_acc), np.zeros(n_acc, dtype=np.int64)
    for j in range(0, len(db_idx), 1000):
        t_s, t_n = orc.match_gts_accs(wei[s_idx[j:j + 1000]], codes[j:j + 1000].copy(), skip)
        score, ninfo = score + t_s, ninfo + t_n
    return score, ninfo


def _check_oracle(r, i, pairs, wei, n_acc, skip=False):
    ref_s, ref_n = _oracle_sample(pairs[0], pairs[1], wei, n_acc, skip)
    lik, lr = orc.calculate_likelihoods(ref_s.astype(np.int64), ref_n)
    assert np.array_equal(r["matches"][i], ref_s.astype(np.int64)) and np.array_equal(r["ninfo"][i], ref_n)
    np.testing.assert_allclose(r["score"][i], ref_s, rtol=SCORE_RTOL, atol=0)
    np.testing.assert_allclose(r["L"][i], lik, rtol=RTOL, equal_nan=True)
    np.testing.assert_allclose(r["LR"][i], lr, rtol=RTOL, equal_nan=True)


def _check_against(r, ref, i, exact_scores=False):
    assert np.array_equal(r["matches"][i], ref["matches"]), "matches differ"
    assert np.array_equal(r["ninfo"][i], ref["ninfo"]), "ninfo differs"
    assert int(r["m"][i]) == int(ref["m"])
    if exact_scores:
        assert np.array_equal(r["score"][i], ref["score"])
    else:
        np.testing.assert_allclose(r["score"][i], ref["score"], rtol=SCORE_RTOL, atol=0)
    np.testing.assert_array_equal(r["prob"][i], ref["prob"])
    np.testing.assert_allclose(r["L"][i], ref["L"], rtol=RTOL, equal_nan=True)
    np.testing.assert_allclose(r["LR"][i], ref["LR"], rtol=RTOL, equal_nan=True)


def _row(res, i):
    return {k: v[i] for k, v in res.items()}


def _copy(res):
    return {k: v.copy() for k, v in res.items()}


def _run_exact(b, skip=False, mode=0):
    b.run(skip_db_hets=skip, kernel_mode=mode)
    b.epilogue()
    return _copy(b.fetch())


def _run_coded(lib, b, cs, skip=False):
    b.upload_coded(cs)
    b.run(skip_db_hets=skip, kernel_mode=lib.KERNEL_GROUPED)
    b.epilogue()
    return _copy(b.fetch()), b.guard_counts().copy()


def _spread(n, phase):
    """n distinct weights in (0.05, 0.95) without a short binary expansion: sums of them lie near an integer only by chance, so
    the truncation guard stays silent and a flag means overflow."""
    return 0.05 + 0.9 * np.modf((np.arange(n) + 1) * phase)[0]


_GRID = _spread(64, 0.6180339887498949)


def _triples(k):
    """k distinct weight triples (columns ref, het, alt), a third of them called as each class: one weight is exactly 1.0, the
    other two come from a 64 x 64 grid of values (at most 3 * 4096 triples)."""
    t = np.arange(k)
    cls, q = t % 3, t // 3
    assert q.max(initial=0) < 64 * 64
    x, y, one = _GRID[q % 64], _GRID[q // 64], np.ones(k)
    return np.where((cls == 0)[:, None], np.stack([one, x, y], 1),
                    np.where((cls == 1)[:, None], np.stack([x, y, one], 1), np.stack([x, one, y], 1)))


def _n_triples(w):
    return len(np.unique(np.asarray(w), axis=0))


def _with_triples(s, k, seed, rows_lo=None, rows_hi=None):
    """Sample s (make_sample_fast) with its matched markers in panel rows [rows_lo, rows_hi) carrying exactly k distinct triples
    (each at least once, the rest drawn at random, order shuffled)."""
    rng = np.random.default_rng(seed)
    rows = s["rows"]
    sel = (rows >= 0) & (rows >= (rows_lo or 0)) & (rows < (rows_hi if rows_hi is not None else np.iinfo(np.int64).max))
    idx = np.flatnonzero(sel)
    assert len(idx) >= k, (len(idx), k)
    pick = rng.permutation(np.concatenate([np.arange(k), rng.integers(0, k, size=len(idx) - k)]))
    s["wei"][idx] = _triples(k)[pick]
    return s


def _sample(pos, regions, n_acc, true_acc, n_db, n_extra, seed):
    s = synth.make_sample_fast(pos, regions, n_acc, true_acc, n_db=n_db, n_extra=n_extra, seed=seed, het=0.05)
    s["wei"] = s["wei"].copy()
    return s


# ---- 1. capacity of the per-sample group table ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("wide", [False, True], ids=["keys32", "keys64"])
@pytest.mark.parametrize("group_kernel", ["sample", "tiled"])
def test_group_table_capacity(lib, wide, group_kernel, monkeypatch):
    """Samples whose matched markers carry exactly 2047 and 2048 distinct weight triples (the last dense id in use: every counter
    slot of k_group_scan / k_group_sample) score like the order-exact kernel and are not flagged; 2049 (one key folded into id
    2047) and 5000 (the 4096-slot hash table full: gh_insert gives up) are flagged and re-scored; the ordinary neighbours in
    the same batch are untouched.  Both key widths (table of <= 1024 values: 32-bit keys; more: 64-bit) and both grouping forms."""
    monkeypatch.setenv("SNPM_GROUP_KERNEL", group_kernel)
    n_rows, n_acc = 40000, 300
    pos, regions = synth.panel_positions(n_rows)
    db = lib.Database(pos, regions, n_acc)
    db.fill_synthetic(synth.SEED_PANEL)
    samples, where = [], {}
    for i, k in enumerate((None, 2047, 2048, None, 2049, 5000)):
        s = _sample(pos, regions, n_acc, true_acc=7 + 31 * i, n_db=3000 if k is None else 9000, n_extra=500, seed=8100 + i)
        if k is not None:
            _with_triples(s, k, seed=8200 + i)
            where[k] = i
            if wide:                # values the join never matches: they widen the codes, not the key table
                extra = np.flatnonzero(s["rows"] < 0)
                s["wei"][extra] = _spread(3 * len(extra), 0.41421356237309503 + 0.001 * i).reshape(-1, 3)
        samples.append(s)
    offs, chrom, p, wei = _concat(samples)
    cs = lib.code_markers(offs, chrom, p, wei)
    assert (len(cs.wtable) > 1024) == wide and (cs.codes32 is None) == wide
    b = lib.Batch(db, offs, chrom, p, wei)
    exact = _run_exact(b)
    pairs = [b.fetch_pairs(i) for i in range(len(samples))]
    for k, i in where.items():                       # the triples the key table sees: those of the matched pairs
        assert _n_triples(samples[i]["wei"][pairs[i][1]]) == k
    raw, guard = _run_coded(lib, b, cs)
    for k, i in where.items():
        if k <= GH_MAX_GROUPS:
            assert guard[i] == 0, "%d triples flagged" % k
            _check_against(raw, _row(exact, i), i)
        else:
            assert guard[i] > 0, "%d triples not flagged" % k
            assert not np.allclose(raw["score"][i], exact["score"][i], rtol=SCORE_RTOL, atol=0)      # folded ids: the flag matters
    for i in (0, 3):
        assert guard[i] == 0
        _check_against(raw, _row(exact, i), i)
    _check_oracle(raw, where[2048], pairs[where[2048]], samples[where[2048]]["wei"], n_acc)
    r = lib.score_coded(db, cs, chrom, p, wei, batch=b)
    rescored = set(r["rescored"].tolist())
    assert rescored == set(np.flatnonzero(guard).tolist()) and {where[2049], where[5000]} <= rescored
    for i in range(len(samples)):
        _check_against(r, _row(exact, i), i, exact_scores=i in rescored)
    _check_oracle(r, where[5000], pairs[where[5000]], samples[where[5000]]["wei"], n_acc)
    b.close()
    db.close()


# ---- 2. one group of GP_MAX_PAIRS pairs ----------------------------------------------------------------------------------
def _all_matched(pos, regions, n, seed):
    rng = np.random.default_rng(seed)
    rows = np.sort(rng.choice(len(pos), size=n, replace=False))
    return dict(chr_ix=np.searchsorted(regions[:, 1], rows, side="right").astype(np.int32), pos=pos[rows].astype(np.int32),
                wei=np.tile([1.0, 0.0, 0.0], (n, 1)), rows=rows)


@pytest.mark.gpu
def test_one_group_of_max_pairs(lib, monkeypatch):
    """A sample of exactly GP_MAX_PAIRS = 65535 markers, all matched, all with one weight triple: the one-CTA grouping's u16 per-warp
    counts and offsets reach 65535.  It must place the pairs as the tiled kernels do (position order inside the one group) and
    score like the popcount kernel bit for bit.  At 65536 markers the one-CTA form no longer fits: the run takes the tiled
    kernels even when the one-CTA form is asked for, with the same results."""
    n_rows, n_acc = 70000, 64
    pos, regions = synth.panel_positions(n_rows)
    db = lib.Database(pos, regions, n_acc)
    db.fill_synthetic(synth.SEED_PANEL)
    for n in (GP_MAX_PAIRS, GP_MAX_PAIRS + 1):
        big = _all_matched(pos, regions, n, seed=n)
        small = synth.make_sample_fast(pos, regions, n_acc, true_acc=9, n_db=700, n_extra=30, seed=4401)
        small["wei"] = synth.hard_weights(small["code"])
        samples = [big, small]
        offs, chrom, p, wei = _concat(samples)
        b = lib.Batch(db, offs, chrom, p, wei)
        ref = _run_exact(b, mode=lib.KERNEL_POPCOUNT)
        ref_pairs = b.fetch_pairs(0)
        assert np.array_equal(ref_pairs[1], np.arange(n)) and int(ref["m"][0]) == n
        cs = lib.code_markers(offs, chrom, p, wei)
        b.set_track_pairs(True)
        got, launches = {}, {}
        for form in ("sample", "tiled"):
            monkeypatch.setenv("SNPM_GROUP_KERNEL", form)
            r, guard = _run_coded(lib, b, cs)
            launches[form] = b.timings()["launches"]
            assert guard.sum() == 0
            for k in ("score", "matches", "ninfo", "m", "prob", "L", "LR"):
                assert np.array_equal(r[k], ref[k], equal_nan=True), (form, k)
            got[form] = b.fetch_pairs(0)
            assert np.array_equal(got[form][0], ref_pairs[0]) and np.array_equal(got[form][1], ref_pairs[1]), form
        # the one-CTA form takes 3 launches for the grouping, the tiled form 7: which form ran is visible in the count
        if n <= GP_MAX_PAIRS:
            assert launches["sample"] < launches["tiled"]
        else:
            assert launches["sample"] == launches["tiled"]
        if n == GP_MAX_PAIRS:
            _check_oracle(ref, 0, ref_pairs, wei[:n], n_acc)
        b.close()
    db.close()


# ---- 3. row shards on one GPU, the exchange done by hand -----------------------------------------------------------------
def _shard_samples(pos, regions, n_acc, third):
    """Six samples: ordinary; pairs only in the first third of the panel (none on later shards); no pairs at all; > 2048 distinct
    triples in the first third but < 100 elsewhere (finished by rank 1 at world 2 and 3); ordinary with the best accession last;
    ordinary."""
    s0 = _sample(pos, regions, n_acc, 5, 4000, 200, 9100)
    s1 = _sample(pos, regions, n_acc, 17, 3000, 100, 9101)
    keep = s1["rows"] < third
    s1 = {k: v[keep] for k, v in s1.items()}
    s2 = _sample(pos, regions, n_acc, 3, 500, 300, 9102)
    s2 = {k: v[s2["rows"] < 0] for k, v in s2.items()}
    s3 = _sample(pos, regions, n_acc, 40, 13000, 200, 9103)
    _with_triples(s3, 3000, 9203, rows_hi=third)
    _with_triples(s3, 50, 9204, rows_lo=third)
    s4 = _sample(pos, regions, n_acc, n_acc - 1, 3500, 100, 9104)
    s5 = _sample(pos, regions, n_acc, 77, 2000, 100, 9105)
    return [s0, s1, s2, s3, s4, s5]


@pytest.mark.gpu
def test_coded_on_row_shards_equals_one_database(lib):
    """The panel cut into world = 2 and 3 SNP-row shards (all on this GPU), each rank grouping and scoring its own rows' pairs;
    the reduce buffers summed by hand as an all-reduce (every rank finishes every sample: the ranks must agree bit for bit,
    guard counts included) and as a reduce-scatter (rank r finishes only its share).  Sample 3 overflows the group table on
    rank 0 only and is finished by rank 1: the overflow must reach rank 1 through the summed buffer and flag it there."""
    import torch
    n_rows, n_acc = 30000, 300
    pos, regions = synth.panel_positions(n_rows)
    third = n_rows // 3
    samples = _shard_samples(pos, regions, n_acc, third)
    S = len(samples)
    OVER = 3
    offs, chrom, p, wei = _concat(samples)
    # one database: the order-exact kernel and the coded path
    db = lib.Database(pos, regions, n_acc)
    db.fill_synthetic(synth.SEED_PANEL)
    b = lib.Batch(db, offs, chrom, p, wei)
    exact = _run_exact(b)
    pairs = [b.fetch_pairs(i) for i in range(S)]
    assert int(exact["m"][2]) == 0 and int(exact["m"][1]) > 0 and pairs[1][0].max() < third
    w3 = samples[OVER]["wei"][pairs[OVER][1]]
    lo = pairs[OVER][0] < third
    assert _n_triples(w3[lo]) > GH_MAX_GROUPS and _n_triples(w3[~lo]) < 100
    full, full_guard = _run_coded(lib, b, lib.code_markers(offs, chrom, p, wei))
    assert np.flatnonzero(full_guard).tolist() == [OVER]
    b.close()
    db.close()
    dev = torch.device("cuda", 0)
    for world in (2, 3):
        share = S // world
        assert OVER // share == 1                                  # rank 1 finishes the overflowing sample
        cuts = [sharding.shard_rows(n_rows, world, r) for r in range(world)]
        assert all(c[0] not in regions.ravel() for c in cuts[1:])  # every cut lies inside a chromosome
        assert cuts[0][1] >= third
        ranks = []
        for r0, r1 in cuts:
            d = lib.Database(pos[r0:r1], sharding.local_regions(regions, r0, r1), n_acc, row0_global=r0)
            d.fill_synthetic(synth.SEED_PANEL)
            sl = []
            for s in samples:
                i0, i1 = sharding.shard_marker_range(s["chr_ix"], s["pos"], regions, pos, r0, r1)
                sl.append({k: s[k][i0:i1] for k in ("chr_ix", "pos", "wei")})
            o, c, pp, w = _concat(sl)
            bb = lib.Batch(d, o, c, pp, w)
            ranks.append((d, bb, lib.code_markers(o, c, pp, w)))

        def run_and_sum():
            views = []
            for d, bb, cs in ranks:
                bb.upload_coded(cs)
                bb.run(kernel_mode=lib.KERNEL_GROUPED)
                ptr, n = bb.reduce_buffer()
                views.append(sharding.device_view(ptr, n, dev))
            torch.cuda.synchronize()
            total = views[0].clone()
            for v in views[1:]:
                total += v
            return views, total

        # (a) all-reduce: every rank finishes every sample
        views, total = run_and_sum()
        for v in views:
            v.copy_(total)
        torch.cuda.synchronize()
        outs = []
        for rank, (d, bb, cs) in enumerate(ranks):
            bb.epilogue()
            res, guard = _copy(bb.fetch()), bb.guard_counts().copy()
            assert guard[OVER] > 0, "world %d, all-reduce: rank %d does not flag the sample that overflowed on rank 0" % (world, rank)
            outs.append((res, guard))
        for res, guard in outs[1:]:
            assert np.array_equal(guard, outs[0][1])
            for k in res:
                assert np.array_equal(res[k], outs[0][0][k], equal_nan=True), k
        allred, allred_guard = outs[0]
        # (b) reduce-scatter: rank r sums and finishes only its rows
        views, total = run_and_sum()
        pitch = views[0].numel() // S
        for rank, v in enumerate(views):
            rows = slice(rank * share * pitch, (rank + 1) * share * pitch)
            v[rows].copy_(total[rows])
        torch.cuda.synchronize()
        parts, guards = [], []
        for rank, (d, bb, cs) in enumerate(ranks):
            bb.set_result_range(rank * share, share)
            bb.epilogue()
            parts.append(_copy(bb.fetch()))
            guards.append(bb.guard_counts().copy())
            bb.set_result_range()
        scat = {k: np.concatenate([x[k] for x in parts]) for k in parts[0]}
        scat_guard = np.concatenate(guards)
        assert scat_guard[OVER] > 0, "world %d, reduce-scatter: rank 1 does not flag the sample that overflowed on rank 0" % world
        for res, guard in ((allred, allred_guard), (scat, scat_guard)):
            assert np.flatnonzero(guard).tolist() == [OVER]
            for i in range(S):
                if i == OVER:
                    continue                 # re-scored by the caller with the order-exact kernel: that is `exact` itself
                _check_against(res, _row(exact, i), i)
                for k in ("matches", "ninfo", "m", "prob"):
                    assert np.array_equal(res[k][i], full[k][i], equal_nan=True), k
                np.testing.assert_allclose(res["score"][i], full["score"][i], rtol=SCORE_RTOL, atol=0)
            assert np.all(np.isnan(res["L"][2])) and int(res["m"][2]) == 0
            assert int(np.nanargmin(res["L"][4])) == n_acc - 1
        _check_oracle(scat, 0, pairs[0], samples[0]["wei"], n_acc)
        _check_oracle(allred, 1, pairs[1], samples[1]["wei"], n_acc)
        for d, bb, cs in ranks:
            bb.close()
            d.close()


def test_overflow_slot_survives_the_host_sum():
    """Host mirror (sharding.finalize_grouped): the overflow slot of one shard, summed with another shard's zero, flags every
    cell of its sample and no other sample."""
    A = 4
    F = np.array([[0.25, 0.375, 1.25, 0.0], [0.75, 0.125, 0.0, 0.25]])      # no sum of two shards is an integer
    I = np.array([[3, 0, 2, 1], [1, 1, 0, 4]])
    ninfo = I + 2
    shard0 = sharding.pack_grouped_rows(F, ninfo, [10, 12], I, overflow=[0, 1])
    shard1 = sharding.pack_grouped_rows(F, ninfo, [10, 12], I)
    assert shard0[:, 2 * A + 1].tolist() == [0.0, 1.0] and shard1[:, 2 * A + 1].tolist() == [0.0, 0.0]
    for total in (shard0 + shard1, shard1 + shard0):
        sc, ma, ni, m, guard = sharding.finalize_grouped(total, A)
        assert guard[1].all() and not guard[0].any()
        assert ma.tolist() == [[6, 0, 6, 2], [3, 2, 0, 8]] and m.tolist() == [20, 24]
    _, _, _, _, guard = sharding.finalize_grouped(shard1 + shard1, A)
    assert not guard.any()


# ---- 4. a second epilogue on the same run --------------------------------------------------------------------------------
@pytest.mark.gpu
def test_second_epilogue_is_refused_on_grouped_batches(lib):
    """k_grouped_finalize turns F into I + F in place, so a second epilogue of a grouped batch on the same run would add I again:
    it is refused (SNPM_E_STATE), also after a first epilogue of a part of the samples, and the results of the first stay.  A
    fresh run allows it again.  Position-order batches may repeat their epilogue and get the same results."""
    n_rows, n_acc = 8000, 40
    pos, regions = synth.panel_positions(n_rows)
    db = lib.Database(pos, regions, n_acc)
    db.fill_synthetic(synth.SEED_PANEL)
    samples = [_sample(pos, regions, n_acc, 3 + 5 * i, 900 + 200 * i, 30, 6600 + i) for i in range(3)]
    offs, chrom, p, wei = _concat(samples)
    b = lib.Batch(db, offs, chrom, p, wei)
    exact = _run_exact(b)
    b.epilogue()                                     # position order: repeatable
    assert all(np.array_equal(v, exact[k], equal_nan=True) for k, v in b.fetch().items())
    b.run()
    b.set_result_range(1, 2)
    b.epilogue()
    b.set_result_range()
    b.epilogue()
    assert all(np.array_equal(v, exact[k], equal_nan=True) for k, v in b.fetch().items())
    cs = lib.code_markers(offs, chrom, p, wei)
    for upload in (lambda: b.upload_coded(cs), lambda: b.upload_grouped(lib.group_markers(offs, chrom, p, wei))):
        upload()
        b.run(kernel_mode=lib.KERNEL_GROUPED)
        b.epilogue()
        first, guard = _copy(b.fetch()), b.guard_counts().copy()
        assert guard.sum() == 0
        for i in range(3):
            _check_against(first, _row(exact, i), i)
        with pytest.raises(lib.SnpmError) as e:
            b.epilogue()
        assert e.value.code == lib.SNPM_E_STATE
        again = b.fetch()
        for k in first:
            assert np.array_equal(again[k], first[k], equal_nan=True), k
        # a part of the samples first, then all of them: the part would be finalised twice
        b.run(kernel_mode=lib.KERNEL_GROUPED)
        b.set_result_range(1, 2)
        b.epilogue()
        part = _copy(b.fetch())
        b.set_result_range()
        with pytest.raises(lib.SnpmError) as e:
            b.epilogue()
        assert e.value.code == lib.SNPM_E_STATE
        for k in first:
            assert np.array_equal(part[k], first[k][1:3], equal_nan=True), k
        b.run(kernel_mode=lib.KERNEL_GROUPED)
        b.epilogue()
        again = b.fetch()
        for k in first:
            assert np.array_equal(again[k], first[k], equal_nan=True), k
    b.close()
    db.close()


# ---- 5. panel widths where the scoring kernel's slices or the epilogue's cluster change ----------------------------------
WIDTHS = [1, 64, 65, 512, 513, 1024, 1025, 1088, 1152, 1153, 2048, 2049]


def _epilogue_cluster(n_acc):
    """CTAs per sample of k_epilogue (csrc/score.cuh launch_epilogue)."""
    e = 1
    while e < 8 and e * 512 < n_acc:
        e *= 2
    return e


def _last_cta_acc(n_acc):
    """The highest accession handled by the last CTA of the epilogue's cluster (CTA e takes the 256-accession stretches e, e + E, ...)."""
    e = _epilogue_cluster(n_acc)
    return max(a for a in range(n_acc) if (a // 256) % e == e - 1)


@pytest.mark.gpu
@pytest.mark.parametrize("n_acc", WIDTHS)
def test_coded_width_sweep(lib, n_acc):
    """Row strides 1..66 words: one slice of WX = 36 or 32 words or of a runtime width (k_score_grouped2), two slices (32 + 6 words,
    32 + 32, 32 + 34), and epilogue clusters of 1, 2 and 4 CTAs.  PL weights: the coded path against the order-exact kernel and
    the oracle; one-hot weights: the coded path, the order-exact kernel and the popcount kernel bit for bit.  The best accession
    sits in the last CTA of the cluster (and at A - 1), and one sample has only nan likelihoods: the cluster's nanmin over
    distributed shared memory."""
    n_rows = 20000
    pos, regions = synth.panel_positions(n_rows)
    db = lib.Database(pos, regions, n_acc)
    db.fill_synthetic(synth.SEED_PANEL)
    tops = [n_acc - 1, _last_cta_acc(n_acc)]
    samples = [_sample(pos, regions, n_acc, t, 2500 - 600 * j, 100, 7300 + j) for j, t in enumerate(tops)]
    zero = _sample(pos, regions, n_acc, 0, 800, 20, 7310)
    zero["wei"][:] = 0.0                             # pairs, informative sites, no match anywhere: every likelihood is nan
    samples.append(zero)
    offs, chrom, p, wei = _concat(samples)
    b = lib.Batch(db, offs, chrom, p, wei)
    cs = lib.code_markers(offs, chrom, p, wei)
    for skip in (False, True):
        exact = _run_exact(b, skip)
        pairs = b.fetch_pairs(0)
        coded = [b]
        if n_acc == 2049 and not skip:               # the smallest group chunk, on a batch of its own (the chunk is latched at upload)
            coded.append(lib.Batch(db, offs, chrom, p, wei))
            coded[1].set_group_chunk(16)
        for bb in coded:
            raw, guard = _run_coded(lib, bb, cs, skip)
            assert guard.sum() <= 1
            for i in np.flatnonzero(guard == 0):
                _check_against(raw, _row(exact, i), i)
        for bb in coded[1:]:
            bb.close()
        b.upload(offs, chrom, p, wei)
        r = lib.score_coded(db, cs, chrom, p, wei, skip, batch=b)
        rescored = set(r["rescored"].tolist())
        for i in range(len(samples)):
            _check_against(r, _row(exact, i), i, exact_scores=i in rescored)
        _check_oracle(r, 0, pairs, samples[0]["wei"], n_acc, skip)
        for i, t in enumerate(tops):
            assert int(np.nanargmin(r["L"][i])) == t and r["LR"][i][t] == 1.0
        assert int(r["m"][2]) > 0 and r["ninfo"][2].max() > 0
        assert np.all(np.isnan(r["L"][2])) and np.all(np.isnan(r["LR"][2]))
        b.upload(offs, chrom, p, wei)
    # one-hot weights: every path counts exactly; the sample without pairs has only nan likelihoods
    hard = [dict(s) for s in samples]
    for s in hard[:2]:
        s["wei"] = synth.hard_weights(s["code"])
    hard[2] = {k: v[samples[2]["rows"] < 0] for k, v in samples[2].items()}
    hard[2]["wei"] = synth.hard_weights(hard[2]["code"])
    offs, chrom, p, wei = _concat(hard)
    b.upload(offs, chrom, p, wei)
    for skip in (False, True):
        pc = _run_exact(b, skip, mode=lib.KERNEL_POPCOUNT)
        fp = _run_exact(b, skip)
        raw, guard = _run_coded(lib, b, lib.code_markers(offs, chrom, p, wei), skip)
        assert guard.sum() == 0
        for k in ("score", "matches", "ninfo", "m", "prob", "L", "LR"):
            assert np.array_equal(fp[k], pc[k], equal_nan=True), k
            assert np.array_equal(raw[k], pc[k], equal_nan=True), k
        assert int(raw["m"][2]) == 0 and np.all(np.isnan(raw["L"][2]))
        for i, t in enumerate(tops):
            assert int(np.nanargmin(raw["L"][i])) == t
        b.upload(offs, chrom, p, wei)
    b.close()
    db.close()
