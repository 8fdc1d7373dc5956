"""The references of tests/test_gpu_cross_limits.py, checked against the oracle without a GPU:

- `f1_reference`, the simulated-F1 sums (csmatch.py:115-126) of every pair of an accession list from one-hot class matrices and
  float64 products, against `orc.f1_pair_scores`;
- `window_panel` / `window_samples`, the panel and samples whose windows reach the edges of the windows run, against
  `orc.window_genotyper` + `orc.window_epilogue`: each promised window is there, and `window_rows_reference` keeps exactly
  the cells the epilogue keeps."""
import numpy as np
import pytest

from oracle import snpmatch_oracle as orc
from snpmatch_b200 import synth

BIN = 300_000
CHR1_WINDOWS = {"all_equal": 2, "all_missing": 4, "one_accession": 6, "one_marker": 8, "dense": 10, "edge": 12}
EMPTY_CHR1 = (3, 5, 7, 9, 11)
DENSE_ROWS = 300


# ---- simulated F1 reference ------------------------------------------------------------------------------------------------
def f1_reference(codes, wei, acc_list):
    """(score f64 [P], ninfo int64 [P]) of every pair i < j of positions in acc_list (itertools.combinations order) over the
    rows of `codes` (int8 [m, A]: 0 ref, 1 alt, 2 het, -1 missing) with the sample weights `wei` [m, 3] (ref, het, alt):
    both hom-alt -> w_alt, both hom-ref -> w_ref, both called and different -> w_het.  With one-hot class matrices O_c [m, U]
    of the distinct accessions: alt = O_1' diag(w_alt) O_1, ref = O_0' diag(w_ref) O_0, het = sum_c O_c' diag(w_het)
    (called - O_c).  With weights of the form k/64 every partial sum is exact, so any summation order gives the same bits."""
    acc_list = np.asarray(acc_list)
    u, inv = np.unique(acc_list, return_inverse=True)
    g = np.asarray(codes)[:, u]
    one = [(g == c).astype(np.float64) for c in (0, 1, 2)]
    called = (g >= 0).astype(np.float64)
    wei = np.asarray(wei, dtype=np.float64)
    w_ref, w_het, w_alt = wei[:, 0:1], wei[:, 1:2], wei[:, 2:3]
    score = one[1].T @ (one[1] * w_alt) + one[0].T @ (one[0] * w_ref)
    count = one[1].T @ one[1] + one[0].T @ one[0]
    for o in one:
        score += o.T @ ((called - o) * w_het)
        count += o.T @ (called - o)
    i, j = np.triu_indices(len(acc_list), 1)
    return score[inv[i], inv[j]], count[inv[i], inv[j]].astype(np.int64)


def dyadic_weights(rng, n):
    """Weights k/64, k in 1..63: sums of up to 2^46 of them are exact in float64."""
    return rng.integers(1, 64, size=(n, 3)) / 64.0


def pl_weights(rng, call):
    """Likelihood-like weights (ref, het, alt): 1.0 for the called class, exp(-PL/10) with PL in 10..90 for the others."""
    w = np.exp(-rng.integers(10, 91, size=(len(call), 3)) / 10.0)
    w[np.arange(len(call)), np.asarray(call)] = 1.0
    return w


def random_codes(rng, n_rows, n_acc, het=0.02, missing=0.05, alt=0.25):
    """int8 panel codes: -1 missing, 2 het, 1 alt, 0 ref with the given shares."""
    lut = np.zeros(100, dtype=np.int8)
    a, b, c = int(round(missing * 100)), int(round((missing + het) * 100)), int(round((missing + het + alt) * 100))
    lut[:a], lut[a:b], lut[b:c] = -1, 2, 1
    return lut[rng.integers(0, 100, size=(n_rows, n_acc), dtype=np.int8)]


# ---- windows panel -----------------------------------------------------------------------------------------------------------
def window_panel(n_acc, n_rows=40_000, seed=11):
    """(positions int32, chr_regions, codes int8 [R, A]) over synth.panel_positions with chromosome 1 rebuilt around its special
    windows (0-based window k covers [k*BIN + 1, (k+1)*BIN]): `dense` holds DENSE_ROWS rows 100 bp apart, `edge` ends with a row
    at 13*BIN and the next window starts with one at 13*BIN + 1; `all_equal` is hom-ref for every accession, `all_missing`
    is missing for every accession."""
    pos, regions = synth.panel_positions(n_rows)
    c0, c1 = int(regions[0][0]), int(regions[0][1])
    p1 = pos[c0:c1].astype(np.int64)
    k = (p1 - 1) // BIN
    edge = (CHR1_WINDOWS["edge"] + 1) * BIN
    p1 = p1[(k != CHR1_WINDOWS["dense"]) & (p1 != edge) & (p1 != edge + 1)]
    dense = CHR1_WINDOWS["dense"] * BIN + 1 + 100 * np.arange(DENSE_ROWS)
    p1 = np.unique(np.concatenate([p1, dense, [edge, edge + 1]]))
    pos = np.concatenate([p1, pos[c1:]]).astype(np.int32)
    delta = len(p1) - (c1 - c0)
    regions = regions.copy()
    regions[0, 1] += delta
    regions[1:] += delta
    rng = np.random.default_rng(seed)
    codes = random_codes(rng, len(pos), n_acc)
    win1 = (p1 - 1) // BIN
    codes[np.flatnonzero(win1 == CHR1_WINDOWS["all_equal"])] = 0
    codes[np.flatnonzero(win1 == CHR1_WINDOWS["all_missing"])] = -1
    # accession A-1 is called on every row of `one_accession`, and every other accession holds the opposite hom on its first
    # three rows: a sample that follows A-1 leaves it alone below the LR threshold there
    one = np.flatnonzero(win1 == CHR1_WINDOWS["one_accession"])
    codes[one, n_acc - 1] = rng.integers(0, 2, size=len(one))
    codes[one[:3], :n_acc - 1] = (1 - codes[one[:3], n_acc - 1])[:, None]
    return pos, regions, codes


def window_samples(pos, regions, codes, seed=21):
    """Three samples [(chrom id int32, pos int32, call int, wei f64 [n, 3])], sorted by (chromosome, position):
    0 follows accession A-1 (the best everywhere), 1 matches no panel row, 2 follows accession (A-1)//2.  A followed sample
    calls what its accession calls (a random hom where that is missing), keeps about 60 % of the rows, none in the chromosome-1
    windows EMPTY_CHR1 or in every fifth window elsewhere, only two rows in every seventh window, exactly one in `one_marker`,
    every row of `dense` and both rows around the `edge`; it also carries markers between panel rows, which join nothing."""
    n_acc = codes.shape[1]
    rng = np.random.default_rng(seed)
    chrom = np.repeat(np.arange(len(regions), dtype=np.int32), regions[:, 1] - regions[:, 0])
    win_local = (pos.astype(np.int64) - 1) // BIN
    counts = np.array([orc.num_windows(l, BIN) for l in synth.TAIR10_CHRLEN])
    gwin = np.concatenate([[0], np.cumsum(counts)])[:-1][chrom] + win_local
    chr1 = chrom == 0
    special = chr1 & np.isin(win_local, list(CHR1_WINDOWS.values()))
    panel_set = set(zip(chrom.tolist(), pos.tolist()))

    def off_panel(n):
        rows = rng.choice(len(pos), size=n, replace=False)
        c, p = chrom[rows], pos[rows].astype(np.int64) + 1
        ok = np.array([(int(a), int(b)) not in panel_set for a, b in zip(c, p)])
        return c[ok], p[ok]

    def follow(acc):
        keep = rng.random(len(pos)) < 0.6
        keep &= ~(chr1 & np.isin(win_local, EMPTY_CHR1))
        keep &= ~(~chr1 & (gwin % 5 == 3))
        few = ~special & (gwin % 7 == 1)
        for w in np.unique(gwin[few]):
            rows = np.flatnonzero(gwin == w)
            keep[rows] = False
            keep[rng.choice(rows, size=min(2, len(rows)), replace=False)] = True
        one = np.flatnonzero(chr1 & (win_local == CHR1_WINDOWS["one_marker"]))
        keep[one] = False
        keep[one[len(one) // 2]] = True
        keep[chr1 & ((win_local == CHR1_WINDOWS["dense"]) | (win_local == CHR1_WINDOWS["one_accession"]))] = True
        edge = (CHR1_WINDOWS["edge"] + 1) * BIN
        keep[chr1 & ((pos == edge) | (pos == edge + 1))] = True
        rows = np.flatnonzero(keep)
        call = codes[rows, acc].astype(np.int64)
        call[call < 0] = rng.integers(0, 2, size=int((call < 0).sum()))
        return rows, call

    out = []
    for acc in (n_acc - 1, None, (n_acc - 1) // 2):
        ec, ep = off_panel(300)
        if acc is None:
            c, p, call = ec, ep, rng.integers(0, 3, size=len(ep))
        else:
            rows, call = follow(acc)
            c = np.concatenate([chrom[rows], ec])
            p = np.concatenate([pos[rows].astype(np.int64), ep])
            call = np.concatenate([call, rng.integers(0, 3, size=len(ep))])
        order = np.lexsort((p, c))
        c, p, call = c[order].astype(np.int32), p[order].astype(np.int32), np.asarray(call)[order]
        cls = np.where(call == 1, 2, np.where(call == 2, 1, 0))      # weight column of the call: ref 0, het 1, alt 2
        out.append((c, p, call, pl_weights(rng, cls)))
    return out


def window_oracle(pos, regions, codes, sample, skip):
    c, p, _, w = sample
    return orc.window_genotyper(codes, np.array(synth.TAIR10_CHRS), regions, pos, np.array(synth.TAIR10_CHRS)[c], p, w,
                                synth.TAIR10_CHRS, synth.TAIR10_CHRLEN, BIN, skip)


def window_rows_reference(w, n_windows):
    """The rows csmatch.get_window_data writes for the oracle's windows (csmatch.py:57-60) in the layout of
    snpm_batch_fetch_window_rows: row_off [W+1], acc, score, ninfo, L, identical, and num_amb [W] (0 for empty windows)."""
    per = {widx: (sc, ni) for widx, sc, ni in w.windows}
    off, num_amb, acc, score, ninfo, lik_rows, ident_rows = [0], np.zeros(n_windows, np.int64), [], [], [], [], []
    for widx in range(1, n_windows + 1):
        if widx in per:
            sc, ni = per[widx]
            lik, _, ident, amb, keep = orc.window_epilogue(sc, ni, 0.02)
            k = np.flatnonzero(keep)
            num_amb[widx - 1] = amb
            acc.append(k); score.append(sc[k]); ninfo.append(ni[k]); lik_rows.append(lik[k]); ident_rows.append(ident[k])
        off.append(off[-1] + (len(acc[-1]) if widx in per else 0))
    cat = (lambda x, t: np.concatenate(x).astype(t) if x else np.zeros(0, t))
    return {"row_off": np.array(off, np.int64), "num_amb": num_amb, "acc": cat(acc, np.int64), "score": cat(score, np.float64),
            "ninfo": cat(ninfo, np.int64), "L": cat(lik_rows, np.float64), "identical": cat(ident_rows, np.int64)}


# ---- tests -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_acc", [1, 40, 97])
def test_f1_reference_equals_the_oracle(n_acc):
    rng = np.random.default_rng(n_acc)
    m = 700
    codes = random_codes(rng, m, n_acc, het=0.1)
    lists = [np.arange(min(n_acc, 10)), rng.integers(0, n_acc, size=17), np.array([0, n_acc - 1, 0, n_acc // 2])]
    for acc_list in lists:
        if len(acc_list) < 2:
            continue
        common = (np.arange(m), rng.permutation(m))
        for wei, exact in ((dyadic_weights(rng, m), True), (pl_weights(rng, rng.integers(0, 3, size=m)), False)):
            _, o_score, o_ninfo = orc.f1_pair_scores(codes, common, wei, acc_list)
            score, ninfo = f1_reference(codes[common[0]], wei[common[1]], acc_list)
            assert np.array_equal(ninfo, o_ninfo)
            if exact:
                assert np.array_equal(score, o_score)
            else:
                np.testing.assert_allclose(score, o_score, rtol=1e-12, atol=0)


def test_f1_reference_counts_het_het_as_equal():
    codes = np.array([[2, 2, 0, -1], [2, 0, 1, 1], [1, 1, -1, 1]], dtype=np.int8)
    wei = np.array([[1, 2, 4], [8, 16, 32], [64, 128, 256]], dtype=np.float64) / 64
    score, ninfo = f1_reference(codes, wei, [0, 1, 2, 3])
    _, o_score, o_ninfo = orc.f1_pair_scores(codes, (np.arange(3), np.arange(3)), wei, [0, 1, 2, 3])
    assert np.array_equal(score, o_score) and np.array_equal(ninfo, o_ninfo)
    assert ninfo[0] == 2 and score[0] == (256 + 16) / 64          # (0, 1): het/het is not counted, het/ref is, alt/alt is


@pytest.mark.parametrize("n_acc", [1, 40, 257])
def test_window_panel_has_the_promised_windows(n_acc):
    pos, regions, codes = window_panel(n_acc, n_rows=12_000)
    assert np.all(np.diff(pos[regions[0][0]:regions[0][1]]) > 0)
    samples = window_samples(pos, regions, codes)
    n_w = sum(orc.num_windows(l, BIN) for l in synth.TAIR10_CHRLEN)
    for skip in (False, True):
        ws = [window_oracle(pos, regions, codes, s, skip) for s in samples]
        assert ws[1].num_snps == 0 and not ws[1].windows
        for w in (ws[0], ws[2]):
            per = {widx - 1: (sc, ni) for widx, sc, ni in w.windows}
            for k in EMPTY_CHR1:
                assert k not in per
            assert all(k in per for k in CHR1_WINDOWS.values()) and CHR1_WINDOWS["edge"] + 1 in per
            amb = {k: orc.window_epilogue(sc, ni)[3] for k, (sc, ni) in per.items()}
            sc, ni = per[CHR1_WINDOWS["all_equal"]]
            assert np.array_equal(sc, ni) and amb[CHR1_WINDOWS["all_equal"]] == n_acc
            assert amb[CHR1_WINDOWS["all_missing"]] == 0
            assert not per[CHR1_WINDOWS["all_missing"]][1].any()
            assert per[CHR1_WINDOWS["one_marker"]][1].max() <= 1
            assert per[CHR1_WINDOWS["dense"]][1].max() >= 257
            rows = window_rows_reference(w, n_w)
            assert np.array_equal(rows["num_amb"][[k for k in per]], [amb[k] for k in per])
            kept = np.diff(rows["row_off"])
            assert kept[CHR1_WINDOWS["all_equal"]] == 0
            if n_acc > 1:
                assert (np.diff(rows["row_off"]) > 0).any()
        # the sample that follows accession A-1: it is the best, and alone below the threshold in `one_accession`
        w = ws[0]
        lik, _ = orc.calculate_likelihoods(w.tot_score, w.tot_ninfo)
        assert int(np.nanargmin(lik)) == n_acc - 1
        per = {widx - 1: (sc, ni) for widx, sc, ni in w.windows}
        _, _, _, amb, keep = orc.window_epilogue(*per[CHR1_WINDOWS["one_accession"]])
        assert amb == 1 and (n_acc == 1 or np.flatnonzero(keep).tolist() == [n_acc - 1])
        if n_acc > 1:
            # windows that keep accessions on both sides of 256 (two passes of the compaction loop)
            rows = window_rows_reference(w, n_w)
            if n_acc > 256:
                spans = [(rows["acc"][a:b].min(), rows["acc"][a:b].max()) for a, b in zip(rows["row_off"][:-1], rows["row_off"][1:]) if b > a]
                assert any(lo < 256 <= hi for lo, hi in spans)
