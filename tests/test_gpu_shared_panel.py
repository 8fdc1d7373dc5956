"""The batched shared-panel mode (snpm_panel_* / snpm_score_shared_panel, csrc/gemm_onehot.cuh) where its tcgen05 GEMM changes
behaviour: the persistent tile loop past one tile per CTA (both TMEM accumulators, the accumulator hand-back waits, k-block ring
stages and phases carried from one tile to the next), tile and k-block edges of S, A and K, codes outside 0-3 in both wire
forms, panel rows that repeat or sit on a row shard, scratch re-use across batch sizes, the largest batches the API takes, and a
second GPU in the same process.

Reference: plain NumPy.  With P the panel's codes (hets -1 when skip_db_hets) and C the sample codes (every code >= 3 absent),
score = sum_{c in 0,1,2} [C == c] @ [P == c] and ninfo = [C < 3] @ [P >= 0].  Every partial sum is an integer below 2^24, so the
float32 products are exact.  In every case a few samples (first, last, both sides of the 64-sample tile boundaries) are also
compared with the oracle's matchGTsAccs directly.  Bars: matches and ninfo == on every sample; L and LR rtol 1e-9 against
orc.calculate_likelihoods (every sample, except a fixed subset of the 4 M-sample batch)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import snpmatch_oracle as orc
from snpmatch_b200 import sharding, synth

RTOL = 1e-9
OG_BM, OG_BN, OG_ROWS = 64, 256, 32          # samples per M-tile, accessions per N-tile, markers per k-block (gemm_onehot.cuh)
MAX_S = 65535 * 64                           # SNPM_PANEL_MAX_SAMPLES
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


def _db(lib, n_acc, n_rows=20000, r0=0, r1=None):
    pos, regions = synth.panel_positions(n_rows)
    if r1 is None:
        db = lib.Database(pos, regions, n_acc)
    else:
        db = lib.Database(pos[r0:r1], sharding.local_regions(regions, r0, r1), n_acc, row0_global=r0)
    db.fill_synthetic(synth.SEED_PANEL)
    return db


def _codes(rng, S, K, p=(0.45, 0.3, 0.1, 0.15)):
    return rng.choice(np.array([0, 1, 2, 3], dtype=np.uint8), size=(S, K), p=list(p))


def _tiles(S, A):
    return -(-S // OG_BM) * -(-A // OG_BN)


def _n_kb(K):
    return max(1, -(-K // OG_ROWS))


def _reference(P, C):
    """score, ninfo int64 [S, A] as products of one-hot indicator matrices (exact: integer partial sums below 2^24)."""
    assert C.shape[1] < (1 << 24)
    f = np.float32
    score = np.zeros((C.shape[0], P.shape[1]), f)
    for c in (0, 1, 2):
        score += (C == c).astype(f) @ (P == c).astype(f)
    ninfo = (C < 3).astype(f) @ (P >= 0).astype(f)
    return score.astype(np.int64), ninfo.astype(np.int64)


def _likelihoods(score, ninfo):
    """orc.calculate_likelihoods on every row at once: the oracle's elementwise L (a fixed amin of 1 leaves LR = L), each row's
    nanmin as its amin (the "calc" branch)."""
    lik, _ = orc.calculate_likelihoods(score, ninfo, amin=1.0)
    ok = ~np.all(np.isnan(lik), axis=1)
    top = np.full(len(lik), np.nan)
    top[ok] = np.nanmin(lik[ok], axis=1)
    with np.errstate(invalid="ignore"):
        lr = np.where((top > 0)[:, None], lik / np.where(top > 0, top, 1.0)[:, None], np.nan)
    return lik, lr


def _pins(S, every_boundary=True):
    """First, last and both sides of the 64-sample boundaries (only the first and the last boundary when every_boundary=False)."""
    b = list(range(OG_BM, S, OG_BM))
    if not every_boundary:
        b = b[:1] + b[-1:]
    return sorted({0, S - 1} | {x for j in b for x in (j - 1, j)})


def _pin_oracle(score, ninfo, P0, C, skip, pins):
    """The NumPy reference against matchGTsAccs (one-hot weights of the sample's called markers) and calculateLikelihoods."""
    lik, lr = _likelihoods(score[pins], ninfo[pins])
    for i, s in enumerate(pins):
        have = np.flatnonzero(C[s] < 3)
        sc, ni = orc.match_gts_accs(synth.hard_weights(C[s][have].astype(np.int8)), P0[have], skip)
        assert np.array_equal(score[s], sc.astype(np.int64)) and np.array_equal(ninfo[s], ni), "reference != oracle, sample %d" % s
        ol, olr = orc.calculate_likelihoods(sc.astype(np.int64), ni)
        assert np.array_equal(lik[i], ol, equal_nan=True) and np.array_equal(lr[i], olr, equal_nan=True), "sample %d" % s


def _assert_rows(got, want, what):
    bad = np.flatnonzero((np.asarray(got) != want).any(axis=1))
    assert len(bad) == 0, "%s differs on %d of %d samples, first %s" % (what, len(bad), len(want), bad[:8].tolist())


class Ref(object):
    """The reference of one (panel, codes) pair, pinned to the oracle once."""

    def __init__(self, rows, n_acc, skip, C, pins=None, likelihoods=True):
        P0 = synth.panel_codes(synth.SEED_PANEL, rows, n_acc)
        P = P0.copy()
        if skip:
            P[P == 2] = -1
        self.score, self.ninfo = _reference(P, C)
        _pin_oracle(self.score, self.ninfo, P0, C, skip, _pins(len(C)) if pins is None else pins)
        self.lik = _likelihoods(self.score, self.ninfo) if likelihoods else None

    def check(self, r, what="", likelihoods=True):
        _assert_rows(r["matches"], self.score, "matches " + what)
        _assert_rows(r["ninfo"], self.ninfo, "ninfo " + what)
        if likelihoods:
            np.testing.assert_allclose(r["L"], self.lik[0], rtol=RTOL, equal_nan=True, err_msg="L " + what)
            np.testing.assert_allclose(r["LR"], self.lik[1], rtol=RTOL, equal_nan=True, err_msg="LR " + what)


def _packed_with_garbage(lib, rng, C):
    """pack_codes2 with random bits in the spare bit pairs of each row's last byte (zeros there would read as ref calls)."""
    pk = lib.pack_codes2(C)
    K = C.shape[1]
    if K % 4:
        spare = np.uint8((0xFF << (2 * (K % 4))) & 0xFF)
        pk[:, -1] = (pk[:, -1] & ~spare) | (rng.integers(0, 256, size=len(pk)).astype(np.uint8) & spare)
    return pk


# ---- the persistent schedule -----------------------------------------------------------------------------------------------


def _schedule_shapes(n_sm):
    """(name, S, A, K, tiles per CTA at most) reaching the tile counts the persistent loop changes behaviour at."""
    d = 2 if n_sm % 2 == 0 else 1
    s_big = OG_BM * -(-(4 * n_sm + 1) // 79) - 3
    return [
        ("tiles = SMs", OG_BM * d - 5, OG_BN * (n_sm // d) - 7, 100, 1),
        ("tiles = SMs + 1, one-accession last N-tile", 37, OG_BN * n_sm + 1, 200, 2),
        ("5 tiles per CTA, 10 k-blocks", s_big, 20000, 301, 5),
        ("5 tiles per CTA, 5 k-blocks", s_big, 20000, 157, 5),
    ]


@pytest.mark.gpu
def test_persistent_schedule_past_one_tile_per_cta(lib):
    n_sm = lib.device_info(0)["n_sm"]
    rng = np.random.default_rng(101)
    shapes = _schedule_shapes(n_sm)
    assert _tiles(shapes[0][1], shapes[0][2]) == n_sm
    assert _tiles(shapes[1][1], shapes[1][2]) == n_sm + 1 and -(-shapes[1][1] // OG_BM) == 1 and shapes[1][2] % OG_BN == 1
    assert _tiles(shapes[2][1], shapes[2][2]) >= 4 * n_sm + 1 and shapes[2][1] % OG_BM != 0
    assert _n_kb(shapes[2][3]) == 10 and _n_kb(shapes[3][3]) == 5       # n_kb mod 4 = 2 and 1: tiles start on every stage
    dbs = {}
    for name, S, A, K, per_cta in shapes:
        assert -(-_tiles(S, A) // n_sm) == per_cta, name
        if A not in dbs:
            dbs[A] = _db(lib, A)
        db = dbs[A]
        rows = rng.choice(db.n_rows, size=K, replace=False)
        C = _codes(rng, S, K)
        ref = Ref(rows, A, False, C, pins=_pins(S, every_boundary=A <= 2048))
        sp = db.shared_panel(rows)
        ref.check(sp.score(C, likelihoods=True), name + " plain")
        ref.check(sp.score(_packed_with_garbage(lib, rng, C), packed=True, likelihoods=True), name + " packed")
        if per_cta == 5 and K == 157:
            one = db.score_shared_panel(rows, C)                   # the one-shot form (int64 results) at a multi-tile shape
            assert one["matches"].dtype == np.int64
            ref.check(one, name + " one-shot")
        sp.close()
    for db in dbs.values():
        db.close()


@pytest.mark.gpu
def test_bench_configs3_every_sample(lib):
    """BASELINE configs[3] in full: 4096 samples x 20 000 shared markers x 1135 accessions, packed codes; bench.py compares two
    samples with the oracle, this compares all of them with the reference."""
    S, K, A = 4096, 20000, 1135
    db = _db(lib, A)
    rng = np.random.default_rng(9)
    rows = np.sort(rng.choice(db.n_rows, size=K, replace=False))
    C = _codes(rng, S, K, p=(0.6, 0.28, 0.02, 0.1))
    ref = Ref(rows, A, False, C, pins=_pins(S, every_boundary=False))
    sp = db.shared_panel(rows)
    ref.check(sp.score(lib.pack_codes2(C), packed=True, likelihoods=True), "configs[3]")
    sp.close()
    db.close()


# ---- tile and k-block edges --------------------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("A", [1, 255, 256, 257, 513])
def test_tile_and_kblock_edges(lib, A):
    """S on both sides of the 64-sample M-tile, A of the 256-accession N-tile, K of the 32-marker k-block and of the packed
    byte (K % 32 in 29-31: the packed rows fill the k-block and only the tail kernel clears the spare bits; K = 0: no markers)."""
    db = _db(lib, A, n_rows=3000)
    rng = np.random.default_rng(1000 + A)
    for K in (0, 1, 3, 4, 5, 29, 31, 32, 33, 128, 129):
        rows = rng.choice(db.n_rows, size=K, replace=True)
        for skip in (False, True):
            sp = db.shared_panel(rows, skip_db_hets=skip)
            for S in (129, 1, 64, 63, 128, 65):                       # grows and shrinks: the panel's scratch is re-used
                C = _codes(rng, S, K)
                ref = Ref(rows, A, skip, C)
                what = "A=%d K=%d skip=%d S=%d" % (A, K, skip, S)
                ref.check(sp.score(C, likelihoods=True), what + " plain")
                ref.check(sp.score(_packed_with_garbage(lib, rng, C), packed=True, likelihoods=True), what + " packed")
            sp.close()
    db.close()


# ---- codes outside 0-3 -------------------------------------------------------------------------------------------------------


def test_pack_codes2_codes_past_3_are_absent():
    """Every code >= 3 means absent in the unpacked form, so it packs as 3; 0-2 keep their value; the spare bits read 3."""
    from snpmatch_b200 import lib as L
    codes = np.arange(256, dtype=np.uint8).reshape(1, -1)
    pk = L.pack_codes2(codes)
    assert pk.shape == (1, 64)
    got = np.stack([(pk[0] >> (2 * j)) & 3 for j in range(4)], axis=1).ravel()
    assert np.array_equal(got, np.minimum(codes[0], 3))
    assert np.array_equal(L.pack_codes2(np.array([[4, 5, 6, 7], [0, 1, 2, 255]], np.uint8)), np.array([[0xFF], [0xE4]], np.uint8))
    rng = np.random.default_rng(5)
    for K in (1, 2, 3, 5, 31):
        c = rng.integers(0, 256, size=(7, K), dtype=np.uint8)
        pk = L.pack_codes2(c)
        assert pk.shape == (7, (K + 3) // 4)
        got = np.stack([(pk >> (2 * j)) & 3 for j in range(4)], axis=2).reshape(7, -1)
        assert np.array_equal(got[:, :K], np.minimum(c, 3)) and np.all(got[:, K:] == 3)


@pytest.mark.gpu
def test_codes_outside_0_to_3_are_absent_in_both_forms(lib):
    A, K, S = 300, 77, 130
    db = _db(lib, A)
    rng = np.random.default_rng(44)
    rows = rng.choice(db.n_rows, size=K, replace=False)
    C = np.where(rng.random((S, K)) < 0.5, rng.integers(0, 3, size=(S, K)), rng.integers(3, 256, size=(S, K))).astype(np.uint8)
    C[0] = np.arange(K) % 8                                           # 4-7 would read as 0-3 if only the low bits were kept
    for skip in (False, True):
        ref = Ref(rows, A, skip, C)
        sp = db.shared_panel(rows, skip_db_hets=skip)
        ref.check(sp.score(C, likelihoods=True), "plain")
        ref.check(sp.score(lib.pack_codes2(C), packed=True, likelihoods=True), "packed")
        ref.check(db.score_shared_panel(rows, C, skip_db_hets=skip), "one-shot")
        sp.close()
    db.close()


# ---- panel rows --------------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_unsorted_rows_with_repeats(lib):
    A = 257
    db = _db(lib, A)
    rng = np.random.default_rng(55)
    rows = rng.choice(db.n_rows, size=150, replace=True)
    rows[100:140] = rows[:40]                                         # forty rows twice (or more)
    rng.shuffle(rows)
    assert len(np.unique(rows)) < len(rows) and np.any(np.diff(rows) < 0)
    for skip in (False, True):
        C = _codes(rng, 130, len(rows))
        sp = db.shared_panel(rows, skip_db_hets=skip)
        Ref(rows, A, skip, C).check(sp.score(_packed_with_garbage(lib, rng, C), packed=True, likelihoods=True), "skip=%d" % skip)
        sp.close()
    # a repeated row counts twice: the panel [r, r] scores twice what [r] scores
    r = np.array([int(rows[0])], np.int64)
    C = _codes(rng, 65, 1)
    one = db.shared_panel(r).score(C)
    two = db.shared_panel(np.concatenate([r, r])).score(np.concatenate([C, C], axis=1))
    assert np.array_equal(two["matches"], 2 * one["matches"]) and np.array_equal(two["ninfo"], 2 * one["ninfo"])
    db.close()


@pytest.mark.gpu
def test_row_shard_database(lib):
    """A database holding global rows [r0, r1): panels on those rows give the whole-panel answer; a row outside is refused."""
    A, n_rows, r0, r1 = 300, 20000, 7000, 13000
    full, shard = _db(lib, A, n_rows), _db(lib, A, n_rows, r0, r1)
    rng = np.random.default_rng(66)
    rows = rng.choice(np.arange(r0, r1), size=200, replace=False)
    rows[:2] = (r0, r1 - 1)
    C = _codes(rng, 129, len(rows))
    for skip in (False, True):
        ref = Ref(rows, A, skip, C)
        got = shard.shared_panel(rows, skip_db_hets=skip).score(C, likelihoods=True)
        ref.check(got, "shard skip=%d" % skip)
        whole = full.shared_panel(rows, skip_db_hets=skip).score(C, likelihoods=True)
        for k in ("matches", "ninfo", "L", "LR"):
            assert np.array_equal(got[k], whole[k], equal_nan=True), k
        ref.check(shard.score_shared_panel(rows, C, skip_db_hets=skip), "shard one-shot skip=%d" % skip)
    for bad in (r0 - 1, r1, n_rows + 5):
        with pytest.raises(lib.SnpmError):
            lib.SharedPanel(shard, np.array([r0 + 1, bad], np.int64))
        with pytest.raises(lib.SnpmError):
            shard.score_shared_panel(np.array([bad], np.int64), np.zeros((3, 1), np.uint8))
    shard.close()
    full.close()


# ---- scratch re-use ----------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_scratch_reuse_across_batch_sizes_and_panels(lib):
    A = 300
    db = _db(lib, A)
    rng = np.random.default_rng(77)
    rows = rng.choice(db.n_rows, size=157, replace=False)
    sp = db.shared_panel(rows)
    for S in (509, 1, 130, 65600, 64):                                # 65 600: samples past the 65 535 of a grid's y
        C = _codes(rng, S, len(rows))
        ref = Ref(rows, A, False, C, pins=_pins(S, every_boundary=S < 4096))
        ref.check(sp.score(C, likelihoods=True), "S=%d plain" % S)
        ref.check(sp.score(_packed_with_garbage(lib, rng, C), packed=True, likelihoods=True), "S=%d packed" % S)
    sp.close()
    # two panels of different K and skip on one database, scored alternately
    rows2 = rng.choice(db.n_rows, size=301, replace=True)
    p1, p2 = db.shared_panel(rows), db.shared_panel(rows2, skip_db_hets=True)
    for S in (200, 70, 3):
        for rw, skip, p in ((rows, False, p1), (rows2, True, p2)):
            C = _codes(rng, S, len(rw))
            Ref(rw, A, skip, C).check(p.score(C, likelihoods=True), "K=%d S=%d" % (len(rw), S))
    p1.close()
    p2.close()
    db.close()


# ---- the largest batches -----------------------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_batch_past_65535_samples(lib):
    """More samples than a grid's y dimension holds, with and without the likelihood epilogue."""
    A, K, S = 300, 90, 65600
    db = _db(lib, A)
    rng = np.random.default_rng(88)
    rows = rng.choice(db.n_rows, size=K, replace=False)
    C = _codes(rng, S, K)
    ref = Ref(rows, A, False, C, pins=_pins(S, every_boundary=False))
    ref.check(db.score_shared_panel(rows, C, likelihoods=True), "one-shot, likelihoods")
    ref.check(db.score_shared_panel(rows, C, likelihoods=False), "one-shot, integers", likelihoods=False)
    sp = db.shared_panel(rows)
    ref.check(sp.score(lib.pack_codes2(C), packed=True, likelihoods=True), "packed, likelihoods")
    ref.check(sp.score(lib.pack_codes2(C), packed=True), "packed, integers", likelihoods=False)
    sp.close()
    db.close()


@pytest.mark.gpu
def test_largest_batch_and_the_bound(lib):
    """S = 65 535 x 64 = 4 194 240, the largest batch the API takes (one accession, 5 markers, packed; about 10 GB of device
    memory): integers on every sample, likelihoods on a fixed subset.  One sample more is refused before any device work."""
    S, K, A = MAX_S, 5, 1
    db = _db(lib, A)
    rng = np.random.default_rng(99)
    rows = rng.choice(db.n_rows, size=K, replace=False)
    C = _codes(rng, S, K)
    pk = lib.pack_codes2(C)
    sp = db.shared_panel(rows)
    with pytest.raises(lib.SnpmError):
        sp.score(np.zeros((S + 1, 2), np.uint8), packed=True)
    with pytest.raises(lib.SnpmError):
        db.score_shared_panel(rows, np.zeros((S + 1, K), np.uint8))
    ref = Ref(rows, A, False, C, pins=_pins(S, every_boundary=False), likelihoods=False)
    r = sp.score(pk, packed=True, likelihoods=True)
    ref.check(r, "S=%d" % S, likelihoods=False)
    sub = np.unique(np.concatenate([[0, 1, 63, 64, S - 65, S - 64, S - 1], rng.integers(0, S, size=400)]))
    lik, lr = _likelihoods(ref.score[sub], ref.ninfo[sub])
    np.testing.assert_allclose(r["L"][sub], lik, rtol=RTOL, equal_nan=True)
    np.testing.assert_allclose(r["LR"][sub], lr, rtol=RTOL, equal_nan=True)
    sp.close()
    db.close()


# ---- a second GPU in the same process ----------------------------------------------------------------------------------------

_WORKER = r"""
import os, sys
import numpy as np
from snpmatch_b200 import lib, synth

order, out = [int(x) for x in sys.argv[1].split(",")], sys.argv[2]
n_rows, n_acc = 30000, 1135
pos, regions = synth.panel_positions(n_rows)
rng = np.random.default_rng(12)
rows = rng.choice(n_rows, size=301, replace=False)
codes = rng.choice(np.array([0, 1, 2, 3], np.uint8), size=(130, len(rows)), p=[0.45, 0.3, 0.1, 0.15])
samples = [synth.make_sample_fast(pos, regions, n_acc, true_acc=5 + 17 * i, n_db=6000, n_extra=500, seed=4400 + i) for i in range(5)]
offs = np.concatenate([[0], np.cumsum([len(s["pos"]) for s in samples])])
chrom = np.concatenate([s["chr_ix"] for s in samples]).astype(np.int32)
p = np.concatenate([s["pos"] for s in samples]).astype(np.int32)
wei = np.concatenate([s["wei"] for s in samples])
hard = synth.hard_weights(np.concatenate([s["code"] for s in samples]))
res = {}
for dev in order:
    db = lib.Database(pos, regions, n_acc, device=dev)
    db.fill_synthetic(synth.SEED_PANEL)
    sp = db.shared_panel(rows)
    r = sp.score(codes, likelihoods=True)
    for k in ("matches", "ninfo", "L", "LR"):
        res["%d_panel_%s" % (dev, k)] = r[k]
    def keep(tag, b):
        for k, v in b.fetch().items():
            res["%d_%s_%s" % (dev, tag, k)] = np.array(v, copy=True)
    b = lib.Batch(db, offs, chrom, p, wei)
    b.run(kernel_mode=lib.KERNEL_FP64); b.epilogue(); keep("segments", b)
    b.close()
    b = lib.Batch(db, offs, chrom, p, hard)
    b.run(kernel_mode=lib.KERNEL_POPCOUNT); b.epilogue(); keep("hard", b)
    b.close()
    b = lib.Batch(db, offs, chrom, p, wei)
    cs = lib.code_markers(offs, chrom, p, wei)
    for form in ("sample", "tiled"):
        os.environ["SNPM_GROUP_KERNEL"] = form
        b.upload_coded(cs); b.run(kernel_mode=lib.KERNEL_GROUPED); b.epilogue(); keep("coded_" + form, b)
    del os.environ["SNPM_GROUP_KERNEL"]
    b.upload_grouped(lib.group_markers(offs, chrom, p, wei)); b.run(kernel_mode=lib.KERNEL_GROUPED); b.epilogue(); keep("grouped", b)
    b.close()
    sp.close()
    db.close()
np.savez(out, **res)
"""


@pytest.mark.gpu
def test_second_gpu_in_one_process(lib, tmp_path):
    """Kernels that ask for more than 48 KB of dynamic shared memory need the attribute in every device's context.  A fresh
    process (no earlier test has set anything) scores on device 0 then device 1, another on 1 then 0: the shared-panel GEMM,
    the order-exact and popcount kernels of position-order batches, coded batches with both device groupings, a host-grouped
    upload.  Every device gives the same bits."""
    if lib.device_count() < 2:
        pytest.skip("needs two GPUs")
    got = []
    for order in ("0,1", "1,0"):
        out = str(tmp_path / ("order_%s.npz" % order.replace(",", "")))
        env = dict(os.environ)
        env.pop("SNPM_GROUP_KERNEL", None)
        proc = subprocess.run([sys.executable, "-c", _WORKER, order, out], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
        assert proc.returncode == 0, "device order %s:\n%s" % (order, proc.stderr[-3000:])
        got.append(dict(np.load(out)))
    base = {k[2:]: v for k, v in got[0].items() if k.startswith("0_")}
    assert {k.split("_")[0] for k in base} >= {"panel", "segments", "hard", "coded", "grouped"}
    for run in got:
        for dev in (0, 1):
            for k, v in base.items():
                assert np.array_equal(run["%d_%s" % (dev, k)], v, equal_nan=True), "device %d: %s" % (dev, k)
