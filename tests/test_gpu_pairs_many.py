"""`pairsnp --samples` on the GPU: every pair of many samples in one tensor-core pass (lib.pair_matrix,
core.snpmatch.pairwise_score_many).  Checked against (a) pairwiseScore on the same files, pair by pair, and (b) a NumPy
oracle in this file: dense per-chromosome presence and one-hot matrices multiplied.  All counts are integers: exact."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_golden

pytestmark = pytest.mark.gpu

GT_OF_CODE = np.array(["./.", "0/0", "1/1", "0/1"])          # panel code + 1 -> GT string


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


def _stats_equal(got, want):
    """tests/test_gpu_pairs.py's rules; a nan on either side (None in JSON) equals a nan."""
    def same(a, b):
        return a == b or ((b is None or (isinstance(b, float) and np.isnan(b))) and np.isnan(a))
    assert sorted(got) == sorted(want)
    for k, v in want.items():
        if k == "hdf5":
            assert got[k] == v
        elif k == "unique":
            assert sorted(got[k]) == sorted(v)
            for name in v:
                assert got[k][name][1] == v[name][1]
                assert same(got[k][name][0], v[name][0])
        else:
            assert got[k][1] == v[1], k
            assert same(got[k][0], v[0]), k


def _oracle(samples, db=None):
    """(chromosomes, common, same) [C,S,S] from dense matrices: samples = [(chrs, pos, gt)]; db = set of (normalised chromosome,
    position) that count, or None."""
    import re
    norm = [np.array([re.sub("chr", "", str(c), flags=re.IGNORECASE) for c in s[0]]) for s in samples]
    chroms = np.unique(np.concatenate([n for n in norm] + [np.zeros(0, "U1")]))
    S = len(samples)
    keys, strings = {}, {}
    rows = []
    for n, (_, pos, gt) in zip(norm, samples):
        r = {}
        for c, p, g in zip(n, np.asarray(pos).tolist(), np.asarray(gt).astype("U").tolist()):
            if db is None or (c, p) in db:
                r[(c, p)] = strings.setdefault(g, len(strings))
                keys.setdefault((c, p), None)
        rows.append(r)
    cols = sorted(keys)
    col_of = {k: i for i, k in enumerate(cols)}
    G = np.full((S, len(cols)), -1, np.int64)
    for s, r in enumerate(rows):
        for k, v in r.items():
            G[s, col_of[k]] = v
    chr_of = np.array([np.searchsorted(chroms, c) for c, _ in cols], np.int64)
    common = np.zeros((len(chroms), S, S), np.int64)
    same = np.zeros((len(chroms), S, S), np.int64)
    for c in range(len(chroms)):
        Gc = G[:, chr_of == c]
        P = (Gc >= 0).astype(np.float64)
        common[c] = np.rint(P @ P.T).astype(np.int64)
        for v in range(len(strings)):
            H = (Gc == v).astype(np.float64)
            same[c] += np.rint(H @ H.T).astype(np.int64)
    return chroms, common, same


def _check_oracle(pm, samples, db=None):
    chroms, common, same = _oracle(samples, db)
    assert pm.chromosomes.tolist() == chroms.tolist()
    assert np.array_equal(pm.common, common)
    assert np.array_equal(pm.same, same)


def _write(tmp_path, tag, chrs, pos, gt):
    f = str(tmp_path / ("%s.npz" % tag))
    np.savez(f, chr=np.asarray(chrs), pos=np.asarray(pos), gt=np.asarray(gt), wei=np.ones((len(pos), 3)), dp=np.ones(len(pos)))
    return f


def _golden_files(tmp_path):
    g = load_golden("pairsnp.npz")
    files, samples = [], []
    for i in range(int(g["n_cases"])):
        for side, tag in (("1", "a"), ("2", "b")):
            c, p, gt = g["p%d_c%s" % (i, side)], g["p%d_p%s" % (i, side)], g["p%d_g%s" % (i, side)]
            files.append(_write(tmp_path, "s%d_%s" % (i, tag), c, p, gt))
            samples.append((c, p, gt))
    return files, samples


def _db_keys(panel):
    chrs = np.repeat(panel["chrs"].astype("U"), np.diff(panel["chr_regions"], axis=1).ravel())
    return set(zip(chrs.tolist(), panel["positions"].tolist()))


def _simulated(panel, S, per, seed, n_strings=4, prefixes=("Chr", "chr", "", "CHR")):
    """S samples drawn from the small panel like `simulate` draws them: rows of one accession, GT strings of its calls (no-calls
    included), chromosome names with a per-sample prefix; a few phased calls and calls from outside the panel."""
    rng = np.random.default_rng(seed)
    chr_of_row = np.repeat(panel["chrs"].astype("U"), np.diff(panel["chr_regions"], axis=1).ravel())
    out = []
    strings = np.array(["./.", "0/0", "1/1", "0/1", "1|1", "0|1", "1|0", "0|0"])[:max(n_strings, 1)]
    for s in range(S):
        n = int(rng.integers(0, per + 1)) if s % 7 == 3 else per
        rows = np.sort(rng.choice(len(panel["positions"]), size=min(n, len(panel["positions"])), replace=False))
        acc = int(rng.integers(0, panel["snps"].shape[1]))
        gt = GT_OF_CODE[panel["snps"][rows, acc] + 1]
        gt = np.where(np.isin(gt, strings), gt, strings[0])
        flip = rng.random(len(rows)) < 0.1
        gt = np.where(flip, strings[rng.integers(0, len(strings), size=len(rows))], gt)
        pos = panel["positions"][rows].astype(np.int64)
        extra = rng.random(len(rows)) < 0.05                  # positions the panel does not have
        pos = np.where(extra, pos + 1, pos)
        keep = np.ones(len(pos), bool)
        keep[1:] = pos[1:] != pos[:-1]
        chrs = np.char.add(prefixes[s % len(prefixes)], chr_of_row[rows])
        out.append((chrs[keep], pos[keep], gt[keep]))
    return out


def _inputs(samples):
    from snpmatch_b200.core import parsers
    res = []
    for chrs, pos, gt in samples:
        x = parsers.ParseInputs("")
        x.load_snp_info(np.asarray(chrs), np.asarray(pos), np.asarray(gt), np.ones((len(pos), 3)), "NA")
        res.append(x)
    return res


# ---- 1. golden ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_db", [False, True])
def test_golden_samples_in_one_call(lib, small_geno, small_panel, tmp_path, with_db):
    from snpmatch_b200.core import snpmatch
    files, samples = _golden_files(tmp_path)
    db = small_geno if with_db else None
    pm = snpmatch.pairwise_score_many(files, hdf5File=db)
    _check_oracle(pm, samples, _db_keys(small_panel) if with_db else None)
    for i in range(len(files)):
        for j in range(i + 1, len(files)):
            _stats_equal(pm.stats(i, j), snpmatch.pairwiseScore(files[i], files[j], False, hdf5File=db))
    with open(os.path.join(GOLDEN, "pairsnp.json")) as fh:
        want = json.load(fh)
    for i in range(3):
        got = pm.stats(2 * i, 2 * i + 1)
        assert got.pop("hdf5", None) == ("resident" if with_db else None)
        _stats_equal(got, want["p%d_%s" % (i, "db" if with_db else "plain")])
    ident = pm.identity()
    c, s = pm.common.sum(0), pm.same.sum(0)
    assert np.array_equal(np.isnan(ident), c == 0)
    assert np.allclose(ident[c > 0], s[c > 0] / c[c > 0], rtol=0, atol=0)


# ---- 2. tile and size limits --------------------------------------------------------------------------------------------
def _size_case(lib, small_panel, tmp_path, S, device=0):
    from snpmatch_b200.core import snpmatch
    per = 300 if S < 1600 else 150
    samples = _simulated(small_panel, S, per, seed=S)
    pm = snpmatch.pairwise_score_many(_inputs(samples), device=device, names=["s%d.npz" % i for i in range(S)])
    return pm, samples


@pytest.mark.parametrize("S", [1, 2, 63, 64, 65, 255, 256, 257, 1600])
def test_tile_and_size_limits(lib, small_panel, tmp_path, S):
    from snpmatch_b200.core import snpmatch
    pm, samples = _size_case(lib, small_panel, tmp_path, S)
    _check_oracle(pm, samples)
    if S == 1600:
        assert 25 * 7 > lib.device_info()["n_sm"]            # more tiles than SMs in one chunk
    files = [_write(tmp_path, "s%d" % i, *samples[i]) for i in range(S)] if S <= 65 else None
    rng = np.random.default_rng(S)
    pairs = [(i, j) for i in range(S) for j in range(i + 1, S)] if S <= 65 else \
        [tuple(sorted(rng.choice(S, size=2, replace=False))) for _ in range(200)]
    for i, j in pairs:
        if files is None:
            fi, fj = _write(tmp_path, "s%d" % i, *samples[i]), _write(tmp_path, "s%d" % j, *samples[j])
        else:
            fi, fj = files[i], files[j]
        _stats_equal(pm.stats(i, j), snpmatch.pairwiseScore(fi, fj, False))


# ---- 3. chunking --------------------------------------------------------------------------------------------------------
def _dense(lib_offsets, col, cls, K, chr_start, n_cls):
    S = len(lib_offsets) - 1
    G = np.full((S, K), -1, np.int64)
    for s in range(S):
        G[s, col[lib_offsets[s]:lib_offsets[s + 1]]] = cls[lib_offsets[s]:lib_offsets[s + 1]]
    C = len(chr_start) - 1
    common = np.zeros((C, S, S), np.int64)
    same = np.zeros((C, S, S), np.int64)
    for c in range(C):
        Gc = G[:, chr_start[c]:chr_start[c + 1]]
        P = (Gc >= 0).astype(np.float64)
        common[c] = np.rint(P @ P.T)
        for v in range(n_cls):
            H = (Gc == v).astype(np.float64)
            same[c] += np.rint(H @ H.T).astype(np.int64)
    return common, same


def _random_csr(rng, S, K, n_cls, density=0.4):
    G = np.where(rng.random((S, K)) < density, rng.integers(0, n_cls, size=(S, K)), -1)
    offsets = np.concatenate([[0], np.cumsum((G >= 0).sum(1))]).astype(np.int64)
    s_idx, col = np.nonzero(G >= 0)
    return offsets, col.astype(np.int32), G[s_idx, col].astype(np.uint8)


@pytest.mark.parametrize("n_cls", [1, 4, 5, 8])
def test_chunking_and_classes(lib, n_cls):
    rng = np.random.default_rng(10 + n_cls)
    S = 70
    # per-chromosome columns: 1, 0 (no sample has it), 45, 33 (not multiples of 32 or 16), 17 (only sample 5 has it), 100
    widths = [1, 0, 45, 33, 17, 100]
    chr_start = np.concatenate([[0], np.cumsum(widths)]).astype(np.int64)
    K = int(chr_start[-1])
    offsets, col, cls = _random_csr(rng, S, K, n_cls)
    keep = np.ones(len(col), bool)
    only = (col >= chr_start[4]) & (col < chr_start[5])
    owner = np.repeat(np.arange(S), np.diff(offsets))
    keep &= ~only | (owner == 5)
    offsets = np.concatenate([[0], np.cumsum(np.bincount(owner[keep], minlength=S))]).astype(np.int64)
    col, cls = col[keep], cls[keep]
    want_c, want_s = _dense(offsets, col, cls, K, chr_start, n_cls)
    mk = 32 if n_cls <= 4 else 16
    for chunk in (0, mk, 37, 1):
        common, same, ms = lib.pair_matrix(offsets, col, cls, n_cls, K, chr_start, chunk_markers=chunk)
        assert np.array_equal(common, want_c), chunk
        assert np.array_equal(same, want_s), chunk
        assert ms[1] > 0 and ms[2] >= ms[1]
    assert want_c[4, 5, 5] > 0 and want_c[4].sum() == want_c[4, 5, 5]


def test_api_chunks_and_database_chromosome(lib, small_geno, small_panel):
    """pairwise_score_many with chunk_markers forced to one k-block and to 37 columns equals the default budget; with the
    database, a chromosome the database lacks (ChrM) is listed with no column."""
    from snpmatch_b200.core import snpmatch
    samples = _simulated(small_panel, 40, 200, seed=4, n_strings=6)
    samples[3] = (np.concatenate([samples[3][0], ["ChrM"] * 3]), np.concatenate([samples[3][1], [5, 6, 7]]),
                  np.concatenate([samples[3][2], ["0/0"] * 3]))
    base = snpmatch.pairwise_score_many(_inputs(samples), hdf5File=small_geno)
    _check_oracle(base, samples, _db_keys(small_panel))
    assert "M" in base.chromosomes.tolist() and base.common[base.chromosomes.tolist().index("M")].sum() == 0
    for chunk in (16, 37):
        pm = snpmatch.pairwise_score_many(_inputs(samples), hdf5File=small_geno, chunk_markers=chunk)
        assert np.array_equal(pm.common, base.common) and np.array_equal(pm.same, base.same)


# ---- 4. classes ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_strings", [1, 4, 5, 8])
def test_class_counts_against_single_path(lib, small_panel, tmp_path, n_strings):
    from snpmatch_b200.core import snpmatch
    samples = _simulated(small_panel, 12, 250, seed=100 + n_strings, n_strings=n_strings)
    pm = snpmatch.pairwise_score_many(_inputs(samples), names=["c%d.npz" % i for i in range(12)])
    assert pm.n_classes == len(np.unique(np.concatenate([s[2] for s in samples])))
    _check_oracle(pm, samples)
    files = [_write(tmp_path, "c%d" % i, *samples[i]) for i in range(12)]
    for i, j in ((0, 1), (2, 9), (3, 4), (10, 11)):
        _stats_equal(pm.stats(i, j), snpmatch.pairwiseScore(files[i], files[j], False))


# ---- 5. refusals and errors ---------------------------------------------------------------------------------------------
def test_library_refusals(lib):
    off, col, cls = np.array([0, 2, 3]), np.array([0, 1, 1], np.int32), np.array([0, 1, 1], np.uint8)
    ok = lib.pair_matrix(off, col, cls, 2, 2, [0, 2])
    assert ok[0].shape == (1, 2, 2)
    cases = [
        (off, np.array([1, 0, 1], np.int32), cls, 2, 2, [0, 2], "sample 0: columns are not strictly ascending"),
        (off, np.array([0, 1, 2], np.int32), cls, 2, 2, [0, 2], "sample 1: column 2"),
        (off, col, np.array([0, 1, 2], np.uint8), 2, 2, [0, 2], "sample 1: class 2"),
        (off, col, cls, 2, 2, [0, 3], "chr_start"),
        (off, col, cls, 2, 2, [0, 2, 1, 2], "chr_start decreases"),
        (off, col, cls, 9, 2, [0, 2], "bad arguments"),
    ]
    for o, c, k, n_cls, K, cs, msg in cases:
        with pytest.raises(lib.SnpmError, match=msg):
            lib.pair_matrix(o, c, k, n_cls, K, cs)
    n = lib.PAIR_MAX_SAMPLES + 1
    with pytest.raises(lib.SnpmError, match="%d samples" % n):
        lib.pair_matrix(np.zeros(n + 1, np.int64), np.zeros(0, np.int32), np.zeros(0, np.uint8), 1, 0, [0])


def test_empty_sample_and_duplicate_marker(lib, small_panel):
    from snpmatch_b200.core import snpmatch
    samples = _simulated(small_panel, 4, 100, seed=8)
    samples[2] = (np.zeros(0, "U1"), np.zeros(0, np.int64), np.zeros(0, "U3"))
    pm = snpmatch.pairwise_score_many(_inputs(samples))
    _check_oracle(pm, samples)
    ident = pm.identity()
    assert np.all(np.isnan(ident[2])) and np.all(pm.common[:, 2, :] == 0)
    st = pm.stats(1, 2)
    assert st["matches"][1] == 0 and np.isnan(st["matches"][0])
    dup = list(samples)
    dup[1] = (np.concatenate([dup[1][0], dup[1][0][:1]]), np.concatenate([dup[1][1], dup[1][1][:1]]), np.concatenate([dup[1][2], ["0/0"]]))
    with pytest.raises(ValueError, match=r"sample 1 \(sample1\).*appears more than once"):
        snpmatch.pairwise_score_many(_inputs(dup))


# ---- 6. command line ----------------------------------------------------------------------------------------------------
def test_command_line_samples(lib, small_geno, small_panel, tmp_path):
    import snpmatch_b200
    from snpmatch_b200.core import snpmatch
    db_path = str(tmp_path / "panel.npz")
    small_geno.save_packed(db_path)
    files, _ = _golden_files(tmp_path)
    lst = tmp_path / "list.txt"
    lst.write_text("".join("%s\n" % f if k % 2 == 0 else "%s\tlab%d\n" % (f, k) for k, f in enumerate(files)))
    out = str(tmp_path / "p")
    assert snpmatch_b200.main(["pairsnp", "--samples", str(lst), "-d", db_path, "-o", out, "--pairs_json"]) == 0
    pm = snpmatch.pairwise_score_many(files, hdf5File=db_path)
    labels = [os.path.basename(f) if k % 2 == 0 else "lab%d" % k for k, f in enumerate(files)]
    for name, want in (("identity", pm.identity()), ("common", pm.common.sum(0))):
        rows = [line.split("\t") for line in open("%s.%s.tsv" % (out, name)).read().splitlines()]
        assert rows[0] == ["sample"] + labels
        assert [r[0] for r in rows[1:]] == labels
        got = np.array([[float(v) for v in r[1:]] for r in rows[1:]])
        assert np.array_equal(got, want, equal_nan=True)
    lines = open(out + ".pairs.jsonl").read().splitlines()
    assert len(lines) == 15
    k = 0
    for i in range(6):
        for j in range(i + 1, 6):
            rec = json.loads(lines[k])
            k += 1
            assert rec["sample_1"] == files[i] and rec["sample_2"] == files[j]
            single = snpmatch.pairwiseScore(files[i], files[j], False, hdf5File=db_path)
            _stats_equal(rec["stats"], single)
    with pytest.raises(SystemExit):
        snpmatch_b200.main(["pairsnp", "--samples", str(lst), "-i", files[0], "-o", out])


# ---- 7. second GPU ------------------------------------------------------------------------------------------------------
def test_second_gpu_equals_first(lib, small_panel, tmp_path):
    if lib.device_count() < 2:
        pytest.skip("one GPU")
    for S in (1, 2, 63, 64, 65, 255, 256, 257, 1600):
        a, _ = _size_case(lib, small_panel, tmp_path, S, device=0)
        b, _ = _size_case(lib, small_panel, tmp_path, S, device=1)
        assert np.array_equal(a.common, b.common) and np.array_equal(a.same, b.same), S
