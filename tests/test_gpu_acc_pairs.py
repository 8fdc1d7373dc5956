"""`pairsnp --accessions` on the GPU: every pair of panel accessions over the resident panel in one tensor-core pass
(lib.Database.acc_pairs, snpmatch.panel_identity).  Every count is compared == against a NumPy oracle on the int8 panel,
and one pair against `pairsnp -i -j` on the two accessions written as BED."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GT_OF_CODE = {0: "0/0", 1: "1/1", 2: "0/1"}


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


def oracle(snps, sel=None, skip_hets=False, rows_of=None):
    """(common, same) int64 from the int8 panel [rows, A]: accessions sel (default all) against every accession of sel,
    or only the rows `rows_of` (indices into sel) against all of sel."""
    X = snps if sel is None else snps[:, sel]
    called = (X >= 0) & (X <= (1 if skip_hets else 2))
    lhs = slice(None) if rows_of is None else rows_of
    P = called.astype(np.float64)
    common = np.rint(P[:, lhs].T @ P).astype(np.int64)
    same = np.zeros_like(common)
    for c in range(3):
        H = (called & (X == c)).astype(np.float64)
        same += np.rint(H[:, lhs].T @ H).astype(np.int64)
    return common, same


def random_panel(rows, n_acc, seed):
    """Random calls of all four codes (-1 missing, 0, 1, 2); accession 5 all missing, 7 a copy of 3, 64 of 0, 200 of 100 and
    257 of 2 (duplicates inside a tile and across tiles)."""
    rng = np.random.default_rng(seed)
    snps = rng.choice(np.array([-1, 0, 1, 2], np.int8), size=(rows, n_acc), p=[0.15, 0.4, 0.3, 0.15])
    snps[:, 5] = -1
    for dst, src in ((7, 3), (64, 0), (200, 100), (257, 2)):
        if dst < n_acc:
            snps[:, dst] = snps[:, src]
    return snps


def make_db(lib, snps, device=0):
    from snpmatch_b200 import synth
    positions, regions = synth.panel_positions(snps.shape[0])
    db = lib.Database(positions, regions, snps.shape[1], device=device)
    db.load_int8(snps)
    return db


def check(lib, db, snps, sel, skip, **kw):
    common, same, ms = db.acc_pairs(sel, skip_db_hets=skip, **kw)
    want_c, want_s = oracle(snps, sel, skip)
    assert common.dtype == np.int32 and common.shape == (len(sel), len(sel))
    assert np.array_equal(common, want_c), (len(sel), skip, kw)
    assert np.array_equal(same, want_s), (len(sel), skip, kw)
    assert ms[1] > 0 and ms[2] >= ms[1]
    return common, same


# ---- 1. random panels around the tile edges -------------------------------------------------------------------------------
@pytest.mark.parametrize("skip", [False, True])
@pytest.mark.parametrize("rows", [1, 31, 32, 33, 3000])
def test_random_panels_against_oracle(lib, rows, skip):
    snps = random_panel(rows, 320, seed=rows)
    db = make_db(lib, snps)
    try:
        for n in (1, 2, 63, 64, 65, 255, 256, 257, 300):
            sel = np.arange(n)
            common, same = check(lib, db, snps, sel, skip)
            if n > 5:
                assert (common[5] == 0).all() and (common[:, 5] == 0).all()
            if n > 7:
                assert common[3, 7] == same[3, 7] == common[3, 3]
            if n > 257:
                assert common[2, 257] == same[2, 257] == common[2, 2]
            assert np.array_equal(common, common.T) and np.array_equal(same, same.T)
        # a permuted selection that puts the all-missing accession and the duplicates in other tiles
        sel = np.random.default_rng(rows).permutation(320)[:300]
        check(lib, db, snps, sel, skip)
    finally:
        db.close()


def test_identity_of_duplicates_and_missing(lib):
    from snpmatch_b200 import synth
    from snpmatch_b200.core import snp_genotype, snpmatch
    snps = random_panel(500, 70, seed=3)
    positions, regions = synth.panel_positions(500)
    g = snp_genotype.Genotype.from_arrays(snps, positions, np.array(synth.TAIR10_CHRS), regions, synth.accession_ids(70))
    try:
        r = snpmatch.panel_identity(g)
        ident = r.identity()
        assert np.isnan(ident[5]).all() and np.isnan(ident[:, 5]).all()
        assert ident[3, 7] == 1.0 and ident[0, 64] == 1.0
        assert ("1000", "1064", 1.0, int(r.common[0, 64]), int(r.common[0, 64])) in r.close_pairs(1.0)
        assert r.accessions.tolist() == [str(1000 + a) for a in range(70)]
    finally:
        g.close()


# ---- 2. chunks and blocks -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [300, 600])
def test_forced_chunks_and_blocks(lib, n):
    snps = random_panel(3000, 640, seed=n)
    db = make_db(lib, snps)
    try:
        sel = np.arange(n)
        for skip in (False, True):
            base = check(lib, db, snps, sel, skip)
            for kw in ({"chunk_rows": 32}, {"chunk_rows": 37}, {"block_acc": 256}, {"block_acc": 256, "chunk_rows": 37}):
                got = db.acc_pairs(sel, skip_db_hets=skip, **kw)
                assert np.array_equal(got[0], base[0]) and np.array_equal(got[1], base[1]), (skip, kw)
    finally:
        db.close()


# ---- 3. subsets and refusals ----------------------------------------------------------------------------------------------
def test_unsorted_subset_is_a_submatrix(lib):
    snps = random_panel(2000, 300, seed=11)
    db = make_db(lib, snps)
    try:
        full_c, full_s, _ = db.acc_pairs()
        assert full_c.shape == (300, 300)
        sub = np.array([257, 3, 299, 0, 64, 5, 7, 128, 3 + 256, 1])
        c, s, _ = db.acc_pairs(sub)
        assert np.array_equal(c, full_c[np.ix_(sub, sub)]) and np.array_equal(s, full_s[np.ix_(sub, sub)])
        c, s, _ = db.acc_pairs(sub, block_acc=256, chunk_rows=37)
        assert np.array_equal(c, full_c[np.ix_(sub, sub)]) and np.array_equal(s, full_s[np.ix_(sub, sub)])
    finally:
        db.close()


def test_refusals(lib):
    snps = random_panel(100, 40, seed=12)
    db = make_db(lib, snps)
    try:
        cases = [
            (dict(acc_idx=np.zeros(0, np.int32)), "n_sel = 0"),
            (dict(acc_idx=[0, 40]), "accession index 40 \\(entry 1\\) is outside 0..39"),
            (dict(acc_idx=[-1]), "accession index -1"),
            (dict(block_acc=100), "block_acc = 100 is not a positive multiple of 256"),
            (dict(block_acc=-256), "block_acc = -256"),
            (dict(chunk_rows=-1), "chunk_rows = -1"),
        ]
        for kw, msg in cases:
            with pytest.raises(lib.SnpmError, match=msg):
                db.acc_pairs(**kw)
        check(lib, db, snps, np.arange(40), False, block_acc=512)
    finally:
        db.close()


# ---- 4. row shards --------------------------------------------------------------------------------------------------------
def test_row_shards_sum_to_the_panel(lib):
    from snpmatch_b200.core import snp_genotype, snpmatch
    N, A = 5000, 300
    whole = snp_genotype.Genotype.synthetic(N, A)
    shards = [snp_genotype.Genotype.synthetic(N, A, row_range=rr) for rr in ((0, 1999), (1999, N))]
    try:
        sel = np.random.default_rng(4).permutation(A)[:280]
        for skip in (False, True):
            c, s, _ = whole.db.acc_pairs(sel, skip_db_hets=skip)
            want_c, want_s = oracle(whole.db.read_columns(np.arange(A)).T, sel, skip)
            assert np.array_equal(c, want_c) and np.array_equal(s, want_s)
            parts = [g.db.acc_pairs(sel, skip_db_hets=skip) for g in shards]
            assert np.array_equal(parts[0][0].astype(np.int64) + parts[1][0], c)
            assert np.array_equal(parts[0][1].astype(np.int64) + parts[1][1], s)
        with pytest.raises(ValueError, match="shard"):
            snpmatch.panel_identity(shards[1])
    finally:
        for g in [whole] + shards:
            g.close()


# ---- 5. the link to pairsnp -i -j -----------------------------------------------------------------------------------------
def test_two_accessions_as_bed_match_pairsnp(lib, small_panel, tmp_path):
    from snpmatch_b200.core import snp_genotype, snpmatch
    p = small_panel
    g = snp_genotype.Genotype.from_arrays(p["snps"], p["positions"], p["chrs"], p["chr_regions"], p["accessions"])
    try:
        A = g.g.num_accessions
        rng = np.random.default_rng(5)
        pairs = [tuple(rng.choice(A, size=2, replace=False)) for _ in range(4)]
        sel = np.unique(np.array(pairs).ravel())
        res = snpmatch.panel_identity(g, [g.accessions[a] for a in sel])
        ident = res.identity()
        cols = g.g.snps[:, sel]                                      # the column read
        chr_of_row = np.repeat(g.chrs, np.diff(g.g.chr_regions, axis=1).ravel())
        files = {}
        for k, a in enumerate(sel):
            keep = cols[:, k] >= 0
            f = str(tmp_path / ("acc%d.bed" % a))
            with open(f, "w") as fh:
                for c, pos, code in zip(chr_of_row[keep], g.g.positions[keep], cols[keep, k]):
                    fh.write("%s\t%d\t%s\n" % (c, pos, GT_OF_CODE[int(code)]))
            files[a] = (k, f)
        for a, b in pairs:
            (i, fa), (j, fb) = files[a], files[b]
            st = snpmatch.pairwiseScore(fa, fb, False)
            assert st["matches"][1] == int(res.common[i, j])
            assert st["matches"][0] == ident[i, j] or (np.isnan(st["matches"][0]) and np.isnan(ident[i, j]))
    finally:
        g.close()


# ---- 6. 20 000 accessions -------------------------------------------------------------------------------------------------
def test_twenty_thousand_accessions(lib):
    from snpmatch_b200.core import snp_genotype
    N, A = 3000, 20000
    g = snp_genotype.Genotype.synthetic(N, A)
    try:
        common, same, ms = g.db.acc_pairs()
        snps = g.db.read_columns(np.arange(A)).T
        rows = np.random.default_rng(6).choice(A, size=64, replace=False)
        want_c, want_s = oracle(snps, None, False, rows_of=rows)
        assert np.array_equal(common[rows], want_c) and np.array_equal(same[rows], want_s)
        called = (snps >= 0).sum(0)
        assert np.array_equal(np.diagonal(common), called) and np.array_equal(np.diagonal(same), called)
        assert np.array_equal(common[:, rows].T, want_c)           # the mirrored blocks
    finally:
        g.close()


# ---- 7. command line ------------------------------------------------------------------------------------------------------
def test_command_line_accessions(lib, tmp_path, capsys):
    import snpmatch_b200
    from snpmatch_b200 import synth
    from snpmatch_b200.core import snp_genotype, snpmatch
    snps = random_panel(1500, 90, seed=7)
    positions, regions = synth.panel_positions(1500)
    g = snp_genotype.Genotype.from_arrays(snps, positions, np.array(synth.TAIR10_CHRS), regions, synth.accession_ids(90))
    db_path = str(tmp_path / "panel.npz")
    try:
        g.save_packed(db_path)
        api = snpmatch.panel_identity(g)
        api.write(str(tmp_path / "api"), min_identity=0.5)
        sub_ids = ["1064", "1003", "1089", "1000", "1007"]
        api_sub = snpmatch.panel_identity(g, sub_ids, skip_db_hets=True)
        api_sub.write(str(tmp_path / "api_sub"))
    finally:
        g.close()
    out = str(tmp_path / "cli")
    assert snpmatch_b200.main(["pairsnp", "-d", db_path, "--accessions", "all", "--min_identity", "0.5", "-o", out]) == 0
    for ext in ("identity.tsv", "common.tsv", "close_pairs.tsv"):
        assert open("%s.%s" % (out, ext)).read() == open(str(tmp_path / ("api." + ext))).read(), ext
    # random calls agree on about 38 % of the rows both have called: only the two duplicated accessions pass 0.5
    assert [line.split("\t")[:3] for line in open(out + ".close_pairs.tsv").read().splitlines()[1:]] == \
        [["1000", "1064", "1.0"], ["1003", "1007", "1.0"]]
    assert open(out + ".common.tsv").readline() == "\t".join(["sample"] + [str(1000 + a) for a in range(90)]) + "\n"
    ids = tmp_path / "ids.txt"
    ids.write_text("\n".join(sub_ids) + "\n")
    out_sub = str(tmp_path / "cli_sub")
    assert snpmatch_b200.main(["pairsnp", "-d", db_path, "--accessions", str(ids), "--skip_db_hets", "-o", out_sub]) == 0
    for ext in ("identity.tsv", "common.tsv"):
        assert open("%s.%s" % (out_sub, ext)).read() == open(str(tmp_path / ("api_sub." + ext))).read(), ext
    import os
    assert not os.path.exists(out_sub + ".close_pairs.tsv")
    capsys.readouterr()
    unknown = tmp_path / "unknown.txt"
    unknown.write_text("1003\n4242\n")
    rep = tmp_path / "rep.txt"
    rep.write_text("1003\n1004\n1003\n")
    a_bed = tmp_path / "a.bed"
    a_bed.write_text("Chr1\t5\t0/0\n")
    cases = [
        (["pairsnp", "--accessions", "all", "-o", out], "-d"),
        (["pairsnp", "-d", db_path, "--accessions", "all", "-i", str(a_bed)], "cannot be combined"),
        (["pairsnp", "-d", db_path, "--accessions", "all", "-j", str(a_bed)], "cannot be combined"),
        (["pairsnp", "-d", db_path, "--accessions", "all", "--samples", str(ids)], "cannot be combined"),
        (["pairsnp", "-d", db_path, "--accessions", str(unknown), "-o", out], "accession 4242 is not in the database"),
        (["pairsnp", "-d", db_path, "--accessions", str(rep), "-o", out], "1003 is listed twice"),
    ]
    for argv, msg in cases:
        with pytest.raises(SystemExit) as e:
            snpmatch_b200.main(argv)
        assert e.value.code == 1, argv
        assert msg in capsys.readouterr().err, argv


# ---- 8. second GPU --------------------------------------------------------------------------------------------------------
def test_second_gpu_equals_first(lib):
    if lib.device_count() < 2:
        pytest.skip("one GPU")
    snps = random_panel(3000, 640, seed=8)
    got = []
    for dev in (0, 1):
        db = make_db(lib, snps, device=dev)
        try:
            got.append([db.acc_pairs(np.arange(600), skip_db_hets=skip, block_acc=bs)[:2] for skip in (False, True) for bs in (0, 256)])
        finally:
            db.close()
    for (c0, s0), (c1, s1) in zip(*got):
        assert np.array_equal(c0, c1) and np.array_equal(s0, s1)
    want = oracle(snps, np.arange(600))
    assert np.array_equal(got[1][0][0], want[0]) and np.array_equal(got[1][0][1], want[1])
