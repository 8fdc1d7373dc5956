"""`inbred --samples_vcf` / `cross --samples_vcf`: every sample column of one VCF parsed on the device (parsers.read_vcf_many,
lib.VcfParser, csrc/vcf.cuh).  Sample s's ParseInputs equals ParseInputs of the single-sample VCF of column s (same header,
the 9 fixed columns and column s) array for array and bit for bit, whatever the chunking; the records the device hands to the
Python code are the known ones; and the files written for every sample are byte for byte the ones `-i` writes for its
single-sample VCF."""
import gzip
import os
import re

import numpy as np
import pytest

from snpmatch_b200 import synth


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


def _write(path, text):
    with open(path, "w", encoding="utf-8", newline="") as fh:
        fh.write(text)


def _same_inputs(a, b, what):
    for k in ("chrs", "pos", "gt", "dp"):
        x, y = getattr(a, k), getattr(b, k)
        assert x.dtype == y.dtype and x.shape == y.shape and np.array_equal(x, y), (what, k)
    assert a.wei.shape == b.wei.shape and np.array_equal(a.wei.view(np.int64), b.wei.view(np.int64)), (what, "wei")
    ca, cb = a.coded_weights(), b.coded_weights()
    assert (ca is None) == (cb is None), what
    if ca is not None:
        assert np.array_equal(ca[0], cb[0]) and np.array_equal(ca[1].view(np.int64), cb[1].view(np.int64)), (what, "codes")


def _singles(tmp_path, text, n_samples):
    from snpmatch_b200.core import parsers
    out = []
    for s in range(n_samples):
        p = str(tmp_path / ("col%d.vcf" % s))
        _write(p, synth.split_vcf_column(text, s))
        out.append(parsers.ParseInputs(p))
    return out


def _chunk_sizes(text):
    """A chunk a little longer than the longest line (lines straddle chunks), one whose first chunk ends exactly at a line end,
    and for CRLF files one whose first chunk ends between the '\\r' and the '\\n'."""
    body = text.split("#CHROM", 1)[1].encode("utf-8")
    body = body[re.search(rb"\r\n|\r|\n", body).end():]
    lines = body.replace(b"\r\n", b"\n").replace(b"\r", b"\n").split(b"\n")
    longest = max(len(x) for x in lines) + 2
    ends = [i + 1 for i, c in enumerate(body) if c == 10 or (c == 13 and (i + 1 == len(body) or body[i + 1] != 10))]
    aligned = next(e for e in ends if e >= longest)
    sizes = [longest + 37, aligned]
    if b"\r\n" in body[:aligned]:
        sizes.append(aligned - 1 if body[aligned - 2:aligned] == b"\r\n" else aligned + 1)
    return sizes


CASES = {"lf": {}, "crlf": {"line_end": "\r\n"}, "cr": {"line_end": "\r"}, "mixed": {"line_end": ["\n", "\r\n", "\r"]},
         "no_dp_header": {"info_dp_header": False}, "late_dp": {"info_dp_header": False, "late_info_dp": True}}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_parser_parity_with_single_sample_files(lib, tmp_path, case):
    from snpmatch_b200.core import parsers
    S = 37
    text, fallback = synth.multi_sample_vcf(301, S, seed=11 + len(case), **CASES[case])
    path = str(tmp_path / "multi.vcf")
    _write(path, text)
    singles = _singles(tmp_path, text, S)
    assert fallback, "the file exercises the Python fallback"
    for chunk in [parsers.VCF_CHUNK_BYTES] + _chunk_sizes(text):
        tm = {}
        many = parsers.read_vcf_many(path, chunk_bytes=chunk, timings=tm)
        assert [n for n, _ in many] == ["smp%d" % s for s in range(S)]
        assert tm["fallback"] == fallback, chunk
        for s, ((_, inp), one) in enumerate(zip(many, singles)):
            _same_inputs(inp, one, (case, chunk, s))
    assert not any(f.startswith("multi.vcf.") for f in os.listdir(tmp_path)), "no parser dump next to the VCF"


@pytest.mark.gpu
def test_gzip_equals_plain(lib, tmp_path):
    from snpmatch_b200.core import parsers
    text, _ = synth.multi_sample_vcf(501, 33, seed=5, line_end=["\n", "\r\n"])
    plain, gz = str(tmp_path / "m.vcf"), str(tmp_path / "m.vcf.gz")
    _write(plain, text)
    with open(gz, "wb") as fh:
        fh.write(gzip.compress(text.encode("utf-8")))
    a, b = parsers.read_vcf_many(plain), parsers.read_vcf_many(gz, chunk_bytes=_chunk_sizes(text)[0])
    for s, ((na, x), (nb, y)) in enumerate(zip(a, b)):
        assert na == nb
        _same_inputs(x, y, s)
    for s, one in enumerate(_singles(tmp_path, text, 33)):
        _same_inputs(b[s][1], one, s)


@pytest.mark.gpu
def test_line_longer_than_the_chunk_is_refused(lib, tmp_path):
    from snpmatch_b200.core import parsers
    text, _ = synth.multi_sample_vcf(40, 8, seed=2, edge_cases=False)
    lines = text.split("\n")
    lines[10] = lines[10] + "\t" + "\t".join(["0/1:1,0,9"] * 200)      # header lines 1-3, so this is line 11
    path = str(tmp_path / "long.vcf")
    _write(path, "\n".join(lines))
    with pytest.raises(ValueError, match=r"line 11 is longer than the chunk of 2000 bytes"):
        parsers.read_vcf_many(path, chunk_bytes=2000)
    assert len(parsers.read_vcf_many(path, chunk_bytes=4000)) == 8
    with pytest.raises(lib.SnpmError, match="chunk_bytes"):
        lib.VcfParser(0, 8, 0)
    no_samples = str(tmp_path / "none.vcf")
    _write(no_samples, "##x\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\nChr1\t1\t.\tA\tT\t.\tPASS\t.\tGT\n")
    with pytest.raises(ValueError, match="no sample columns"):
        parsers.read_vcf_many(no_samples)


@pytest.mark.gpu
def test_second_gpu(lib, tmp_path):
    from snpmatch_b200.core import parsers
    if lib.device_count() < 2:
        pytest.skip("one GPU")
    text, _ = synth.multi_sample_vcf(301, 37, seed=9)
    path = str(tmp_path / "m.vcf")
    _write(path, text)
    for (_, a), (_, b) in zip(parsers.read_vcf_many(path, device=0), parsers.read_vcf_many(path, device=1)):
        _same_inputs(a, b, "device 1")


# ---- end to end: the files of every sample against `-i` on its single-sample VCF ---------------------------------------------
def _cluster_panel(n_rows=8000, n_acc=40, frac=0.004, seed=77):
    """The clustered synthetic panel of the many-sample inbred tests: 1 copies 0, 11-12 copy 10 and 21-24 copy 20, each with
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
def e2e(lib, tmp_path_factory):
    """panel.npz and a VCF of samples drawn from the panel's clusters (called GT with PLs, some phased, some without PL),
    plus one sample without any called genotype."""
    from snpmatch_b200.core import snp_genotype
    p = _cluster_panel()
    d = tmp_path_factory.mktemp("vcf_e2e")
    g = snp_genotype.Genotype.from_arrays(p["snps"], p["positions"], p["chrs"], p["chr_regions"], p["accessions"])
    db = str(d / "panel.npz")
    g.save_packed(db)
    g.close()
    spec = [("pair", 0, 3000), ("trio", 10, 3000), ("five", 20, 7900), ("unique", 30, 3000), ("tiny", 1, 8)]
    samples = [synth.make_sample(p["positions"], p["chr_regions"], p["chrs"], 40, true_acc=a, n_db=n, n_extra=50, seed=i + 1)
               for i, (_, a, n) in enumerate(spec)]
    order = {str(c): i for i, c in enumerate(p["chrs"])}
    keys = sorted({(order[str(c)[3:]] if str(c)[3:] in order else order.get(str(c), 99), str(c), int(x))
                   for s in samples for c, x in zip(s["chrs"], s["pos"])})
    rng = np.random.default_rng(3)
    cells = {}
    for i, s in enumerate(samples):
        for c, x, gt in zip(s["chrs"], s["pos"], s["gt"]):
            gt = str(gt)
            pl = [int(v) for v in rng.integers(10, 90, 3)]
            called = {"0/0": 0, "0/1": 1, "1/0": 1, "1/1": 2}.get(gt.replace("|", "/"))
            if called is not None:
                pl[called] = 0
            if rng.random() < 0.1:
                gt = gt.replace("/", "|")
            cells[(i, str(c), int(x))] = "%s:%s" % (gt, "." if rng.random() < 0.05 else ",".join(map(str, pl)))
    names = [n for n, _, _ in spec] + ["empty"]
    rows = ["##fileformat=VCFv4.2", '##INFO=<ID=DP,Number=1,Type=Integer,Description="depth">',
            "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(names)]
    for _, c, x in keys:
        row = [cells.get((i, c, x), "./.:.") for i in range(len(spec))] + ["./.:0,0,0"]
        rows.append("\t".join([c, str(x), ".", "A", "T", ".", "PASS", "DP=%d" % (x % 50), "GT:PL"] + row))
    text = "\n".join(rows) + "\n"
    vcf = str(d / "population.vcf")
    _write(vcf, text)
    singles = {}
    for s, n in enumerate(names):
        singles[n] = str(d / ("%s.split.vcf" % n))
        _write(singles[n], synth.split_vcf_column(text, s))
    return dict(db=db, vcf=vcf, names=names, singles=singles, dir=d)


def _same_files(a, b, exts):
    for ext in exts:
        assert os.path.exists(a + ext) == os.path.exists(b + ext), b + ext
        if os.path.exists(b + ext):
            assert open(a + ext, "rb").read() == open(b + ext, "rb").read(), b + ext


INBRED_FILES = (".scores.txt", ".matches.json", ".refined.scores.txt")


@pytest.mark.gpu
@pytest.mark.parametrize("refine", [False, True])
@pytest.mark.parametrize("skip", [False, True])
def test_inbred_samples_vcf_files_equal_single_runs(lib, e2e, tmp_path, refine, skip):
    import snpmatch_b200
    flags = (["--refine"] if refine else []) + (["--skip_db_hets"] if skip else [])
    out = str(tmp_path / "many")
    argv = ["inbred", "--samples_vcf", e2e["vcf"], "-d", e2e["db"], "-o", out] + flags
    if refine:                                      # "empty" has no top hit: every other sample is written, then status 1
        with pytest.raises(SystemExit) as e:
            snpmatch_b200.main(argv)
        assert e.value.code == 1
    else:
        assert snpmatch_b200.main(argv) == 0
    for name in e2e["names"]:
        one = str(tmp_path / ("one_" + name))
        rc = snpmatch_b200.main(["inbred", "-i", e2e["singles"][name], "-d", e2e["db"], "-o", one] + flags)
        if refine and name == "empty":
            assert rc == 2                          # the single path stops at its assertion
            assert os.path.exists(out + ".empty.scores.txt") and os.path.exists(out + ".empty.matches.json")
            continue
        assert rc == 0
        _same_files(out + "." + name, one, INBRED_FILES)
    if refine:
        assert os.path.exists(out + ".five.refined.scores.txt")


@pytest.mark.gpu
@pytest.mark.parametrize("skip", [False, True])
def test_cross_samples_vcf_files_equal_single_runs(lib, e2e, tmp_path, capsys, skip):
    import snpmatch_b200
    flags = ["-b", "300000"] + (["--skip_db_hets"] if skip else [])
    out = str(tmp_path / "many")
    # "empty" has no chromosome of the genome: every other sample is written, then status 1 naming it
    with pytest.raises(SystemExit) as e:
        snpmatch_b200.main(["cross", "--samples_vcf", e2e["vcf"], "-d", e2e["db"], "-o", out] + flags)
    assert e.value.code == 1
    err = capsys.readouterr().err
    assert "1 sample column(s)" in err and "empty (Please change default --genome option)" in err
    exts = (".scores.txt", ".windowscore.txt", ".scores.txt.matches.json", ".matches.json")
    for name in e2e["names"]:
        one = str(tmp_path / ("one_" + name))
        rc = snpmatch_b200.main(["cross", "-i", e2e["singles"][name], "-d", e2e["db"], "-o", one] + flags)
        if name == "empty":
            assert rc == 2                          # the single path stops at its assertion
            assert not any(os.path.exists(out + ".empty" + ext) for ext in exts)
            continue
        assert rc == 0
        _same_files(out + "." + name, one, exts)


@pytest.mark.gpu
@pytest.mark.parametrize("cmd", ["inbred", "cross"])
def test_sharded_panel_is_refused(lib, e2e, tmp_path, monkeypatch, capsys, cmd):
    import snpmatch_b200
    from snpmatch_b200.core import snp_genotype
    G = snp_genotype.Genotype
    monkeypatch.setattr(snp_genotype, "Genotype", lambda *a, **k: G.synthetic(4000, 40, row_range=(1000, 4000)))
    with pytest.raises(SystemExit) as e:
        snpmatch_b200.main([cmd, "--samples_vcf", e2e["vcf"], "-d", e2e["db"], "-o", str(tmp_path / "x")])
    assert e.value.code == 1 and "shard" in capsys.readouterr().err
    assert not os.listdir(tmp_path)
