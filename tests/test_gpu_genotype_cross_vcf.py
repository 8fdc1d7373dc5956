"""`genotype_cross --gpu_parse` (parsers.read_vcf_gt_codes, lib.VcfParser.parse_gt_codes, csrc/vcf.cuh k_vcf_gt_codes): the
population VCF's samples, CHROM, POS and window-call codes equal read_vcf_samples + parseGT exactly, whatever the GT text, the
FORMAT, the number of sample fields, the line ends, the chunking, plain or gzip; genotype_cross on them writes the golden lines;
the inputs the text route gives no usable result for are refused with exit status 1, the line named and no file written."""
import gzip
import json
import os
import re

import numpy as np
import pytest

from conftest import GOLDEN, load_golden
from snpmatch_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


HEAD = "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"
TOKENS = ["", ".", "0", "1", "2", "00", "01", "10", "A"]
GT_FORMS = ([a + sep + b for sep in "/|" for a in TOKENS for b in TOKENS] + TOKENS
            + ["1/1/0", "0|1|1", "./././", "1/1|", "./.|1", "1/", "/1", "|1", "0|", "/", "|", "//", "/1/1", "1//1", "1/1/"])
# FORMAT -> cell of a GT text (k varies the cell): GT first, last, absent, repeated (the first wins); cells short of GT
FORMATS = {
    "GT": lambda g, k: g,
    "GT:DP": lambda g, k: g + ":7" if k % 3 else g,
    "DP:GT": lambda g, k: "4:" + g if k % 4 else "4",
    "DP:GQ": lambda g, k: "4:30",
    "GT:GT": lambda g, k: g + ":1/1" if k % 2 else g + ":./.",
    "DP:GT:PL": lambda g, k: "3:" + g + ":0,3,30" if k % 5 else "3",
}
# CHROM runs 1,1,2,1, a non-ASCII CHROM, and the POS texts the host converts
SITES = ([("1", str(p)) for p in range(10, 400, 10)] + [("2", str(p)) for p in range(5, 200, 5)] + [("1", str(p)) for p in range(500, 800, 10)]
         + [("Chré", p) for p in ("+5", "007", "1_0", "3000000000", "0000000009", "13")] + [("3", str(p)) for p in range(1, 300, 3)])


def edge_vcf(n_samples, line_end="\n", final_newline=True, seed=0):
    """Every GT form under every FORMAT at every site, records of n_samples - 3, n_samples + 2, 32 and 33 sample fields, empty
    cells, blank, short and '##' lines among the records."""
    lines = ["##fileformat=VCFv4.2", HEAD + "".join("\tsmp %d" % i for i in range(n_samples)), "##contig=<ID=9,length=99>"]
    fmts = list(FORMATS)
    for i, (c, p) in enumerate(SITES):
        f = fmts[(i + seed) % len(fmts)]
        nsf = n_samples if i % 4 else [max(1, n_samples - 3), n_samples + 2, 32, 33][(i // 4) % 4]
        cells = [FORMATS[f](GT_FORMS[(7 * i + 3 * j + seed) % len(GT_FORMS)], i + j) for j in range(nsf)]
        if i % 9 == 4:
            cells[(i // 9) % nsf] = ""
        lines.append("\t".join([c, p, ".", "A", "T", ".", "PASS", ".", f] + cells))
        if i % 50 == 20:
            lines += ["##a comment after records", "", "1\t5\t.\tA\tT\t.\tPASS\t.\tGT"]
    ends = line_end if isinstance(line_end, list) else [line_end]
    text = "".join(l + ends[k % len(ends)] for k, l in enumerate(lines))
    return text if final_newline else text.rstrip("\r\n")


def _write(path, text, gz=False):
    data = text.encode("utf-8") if isinstance(text, str) else text
    with open(path, "wb") as fh:
        fh.write(gzip.compress(data) if gz else data)


def _text_route(path):
    from snpmatch_b200.core import parsers
    r = parsers.read_vcf_samples(path)
    gt = r["gt"]
    r["gt_codes"] = parsers.parseGT(gt.ravel()).reshape(gt.shape) if gt.size else np.zeros(gt.shape, dtype=np.int8)
    return r


def _same(path, chunks=(None,)):
    from snpmatch_b200.core import parsers
    want = _text_route(path)
    for chunk in chunks:
        tm = {}
        got = parsers.read_vcf_gt_codes(path, timings=tm, **({} if chunk is None else {"chunk_bytes": chunk}))
        for k in ("samples", "chr", "pos", "gt_codes"):
            assert got[k].shape == want[k].shape and np.array_equal(got[k], want[k]), (chunk, k)
        assert got["pos"].dtype == np.int64 and got["gt_codes"].dtype == np.int8 and got["chr"].dtype.kind == "U"
        assert set(tm) >= {"read_s", "device_s", "h2d_ms", "kernel_ms", "host_chunk_s", "assemble_s", "h2d_bytes"}
    return want


def _longest_line(text):
    return max(len(l.encode("utf-8")) for l in re.split(r"\r\n|\r|\n", text)) + 2


@pytest.mark.parametrize("line_end", ["\n", "\r\n", "\r", ["\n", "\r\n", "\r"]], ids=["lf", "crlf", "cr", "mixed"])
def test_edge_file_parity(lib, tmp_path, line_end):
    text = edge_vcf(37, line_end=line_end)
    path = str(tmp_path / "e.vcf")
    _write(path, text)
    n = _longest_line(text)
    want = _same(path, chunks=(None, n, n + 37, 3 * n + 1))
    codes = want["gt_codes"]
    assert set(np.unique(codes).tolist()) == {-1, 0, 1, 2}
    assert want["pos"].max() == 3000000000 and "Chré" in want["chr"].tolist()


@pytest.mark.parametrize("S", [1, 31, 32, 33, 64, 65, 1000])
def test_sample_counts(lib, tmp_path, S):
    path = str(tmp_path / "s.vcf")
    _write(path, edge_vcf(S, seed=S))
    _same(path)


def test_every_gt_form_each_format(lib, tmp_path):
    """Each GT form alone in a cell under each FORMAT: one record per form, one sample per FORMAT."""
    lines = ["##fileformat=VCFv4.2", HEAD + "\ta"]
    for i, g in enumerate(GT_FORMS):
        for f in FORMATS:
            lines.append("\t".join(["1", str(i + 1), ".", "A", "T", ".", "PASS", ".", f, FORMATS[f](g, i + 1)]))
    path = str(tmp_path / "g.vcf")
    _write(path, "\n".join(lines) + "\n")
    want = _same(path)
    assert len(want["pos"]) == len(GT_FORMS) * len(FORMATS)


def test_no_final_newline_and_gzip(lib, tmp_path):
    text = edge_vcf(40, line_end=["\r\n", "\n"], final_newline=False)
    for gz in (False, True):
        path = str(tmp_path / ("n.vcf.gz" if gz else "n.vcf"))
        _write(path, text, gz)
        _same(path, chunks=(None, _longest_line(text)))


def test_chrom_run_across_chunks_and_one_line_per_chunk(lib, tmp_path):
    body = "".join("%s\t%d\t.\tA\tT\t.\tPASS\t.\tGT\t0/1\t1/1\n" % (c, p) for c, p in
                   [("1", 1), ("1", 2), ("2", 3), ("1", 4)] + [("Chr5", p) for p in range(10, 400)])
    text = HEAD + "\ta\tb\n" + body
    path = str(tmp_path / "c.vcf")
    _write(path, text)
    n = _longest_line(text)
    _same(path, chunks=(n, n + 1, 5 * n + 3, None))


def test_exact_fit_line_and_one_byte_more(lib, tmp_path):
    from snpmatch_b200.core import parsers
    long = "1\t7\t.\tA\tT\t.\tPASS\t.\tGT:XX\t1/1:" + "x" * 300 + "\t0/1\n"
    text = HEAD + "\ta\tb\n" + "1\t5\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n" + long + "1\t9\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/0\n"
    path = str(tmp_path / "x.vcf")
    _write(path, text)
    _same(path, chunks=(len(long),))
    with pytest.raises(ValueError, match=r"line 3 is longer than the chunk of %d bytes" % (len(long) - 1)):
        parsers.read_vcf_gt_codes(path, chunk_bytes=len(long) - 1)


def test_header_only(lib, tmp_path):
    from snpmatch_b200.core import parsers
    path = str(tmp_path / "h.vcf")
    _write(path, "##x\n" + HEAD + "\ta\tb\tc\n")
    want = _same(path)
    got = parsers.read_vcf_gt_codes(path)
    assert got["gt_codes"].shape == (0, 3) and want["gt_codes"].shape == (0, 3)


def test_seeded_edge_case_vcf_many_chunks(lib, tmp_path):
    text, _ = synth.multi_sample_vcf(1500, 300, seed=5, hash_lines=False)
    path = str(tmp_path / "m.vcf")
    _write(path, text)
    n = len(text.encode("utf-8"))
    _same(path, chunks=(n // 7, None))


# ---- end to end ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def small_geno(lib, small_panel):
    from snpmatch_b200.core import snp_genotype
    p = small_panel
    g = snp_genotype.Genotype.from_arrays(p["snps"], p["positions"], p["chrs"], p["chr_regions"], p["accessions"])
    yield g
    g.close()


@pytest.fixture(scope="module")
def golden():
    with open(os.path.join(GOLDEN, "genotype_cross.json")) as fh:
        return json.load(fh)


def _population(path, gz=False):
    vcf = load_golden("genotype_cross_vcf.npz")
    text = ("##fileformat=VCFv4.2\n##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">\n"
            + "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(vcf["samples"]) + "\n"
            + "".join("%s\t%d\t.\tA\tT\t50\tPASS\t.\tGT\t%s\n" % (c, p, "\t".join(row)) for c, p, row in zip(vcf["chr"], vcf["pos"], vcf["gt"])))
    _write(path, text, gz)


@pytest.mark.parametrize("tag", ["b300k_lr1.5", "b1M_lr3", "b2M_lr1.5"])
def test_genotype_cross_golden(lib, small_geno, golden, tmp_path, tag):
    from snpmatch_b200.core import genotype_cross as gc
    c = golden[tag]
    path = str(tmp_path / "population.vcf")
    _population(path)
    x = gc.GenotypeCross(small_geno, c["parents"], c["bin_len"], None, False, genome_id="athaliana_tair10")
    assert [str(l) for l in x.genotype_cross(path, c["lr_thres"], gpu_parse=True)] == c["lines"]


def test_cli_golden_plain_and_gzip_and_parent_files(lib, small_geno, golden, tmp_path):
    import snpmatch_b200
    from snpmatch_b200.core import genotype_cross as gc
    c = golden["b1M_lr3"]
    db_path = str(tmp_path / "panel.npz")
    small_geno.save_packed(db_path)
    for gz in (False, True):
        path = str(tmp_path / ("population.vcf" + (".gz" if gz else "")))
        _population(path, gz)
        out = str(tmp_path / ("cli%d.csv" % gz))
        assert snpmatch_b200.main(["genotype_cross", "-i", path, "-d", db_path, "-p", c["parents"], "-b", str(c["bin_len"]),
                                   "--lr_thres", str(c["lr_thres"]), "-o", out, "--gpu_parse"]) == 0
        assert open(out).read().split("\n")[:-1] == c["lines"]
    # parents as BED files over all panel positions
    ids = small_geno.accessions
    i1, i2 = [int(np.flatnonzero(ids == x)[0]) for x in c["parents"].split("x")]
    cols = small_geno.g_acc.snps[:, [i1, i2]]
    chrom = np.array(small_geno.g.chromosomes)
    names = np.array(["./.", "0/0", "1/1", "0/1"])
    for tag, col in (("mother", cols[:, 0]), ("father", cols[:, 1])):
        with open(str(tmp_path / (tag + ".bed")), "w") as fh:
            for ch, p, g in zip(chrom, small_geno.g.positions, names[col.astype(int) + 1]):
                fh.write("%s\t%d\t%s\n" % (ch, p, g))
    x = gc.GenotypeCross(small_geno, str(tmp_path / "mother.bed"), c["bin_len"], str(tmp_path / "father.bed"), False, genome_id="athaliana_tair10")
    assert [str(l) for l in x.genotype_cross(str(tmp_path / "population.vcf"), c["lr_thres"], gpu_parse=True)] == c["lines"]


def test_random_population_multi_chunk_equals_text_route(lib, small_geno, tmp_path, monkeypatch):
    import snpmatch_b200
    from snpmatch_b200.core import parsers
    g = small_geno
    rng = np.random.default_rng(3)
    rows = np.sort(rng.choice(len(g.g.positions), 2500, replace=False))
    path = str(tmp_path / "pop.vcf")
    with open(path, "wb") as fh:
        synth.population_vcf(fh, np.array(g.g.chromosomes)[rows], np.asarray(g.g.positions)[rows], 300, seed=4)
    db_path = str(tmp_path / "panel.npz")
    g.save_packed(db_path)
    acc = g.accessions
    parents = "%sx%s" % (acc[0].decode() if isinstance(acc[0], bytes) else acc[0], acc[3].decode() if isinstance(acc[3], bytes) else acc[3])
    outs = []
    size = os.path.getsize(path)
    real = parsers.read_vcf_gt_codes
    monkeypatch.setattr(parsers, "read_vcf_gt_codes", lambda p, **k: real(p, chunk_bytes=size // 5, **k))
    for flag in ([], ["--gpu_parse"]):
        out = str(tmp_path / ("out%d.csv" % len(flag)))
        assert snpmatch_b200.main(["genotype_cross", "-i", path, "-d", db_path, "-p", parents, "-b", "300000", "-o", out] + flag) == 0
        outs.append(open(out).read())
    assert outs[0] == outs[1] and outs[0].count("\n") > 100


@pytest.mark.parametrize("case", ["hash_line", "long_line", "bad_pos", "huge_pos"])
def test_refusals_exit_1_and_write_nothing(lib, small_geno, golden, tmp_path, capsys, monkeypatch, case):
    import snpmatch_b200
    from snpmatch_b200.core import parsers
    body = "".join("1\t%d\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n" % p for p in range(1, 40))
    bad = {"hash_line": ("#x\n", "line 41 is a '#' line after the #CHROM line"),
           "long_line": ("1\t50\t.\tA\tT\t.\tPASS\t.\tGT:XX\t0/0:" + "x" * 5000 + "\t1/1\n", "line 41 is longer than the chunk of 4096 bytes"),
           "bad_pos": ("1\t1e3\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n", "line 41 has the POS '1e3'"),
           "huge_pos": ("1\t99999999999999999999\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n", "line 41 has the POS '99999999999999999999'")}[case]
    path = str(tmp_path / "r.vcf")
    _write(path, HEAD + "\ta\tb\n" + body + bad[0] + body)
    db = tmp_path / "db"
    db.mkdir()
    small_geno.save_packed(str(db / "panel.npz"))
    real = parsers.read_vcf_gt_codes
    monkeypatch.setattr(parsers, "read_vcf_gt_codes", lambda p, **k: real(p, chunk_bytes=4096, **k))
    before = sorted(os.listdir(tmp_path))
    with pytest.raises(SystemExit) as e:
        snpmatch_b200.main(["genotype_cross", "-i", path, "-d", str(db / "panel.npz"), "-p", golden["b1M_lr3"]["parents"],
                            "-o", str(tmp_path / "out.csv"), "--gpu_parse"])
    assert e.value.code == 1
    assert sorted(os.listdir(tmp_path)) == before, "nothing may be written"
    assert re.search(re.escape(bad[1]), capsys.readouterr().err)
