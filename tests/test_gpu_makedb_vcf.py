"""`makedb --no_csv` (makedb.makeDB_from_vcf, lib.VcfParser.parse_gt_packed, csrc/vcf.cuh k_vcf_gt_packed): the database built
straight from the VCF equals the one vcf_to_csv + makeDB build through the CSV: every array of the .npz with its dtype and shape,
the .json and the count of the warning about calls other than 0/0, 1/1, 0/1, ./.; whatever the chunking, plain or gzip.  The
inputs the CSV route fails on are refused with exit status 1, the line named and no file written."""
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


HEAD = "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"
META = ["##fileformat=VCFv4.2", '##INFO=<ID=DP,Number=1,Type=Integer,Description="depth">', "##contig=<ID=1,length=3000>",
        "##contig=<ID=2,length=2000>"]
GT_CODES = ["0/0", "0|0", "1/1", "1|1", "0/1", "0|1", "1/0", "1|0", "./.", ".|.", "."]
GT_OTHER = ["0", "./0", "1/2", "0/0/0", "00/1", "0/0 ", "", "2/2", "1/."]
GT_ALL = GT_CODES + GT_OTHER
# FORMAT -> cell of a GT text (k varies the cell): GT first, last, absent, repeated; cells short of the GT subfield
FORMATS = {
    "GT": lambda g, k: g,
    "GT:DP": lambda g, k: g + ":7" if k % 3 else g,
    "DP:GT": lambda g, k: "4:" + g if k % 4 else "4",
    "DP:GQ": lambda g, k: "4:30",
    "GT:GT": lambda g, k: g + ":1/1" if k % 2 else ":" + g,
    "DP:GT:PL": lambda g, k: "3:" + g + ":0,3,30" if k % 5 else "3",
}
# (CHROM, POS) of the records, in file order: runs 1,1,2,1; NA / nan neighbours; a non-ASCII CHROM; POS the device hands the
# host (+5, 007, 1_0, ' 12', and 3000000000, which wraps, alone on its chromosome)
SITES = ([("1", str(p)) for p in range(10, 130, 10)] + [("2", str(p)) for p in range(5, 50, 5)] + [("1", str(p)) for p in range(200, 260, 10)]
         + [("NA", "3"), ("nan", "4"), ("NA", "9")] + [("Chré", p) for p in ("+5", "007", "1_0", " 12", "13")] + [("big", "3000000000")]
         + [("3", str(p)) for p in range(1, 40, 3)])


def edge_vcf(n_samples, line_end="\n", final_newline=True, names=None, info="DP=.", seed=0):
    """Every _GT_CODE and counted-other string under every FORMAT of FORMATS, at every site of SITES, with ##contig lines after
    the #CHROM line and a comment line among the records."""
    names = names if names is not None else ["s %d " % i if i % 5 else "dup" for i in range(n_samples)]
    lines = META + [HEAD + "".join("\t" + n for n in names), "##contig=<ID=9,length=99>"]
    fmts = list(FORMATS)
    for i, (c, p) in enumerate(SITES):
        f = fmts[(i + seed) % len(fmts)]
        cells = [FORMATS[f](GT_ALL[(7 * i + 3 * j + seed) % len(GT_ALL)], i + j) for j in range(n_samples)]
        lines.append("\t".join([c, p, ".", "A", "T", ".", "PASS", info, f] + cells))
        if i == 20:
            lines.append("##a comment after records")
    ends = line_end if isinstance(line_end, list) else [line_end]
    text = "".join(l + ends[k % len(ends)] for k, l in enumerate(lines))
    return text if final_newline else text.rstrip("\r\n")


def _write(path, text, gz=False):
    data = text.encode("utf-8")
    with open(path, "wb") as fh:
        fh.write(gzip.compress(data) if gz else data)


def _warned(caplog):
    n = [int(m.group(1)) for m in (re.match(r"(\d+) genotype calls are neither", r.getMessage()) for r in caplog.records) if m]
    caplog.clear()
    return n


def _csv_route(path, out, caplog):
    from snpmatch_b200.core import makedb
    makedb.vcf_to_csv(path, out)
    makedb.makeDB(out + ".csv", out).close()
    return _warned(caplog)


def _same_db(a, b, what=""):
    with np.load(a + ".npz") as x, np.load(b + ".npz") as y:
        assert sorted(x.files) == sorted(y.files)
        for k in ("packed", "positions", "chrs", "chr_regions", "accessions"):
            assert x[k].dtype == y[k].dtype and x[k].shape == y[k].shape and np.array_equal(x[k], y[k]), (what, k)
    with open(a + ".json", "rb") as x, open(b + ".json", "rb") as y:
        assert x.read() == y.read(), (what, "json")


def _parity(tmp_path, caplog, text, gz=False, chunks=(None,), name="m"):
    from snpmatch_b200.core import makedb
    path = str(tmp_path / (name + (".vcf.gz" if gz else ".vcf")))
    _write(path, text, gz)
    ref = str(tmp_path / (name + "_csv"))
    caplog.set_level("WARNING")
    want = _csv_route(path, ref, caplog)
    tms = []
    for chunk in chunks:
        out = str(tmp_path / (name + "_dev"))
        tm = {}
        kw = {} if chunk is None else {"chunk_bytes": chunk}
        makedb.makeDB_from_vcf(path, out, timings=tm, **kw).close()
        assert _warned(caplog) == want, chunk
        _same_db(out, ref, chunk)
        assert not os.path.exists(out + ".csv")
        tms.append(tm)
    return ref, want, tms


def _longest_line(text):
    return max(len(l.encode("utf-8")) for l in re.split(r"\r\n|\r|\n", text)) + 2


@pytest.mark.gpu
@pytest.mark.parametrize("line_end", ["\n", "\r\n", "\r", ["\n", "\r\n", "\r"]], ids=["lf", "crlf", "cr", "mixed"])
def test_edge_file_parity(lib, tmp_path, caplog, line_end):
    text = edge_vcf(37, line_end=line_end)
    n = _longest_line(text)
    _, want, tms = _parity(tmp_path, caplog, text, chunks=(None, n, n + 37, 3 * n + 1))
    assert want and want[0] > 0, "the file holds counted calls"
    # the device hands the host exactly the POS texts that are not 1-9 plain digits (+5, 1_0, ' 12', 3000000000; 007 is read
    # on the device); DP=. in INFO flags nothing
    first = next(i for i, s in enumerate(SITES) if s[0] == "Chré")
    for tm in tms:
        assert tm["flagged"] == [first, first + 2, first + 3, first + 5]
        assert tm["h2d_bytes"] > 0 and tm["kernel_ms"] > 0


@pytest.mark.gpu
def test_no_final_newline_and_gzip(lib, tmp_path, caplog):
    text = edge_vcf(33, line_end="\r\n", final_newline=False, seed=3)
    _parity(tmp_path, caplog, text, name="a")
    _parity(tmp_path, caplog, text, gz=True, chunks=(None, _longest_line(text) + 5), name="b")
    _parity(tmp_path, caplog, edge_vcf(33, line_end="\r", final_newline=False, seed=4), gz=True, name="c")


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 31, 32, 33, 63, 64, 65, 1135, 2049])
def test_word_and_padding_boundaries(lib, tmp_path, caplog, S):
    _parity(tmp_path, caplog, edge_vcf(S, seed=S), chunks=(None, 3 * _longest_line(edge_vcf(S, seed=S))))


@pytest.mark.gpu
def test_chunks_of_one_line_and_runs_across_chunks(lib, tmp_path, caplog):
    text = edge_vcf(40, seed=1)
    n = _longest_line(text)
    # a chunk of about one line: every run of CHROM crosses chunks; a chunk of two lines ends some runs mid-way
    _parity(tmp_path, caplog, text, chunks=(n, 2 * n - 3))


@pytest.mark.gpu
def test_header_only_and_no_records(lib, tmp_path, caplog):
    _parity(tmp_path, caplog, "\n".join(META + [HEAD + "\ta\tb"]) + "\n", name="h")
    _parity(tmp_path, caplog, "\n".join(META + [HEAD + "\ta", "##x", "1\t2\t3"]) + "\n", name="i")


@pytest.mark.gpu
def test_info_dp_dot_is_never_flagged(lib, tmp_path, caplog):
    from snpmatch_b200.core import makedb
    text = "".join("%s\n" % l for l in META + [HEAD + "\ta\tb"]) + "".join(
        "1\t%d\t.\tA\tT\t.\tPASS\tDP=.;PL=x\tGT:GT\t0/1:1/1\t1|1\n" % p for p in range(1, 500))
    path = str(tmp_path / "dp.vcf")
    _write(path, text)
    tm = {}
    makedb.makeDB_from_vcf(path, str(tmp_path / "dp"), timings=tm).close()
    assert tm["flagged"] == []
    _parity(tmp_path, caplog, text, name="dp2")


@pytest.mark.gpu
def test_synthetic_panel_at_scale(lib, tmp_path):
    from snpmatch_b200.core import makedb
    A, R = 1135, 200000
    path = str(tmp_path / "panel.vcf.gz")
    with gzip.open(path, "wb", compresslevel=1) as fh:
        positions, regions = synth.panel_vcf(fh, R, A)
    tm = {}
    g = makedb.makeDB_from_vcf(path, str(tmp_path / "panel"), chunk_bytes=48 << 20, timings=tm)
    g.close()
    assert tm["flagged"] == []
    db = lib.Database(positions, regions, A)
    with np.load(str(tmp_path / "panel.npz")) as z:
        for r0 in range(0, R, 50000):
            db.load_int8(synth.panel_codes(synth.SEED_PANEL, np.arange(r0, r0 + 50000), A), row0=r0)
            assert np.array_equal(z["packed"][r0:r0 + 50000], db.read_packed(r0, 50000)), r0
        assert np.array_equal(z["positions"], positions) and np.array_equal(z["chr_regions"], regions)
        assert z["chrs"].tolist() == synth.TAIR10_CHRS and np.array_equal(z["accessions"], synth.accession_ids(A))
    db.close()


# ---- refusals ------------------------------------------------------------------------------------------------------------------
def _main_fails(tmp_path, capsys, path, match, extra=()):
    import snpmatch_b200
    before = sorted(os.listdir(tmp_path))
    with pytest.raises(SystemExit) as e:
        snpmatch_b200.main(["makedb", "-i", path, "-o", str(tmp_path / "out"), "--no_csv"] + list(extra))
    assert e.value.code == 1
    assert sorted(os.listdir(tmp_path)) == before, "nothing may be written"
    err = capsys.readouterr().err
    assert re.search(match, err), err


BODY = "".join("1\t%d\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n" % p for p in range(1, 40))
REFUSALS = {
    "more_fields": (BODY + "1\t50\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\t0/1\n" + BODY, "line 42 has 3 sample fields"),
    "fewer_fields": (BODY + "1\t50\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\n", "line 42 has 1 sample fields"),
    "hash_line": (BODY + "#x\n" + BODY, "line 42 is a '#' line"),
    "pos_na": (BODY + "1\tNA\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n", "line 42 has the POS 'NA'"),
    "chrom_comma": (BODY + "1,2\t50\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n", "line 42 has the CHROM '1,2'"),
    "chrom_quote": (BODY + '"1\t50\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n', "line 42 has the CHROM"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(REFUSALS))
def test_refusals_name_the_line(lib, tmp_path, capsys, case):
    body, match = REFUSALS[case]
    path = str(tmp_path / "r.vcf")
    _write(path, "##fileformat=VCFv4.2\n" + HEAD + "\ta\tb\n" + body)
    _main_fails(tmp_path, capsys, path, match)
    for chunk in (200, 1000):                 # the offending line in a later chunk
        from snpmatch_b200.core import makedb
        with pytest.raises(ValueError, match=match.replace("(", r"\(")):
            makedb.makeDB_from_vcf(path, str(tmp_path / "x"), chunk_bytes=chunk)
    assert not any(f.startswith("x.") for f in os.listdir(tmp_path))


@pytest.mark.gpu
def test_header_refusals(lib, tmp_path, capsys):
    cases = [(HEAD + "\n" + BODY.replace("\t0/0\t1/1", ""), "no sample columns"),
             (HEAD + "\ta,b\tc\n" + BODY, "sample column 1 .* 'a,b'"),
             (HEAD + '\ta\t"c\n' + BODY, "sample column 2"),
             (HEAD + "\ta\tcé\n" + BODY, "not ASCII"),
             ("##x\n" + BODY, "line 2 is a record before the #CHROM line"),
             ("##x\n", "no #CHROM line")]
    for k, (text, match) in enumerate(cases):
        path = str(tmp_path / ("h%d.vcf" % k))
        _write(path, text)
        _main_fails(tmp_path, capsys, path, match)


@pytest.mark.gpu
def test_line_longer_than_the_chunk(lib, tmp_path):
    from snpmatch_b200.core import makedb
    path = str(tmp_path / "l.vcf")
    _write(path, HEAD + "\ta\tb\n" + BODY + "1\t99\t.\tA\tT\t.\tPASS\t" + "x" * 500 + "\tGT\t0/0\t1/1\n")
    with pytest.raises(ValueError, match="line 41 is longer than the chunk of 300 bytes"):
        makedb.makeDB_from_vcf(path, str(tmp_path / "x"), chunk_bytes=300)
    assert sorted(os.listdir(tmp_path)) == ["l.vcf"]


@pytest.mark.gpu
def test_cli_writes_npz_and_json_only(lib, tmp_path):
    import snpmatch_b200
    from snpmatch_b200.core import snp_genotype
    path = str(tmp_path / "c.vcf")
    _write(path, edge_vcf(40))
    out = str(tmp_path / "db")
    assert snpmatch_b200.main(["makedb", "-i", path, "-o", out, "--no_csv"]) == 0
    assert sorted(os.listdir(tmp_path)) == ["c.vcf", "db.json", "db.npz"]
    g = snp_genotype.Genotype(out + ".npz")
    assert g.g.num_snps == len(SITES) and len(g.accessions) == 40
    g.close()
