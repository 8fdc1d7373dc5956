"""`makedb --no_csv` without a device: the header reader hands back the '##' lines vcf_to_csv collects, the CSV route's reading of
CHROM and POS texts, the refusals are inputs the CSV route (vcf_to_csv + load_csv + makeDB's accession check) fails on too, and
the command-line refusals that need no device."""
import os
import re

import numpy as np
import pytest

from snpmatch_b200.core import makedb, parsers

HEAD = "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"
BODY = "".join("1\t%d\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n" % p for p in range(1, 40))


def _write(path, text):
    with open(path, "w", encoding="utf-8", newline="") as fh:
        fh.write(text)


@pytest.mark.parametrize("end", ["\n", "\r\n", "\r"])
def test_header_meta_lines_are_the_ones_vcf_to_csv_collects(tmp_path, end):
    meta = ["##fileformat=VCFv4.2", "##contig=<ID=1,length=3000>", "##contig=<ID=Chr2,length=20,assembly=x>", "##x=<a>"]
    text = end.join(meta[:2] + ["short\tline"] + meta[2:] + [HEAD + "\ta", "##contig=<ID=9,length=99>", "1\t5\t.\tA\tT\t.\tPASS\t.\tGT\t0/0"]) + end
    path = str(tmp_path / "h.vcf")
    _write(path, text)
    got = []
    with parsers._open_binary(path) as fh:
        names, _, n, _ = parsers.read_vcf_header(fh, meta_lines=got)
    assert got == meta and names == ["a"] and n == 6
    makedb.vcf_to_csv(path, str(tmp_path / "ref"))
    with open(str(tmp_path / "ref.json")) as js:
        assert js.read() == __import__("json").dumps(makedb.get_contigs(got), sort_keys=True, indent=4)


def test_csv_reading_of_chrom_and_pos():
    labels, bad = makedb._csv_read(["1", "NA", "nan", "N/A", " 1 ", "Chré", "null"], "CHROM")
    assert bad is None and labels.tolist() == ["1", "nan", "nan", "nan", " 1 ", "Chré", "nan"]
    pos, bad = makedb._csv_read(["+5", "007", "1_0", "3000000000", " 12", "8"], "POS")
    assert bad is None and pos.dtype == np.int32 and pos.tolist() == [5, 7, 10, -1294967296, 12, 8]
    assert makedb._csv_read(["5", "6", "NA", "1e3"], "POS") == (None, 2)
    assert makedb._csv_read(["", "5"], "POS") == (None, 0)


def test_index_arrays_runs(tmp_path):
    p = str(tmp_path / "a.csv")
    _write(p, "Chromosome,Position,a\n1,5,0\n1,6,0\n2,1,1\n1,9,2\nNA,3,0\nnan,4,0\n")
    chrs, regions, positions = makedb._index_arrays(p, ",")
    assert chrs.tolist() == ["1", "2", "1", "nan"] and chrs.dtype == np.dtype("<U3")
    assert regions.tolist() == [[0, 2], [2, 3], [3, 4], [4, 6]] and positions.tolist() == [5, 6, 1, 9, 3, 4]


# every input makeDB_from_vcf refuses, as a whole file: the CSV route fails on it too
REFUSED = {
    "more_fields_first": HEAD + "\ta\tb\n" + "1\t50\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\t0/1\n" + BODY,
    "fewer_fields": HEAD + "\ta\tb\n" + BODY + "1\t50\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\n",
    "hash_line": HEAD + "\ta\tb\n" + BODY + "#x\n" + BODY,
    "pos_na": HEAD + "\ta\tb\n" + BODY + "1\tNA\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n",
    "pos_exponent": HEAD + "\ta\tb\n" + BODY + "1\t1e3\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n",
    "chrom_quote": HEAD + "\ta\tb\n" + BODY + '"1\t50\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n',
    "sample_comma": HEAD + "\ta,b\tc\n" + BODY,
    "sample_quote": HEAD + '\ta\t"c\n' + BODY,
    "no_samples": HEAD + "\n" + BODY.replace("\t0/0\t1/1", ""),
    "no_chrom_line": "##x\n",
    "record_first": "##x\n" + BODY + HEAD + "\ta\tb\n",
    "non_ascii_sample": HEAD + "\ta\tcé\n" + BODY,
}


@pytest.mark.parametrize("case", sorted(REFUSED))
def test_refused_inputs_fail_the_csv_route(tmp_path, case):
    path = str(tmp_path / "r.vcf")
    _write(path, REFUSED[case])
    out = str(tmp_path / "ref")
    with pytest.raises(Exception):
        makedb.vcf_to_csv(path, out)
        d = makedb.load_csv(out + ".csv")
        assert len(d["accessions"]) > 0, "makeDB: the CSV holds no accession columns"
        d["accessions"].astype("S")


def test_refused_inputs_the_csv_route_misreads(tmp_path):
    """Two refusals the CSV route does not always fail on: it reads the row wrongly instead.  A record with more sample fields
    than the header, after the first record, loses its extra calls without a word (pandas drops the fields past usecols); a
    ',' in CHROM shifts the row, so POS lands in the first genotype column (makeDB's load then fails on a code above 2, or
    stores the POS as a genotype call when it is 0, 1 or 2)."""
    more = HEAD + "\ta\tb\n" + BODY + "1\t50\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\t0/1\n"
    comma = HEAD + "\ta\tb\n" + BODY + "1,2\t1\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n"
    for text, check in ((more, lambda d: d["snps"].shape == (40, 2) and d["snps"][-1].tolist() == [0, 1]),
                        (comma, lambda d: d["positions"][-1] == 2 and d["snps"][-1].tolist() == [1, 0])):
        path = str(tmp_path / "r.vcf")
        _write(path, text)
        makedb.vcf_to_csv(path, str(tmp_path / "ref"))
        assert check(makedb.load_csv(str(tmp_path / "ref.csv")))


def _fails(argv, tmp_path, capsys, match):
    import snpmatch_b200
    before = sorted(os.listdir(tmp_path))
    with pytest.raises(SystemExit) as e:
        snpmatch_b200.main(argv)
    assert e.value.code == 1
    assert sorted(os.listdir(tmp_path)) == before, "nothing may be written"
    assert re.search(match, capsys.readouterr().err)


def test_no_csv_needs_a_vcf(tmp_path, capsys):
    csv = tmp_path / "p.csv"
    csv.write_text("Chromosome,Position,a\n1,5,0\n")
    _fails(["makedb", "-i", str(csv), "-o", str(tmp_path / "db"), "--no_csv"], tmp_path, capsys, "--no_csv .* not one")
    _fails(["makedb", "-i", str(tmp_path / "none.vcf"), "-o", str(tmp_path / "db"), "--no_csv"], tmp_path, capsys, "does not exist")


def test_no_csv_header_refusals_need_no_device(tmp_path, capsys, monkeypatch):
    """Refusals of the header come before the device is touched."""
    from snpmatch_b200 import lib

    def no_device(*a, **k):
        raise AssertionError("the device must not be used")
    monkeypatch.setattr(lib, "VcfParser", no_device)
    for k, (case, match) in enumerate([("no_samples", "no sample columns"), ("sample_comma", "sample column 1 .* 'a,b'"),
                                       ("non_ascii_sample", "not ASCII"), ("no_chrom_line", "no #CHROM line"),
                                       ("record_first", "line 2 is a record before the #CHROM line")]):
        path = tmp_path / ("h%d.vcf" % k)
        _write(str(path), REFUSED[case])
        _fails(["makedb", "-i", str(path), "-o", str(tmp_path / "db"), "--no_csv"], tmp_path, capsys, match)
