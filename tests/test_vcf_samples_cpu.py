"""`inbred --samples_vcf` / `cross --samples_vcf` without a GPU: the command-line checks (they fail before the panel is loaded),
the header reader, and the Python pieces the device parser shares with the single-sample path (parsers.vcf_record,
parsers.vcf_called_inputs) against the single-sample reader as it was before they were factored out."""
import gzip
import os
import re

import numpy as np
import pytest

from snpmatch_b200 import synth
from snpmatch_b200.core import parsers


# ---- the single-sample reader before vcf_record / vcf_called_inputs were factored out of it --------------------------------
def _old_read_vcf_minimal(inFile, sample_index=0):
    opener = gzip.open if str(inFile).endswith(".gz") else open
    chrom, pos, gts, pls, dps = [], [], [], [], []
    has_info_dp = False
    has_pl = False
    dp_re = re.compile(r"(?:^|;)DP=([^;]+)")
    with opener(inFile, "rt") as fh:
        for line in fh:
            if line.startswith("##"):
                if line.startswith("##INFO=<ID=DP,"):
                    has_info_dp = True
                continue
            if line.startswith("#"):
                continue
            f = line.rstrip("\n").split("\t")
            if len(f) < 10 + sample_index:
                continue
            chrom.append(f[0])
            pos.append(int(f[1]))
            m = dp_re.search(f[7])
            try:
                dps.append(int(m.group(1)) if m else -1)
            except ValueError:
                dps.append(-1)
            keys = f[8].split(":")
            vals = f[9 + sample_index].split(":")
            rec = dict(zip(keys, vals))
            alleles = re.split(r"[/|]", rec.get("GT", "."))
            if len(alleles) == 1:
                alleles = [alleles[0], "."] if alleles[0] != "." else [".", "."]
            gts.append("/".join(a if a != "" else "." for a in alleles[:2]))
            pl = [-1.0, -1.0, -1.0]
            if "PL" in rec:
                has_pl = True
                for i, v in enumerate(rec["PL"].split(",")[:3]):
                    if v not in (".", ""):
                        pl[i] = float(v)
            elif "PL" in keys:
                has_pl = True
            pls.append(pl)
    out = {"chr": np.array(chrom, dtype="str"), "pos": np.array(pos, dtype=np.int64), "gt": np.array(gts, dtype="str")}
    if has_pl:
        out["wei"] = np.array(pls, dtype=float).reshape(-1, 3)
    out["dp"] = np.array(dps, dtype=np.int64) if has_info_dp else np.repeat("NA", len(pos))
    return out


def _old_read_vcf(v):
    gt_all = v['gt']
    req = np.flatnonzero((gt_all != './.') & (gt_all != '.|.'))
    gt = gt_all[req]
    pl_codes = None
    if 'wei' in v:
        pl = v['wei'][req]
        no_pl = np.all(pl == -1, axis=1)
        wei = np.exp(pl / (-10))
        wei[no_pl, ] = parsers.ParseInputs.get_wei_from_GT(gt[no_pl])
        if len(pl) and np.all(pl == np.floor(pl)) and pl.min() >= -1 and pl.max() < 65000:
            top = int(pl.max()) + 1
            table = np.append(np.exp(np.arange(top) / (-10)), 0.0)
            codes = np.where(pl < 0, 0, pl).astype(np.uint16)
            if no_pl.any():
                hard = wei[no_pl]
                codes[no_pl] = np.where(hard == 1.0, 0, top).astype(np.uint16)
            if np.array_equal(table[codes.astype(np.int64)], wei):
                pl_codes = (codes, table)
    else:
        wei = parsers.ParseInputs.get_wei_from_GT(gt)
    return (v['chr'][req], v['pos'][req], gt, wei, v['dp'][req]), pl_codes


def _write(path, text):
    with open(path, "w", encoding="utf-8", newline="") as fh:
        fh.write(text)


CASES = {"lf": {}, "crlf": {"line_end": "\r\n"}, "cr": {"line_end": "\r"}, "mixed": {"line_end": ["\n", "\r\n", "\r"]},
         "no_dp_header": {"info_dp_header": False}, "late_dp": {"info_dp_header": False, "late_info_dp": True}}


@pytest.mark.parametrize("case", sorted(CASES))
def test_shared_helpers_equal_the_single_sample_reader(tmp_path, case):
    text, _ = synth.multi_sample_vcf(301, 37, seed=len(case), **CASES[case])
    path = str(tmp_path / "m.vcf")
    _write(path, text)
    for s in (0, 1, 17, 36):
        new, old = parsers.read_vcf_minimal(path, sample_index=s), _old_read_vcf_minimal(path, sample_index=s)
        assert sorted(new) == sorted(old)
        for k in old:
            assert new[k].dtype == old[k].dtype and np.array_equal(new[k], old[k]), (s, k)
        parsed, codes = parsers.vcf_called_inputs(new["chr"], new["pos"], new["gt"], new.get("wei"), new["dp"])
        ref, ref_codes = _old_read_vcf(old)
        for a, b in zip(parsed, ref):
            assert a.dtype == b.dtype and a.shape == b.shape
            if a.dtype == np.float64:
                assert np.array_equal(a.view(np.int64), b.view(np.int64))
            else:
                assert np.array_equal(a, b)
        assert (codes is None) == (ref_codes is None)
        if codes is not None:
            assert np.array_equal(codes[0], ref_codes[0]) and np.array_equal(codes[1].view(np.int64), ref_codes[1].view(np.int64))


def test_parse_inputs_of_a_vcf_unchanged(tmp_path):
    text, _ = synth.multi_sample_vcf(200, 3, seed=3)
    path = str(tmp_path / "one.vcf")
    _write(path, synth.split_vcf_column(text, 1))
    inp = parsers.ParseInputs(path)
    (chrs, pos, gt, wei, dp), codes = _old_read_vcf(_old_read_vcf_minimal(path))
    assert np.array_equal(inp.chrs, chrs) and np.array_equal(inp.pos, pos) and np.array_equal(inp.gt, gt)
    assert np.array_equal(inp.wei.view(np.int64), wei.view(np.int64)) and np.array_equal(inp.dp, dp)
    cw = inp.coded_weights()
    if codes is not None:
        assert np.array_equal(cw[0], codes[0]) and np.array_equal(cw[1], codes[1])


def test_vcf_record_skips_short_lines_and_keeps_python_semantics():
    f = "Chr1\t+12\t.\tA\tT\t.\tPASS\tDP=;ADP=3;DP=1_0\tGT:PL:GT\t0/1:3.5,1e2:1|1".split("\t")
    assert parsers.vcf_record(f, 0) == ("Chr1", 12, 10, "1/1", [3.5, 100.0, -1.0], True)
    assert parsers.vcf_record(f, 1) is None
    f = "Chr1\t5\t.\tA\tT\t.\tPASS\tDP=x\tAD:PL\t3\t4".split("\t")
    assert parsers.vcf_record(f, 1) == ("Chr1", 5, -1, "./.", [-1.0, -1.0, -1.0], True)


@pytest.mark.parametrize("end", ["\n", "\r\n", "\r"])
def test_header_reader(tmp_path, end):
    text, _ = synth.multi_sample_vcf(20, 5, seed=1, line_end=end)
    path = tmp_path / "h.vcf.gz"
    path.write_bytes(gzip.compress(text.encode("utf-8")))
    with gzip.open(path, "rb") as fh:
        names, has_dp, n, rest = parsers.read_vcf_header(fh, block=7)
    assert names == ["smp%d" % i for i in range(5)] and has_dp and n == 3
    assert rest.decode("utf-8") == text.split(end, 3)[3][:len(rest)]
    assert parsers.vcf_sample_names(str(path)) == names
    no_head = tmp_path / "r.vcf"
    _write(no_head, "##x\nChr1\t1\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\ta\n")
    with pytest.raises(ValueError, match="line 2"):
        parsers.vcf_sample_names(str(no_head))
    _write(no_head, "##x\n")
    with pytest.raises(ValueError, match="#CHROM"):
        parsers.vcf_sample_names(str(no_head))


def test_whole_lines_cut():
    assert parsers._whole_lines(bytearray(b"ab\ncd\r\nef"), 100, False) == 7
    assert parsers._whole_lines(bytearray(b"ab\ncd\r"), 100, False) == 3          # '\r' may be the first half of "\r\n"
    assert parsers._whole_lines(bytearray(b"ab\ncd\r"), 100, True) == 6
    assert parsers._whole_lines(bytearray(b"ab\rcd\r\n"), 6, False) == 3
    assert parsers._whole_lines(bytearray(b"abcdef\n"), 4, False) == 0


# ---- command line ------------------------------------------------------------------------------------------------------------
def _fails(argv, tmp_path, monkeypatch, code=1, match=None, capsys=None):
    import snpmatch_b200
    from snpmatch_b200.core import snp_genotype

    def no_panel(*a, **k):
        raise AssertionError("the panel must not be loaded")
    monkeypatch.setattr(snp_genotype.Genotype, "__init__", no_panel)
    before = sorted(os.listdir(tmp_path))
    with pytest.raises(SystemExit) as e:
        snpmatch_b200.main(argv)
    assert e.value.code == code
    assert sorted(os.listdir(tmp_path)) == before, "nothing may be written"
    if match is not None:
        assert re.search(match, capsys.readouterr().err)


HEAD = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"
REC = "\nChr1\t10\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t0/1\n"


@pytest.mark.parametrize("cmd", ["inbred", "cross"])
def test_samples_vcf_excludes_other_inputs(tmp_path, monkeypatch, cmd):
    vcf = tmp_path / "m.vcf"
    _write(vcf, HEAD + "\ta\tb" + REC)
    lst = tmp_path / "list.txt"
    lst.write_text("%s\n" % vcf)
    for other in (["-i", str(vcf)], ["--samples", str(lst)]):
        _fails([cmd, "--samples_vcf", str(vcf)] + other + ["-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "o")], tmp_path,
               monkeypatch, code=2)


@pytest.mark.parametrize("cmd", ["inbred", "cross"])
@pytest.mark.parametrize("columns,match", [("", "without sample columns"), ("\ta\t\tb", "column 2 .* name ''"),
                                           ("\ta\tb\ta", "sample name a appears twice"), ("\ta\tx/y", "column 2 .* 'x/y'")])
def test_samples_vcf_names_are_checked(tmp_path, monkeypatch, capsys, cmd, columns, match):
    vcf = tmp_path / "m.vcf"
    _write(vcf, HEAD + columns + REC)
    _fails([cmd, "--samples_vcf", str(vcf), "-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "o")], tmp_path, monkeypatch,
           match=match, capsys=capsys)


def test_samples_vcf_missing_file_and_record_before_header(tmp_path, monkeypatch, capsys):
    _fails(["inbred", "--samples_vcf", str(tmp_path / "none.vcf"), "-d", str(tmp_path / "db.npz")], tmp_path, monkeypatch)
    vcf = tmp_path / "m.vcf"
    _write(vcf, REC.lstrip("\n") + HEAD + "\ta\tb" + REC)
    _fails(["inbred", "--samples_vcf", str(vcf), "-d", str(tmp_path / "db.npz")], tmp_path, monkeypatch, match="line 1 is a record",
           capsys=capsys)
