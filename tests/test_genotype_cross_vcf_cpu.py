"""`genotype_cross --gpu_parse` without a device: the header refusals exit before the database or the VCF parser touch the device,
what the text route (read_vcf_samples) does on each input the device route refuses, and the flag reaching genotype_cross."""
import os
import re

import numpy as np
import pytest

from snpmatch_b200.core import parsers

HEAD = "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"
BODY = "".join("1\t%d\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n" % p for p in range(1, 40))

REFUSED = {
    "hash_line": HEAD + "\ta\tb\n" + BODY + "#x\n" + BODY,
    "hash_line_same_width": HEAD + "\ta\tb\n" + BODY + "#x\t1\t2\t3\t4\t5\t6\t7\t8\tc\td\n" + BODY,
    "pos_na": HEAD + "\ta\tb\n" + BODY + "1\tNA\t.\tA\tT\t.\tPASS\t.\tGT\t0/0\t1/1\n",
    "no_samples": HEAD + "\n" + BODY,
    "no_chrom_line": "##x\n" + BODY,
    "header_only_meta": "##x\n##y\n",
    "record_first": "##x\n" + BODY + HEAD + "\ta\tb\n" + BODY,
    "long_line": HEAD + "\ta\tb\n" + BODY + "1\t50\t.\tA\tT\t.\tPASS\t.\tGT:XX\t0/0:" + "x" * 5000 + "\t1/1:y\n",
}


def _write(path, text):
    with open(path, "w", encoding="utf-8", newline="") as fh:
        fh.write(text)


def test_text_route_on_the_refused_inputs(tmp_path):
    """What read_vcf_samples makes of each input read_vcf_gt_codes refuses: a mid-file '#' line resets the samples, so ragged
    rows raise, or the samples are silently renamed when the widths match; a POS int() rejects raises; no #CHROM line and no
    sample columns give zero samples; a record before the #CHROM line gives ragged rows; an over-long line reads as any other."""
    def read(case):
        path = str(tmp_path / (case + ".vcf"))
        _write(path, REFUSED[case])
        return parsers.read_vcf_samples(path)
    for case in ("hash_line", "record_first", "pos_na"):
        with pytest.raises(ValueError):
            read(case)
    r = read("hash_line_same_width")
    assert r["samples"].tolist() == ["c", "d"] and r["gt"].shape == (78, 2)
    for case in ("no_samples", "no_chrom_line"):
        r = read(case)
        assert r["samples"].shape == (0,) and r["gt"].shape == (39, 0)
    assert read("header_only_meta")["gt"].shape == (0, 0)
    r = read("long_line")
    assert r["gt"].shape == (40, 2) and r["gt"][-1].tolist() == ["0/0", "1/1"]


def _fails(argv, tmp_path, capsys, match):
    import snpmatch_b200
    before = sorted(os.listdir(tmp_path))
    with pytest.raises(SystemExit) as e:
        snpmatch_b200.main(argv)
    assert e.value.code == 1
    assert sorted(os.listdir(tmp_path)) == before, "nothing may be written"
    assert re.search(match, capsys.readouterr().err)


def test_header_refusals_need_no_device(tmp_path, capsys, monkeypatch):
    from snpmatch_b200 import lib

    def no_device(*a, **k):
        raise AssertionError("the device must not be used")
    monkeypatch.setattr(lib, "VcfParser", no_device)
    monkeypatch.setattr(lib, "Database", no_device)
    for k, (case, match) in enumerate([("no_samples", "no sample columns"), ("header_only_meta", "no #CHROM line"),
                                       ("no_chrom_line", "line 2 is a record before the #CHROM line"), ("record_first", "line 2 is a record before the #CHROM line")]):
        path = str(tmp_path / ("h%d.vcf" % k))
        _write(path, REFUSED[case])
        _fails(["genotype_cross", "-i", path, "-d", str(tmp_path / "db.npz"), "-p", "1x2", "-o", str(tmp_path / "out.csv"),
                "--gpu_parse"], tmp_path, capsys, match)


@pytest.mark.parametrize("flag", [False, True])
def test_gpu_parse_reaches_genotype_cross(tmp_path, monkeypatch, flag):
    from snpmatch_b200.core import genotype_cross as gtm
    import snpmatch_b200
    seen = {}

    class Fake(object):
        def __init__(self, *a, **k):
            pass

        def genotype_cross(self, input_file, lr_thres, good_samples_file=None, gpu_parse=False):
            seen.update(input_file=input_file, lr_thres=lr_thres, gpu_parse=gpu_parse)
            return np.array(["id,,,a,b"])

        write_output_genotype_cross = staticmethod(gtm.GenotypeCross.write_output_genotype_cross)
    monkeypatch.setattr(gtm.snp_genotype, "Genotype", lambda *a: None)
    monkeypatch.setattr(gtm, "GenotypeCross", Fake)
    path = str(tmp_path / "p.vcf")
    _write(path, HEAD + "\ta\tb\n" + BODY)
    out = str(tmp_path / "out.csv")
    argv = ["genotype_cross", "-i", path, "-d", "db.npz", "-p", "1x2", "--lr_thres", "2.5", "-o", out] + (["--gpu_parse"] if flag else [])
    assert snpmatch_b200.main(argv) == 0
    assert seen == dict(input_file=path, lr_thres=2.5, gpu_parse=flag)
    assert open(out).read() == "id,,,a,b\n"
