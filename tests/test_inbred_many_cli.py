"""`inbred --samples` input checks: they fail before the panel is loaded, so they run without a GPU."""
import os

import pytest


def _write_bed(path, s):
    with open(path, "w") as fh:
        for c, pos, gt in zip(s["chrs"], s["pos"], s["gt"]):
            fh.write("%s\t%d\t%s\n" % (c, pos, gt))


def _bed_files(tmp_path, sample_inbred, n=2):
    paths = []
    for i in range(n):
        paths.append(str(tmp_path / ("s%d.sample.bed" % i)))
        _write_bed(paths[-1], sample_inbred)
    return paths


def _fails(argv, tmp_path, monkeypatch):
    import snpmatch_b200
    from snpmatch_b200.core import snp_genotype

    def no_panel(*a, **k):
        raise AssertionError("the panel must not be loaded")
    monkeypatch.setattr(snp_genotype.Genotype, "__init__", no_panel)
    before = sorted(os.listdir(tmp_path))
    with pytest.raises(SystemExit) as e:
        snpmatch_b200.main(argv)
    assert e.value.code != 0
    assert sorted(os.listdir(tmp_path)) == before, "nothing may be written"


def test_input_and_samples_exclusive(tmp_path, sample_inbred, monkeypatch):
    a, _ = _bed_files(tmp_path, sample_inbred)
    lst = tmp_path / "list.txt"
    lst.write_text("%s\n" % a)
    _fails(["inbred", "-i", a, "--samples", str(lst), "-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "out")], tmp_path, monkeypatch)


def test_empty_list_and_missing_file(tmp_path, sample_inbred, monkeypatch):
    a, _ = _bed_files(tmp_path, sample_inbred)
    lst = tmp_path / "list.txt"
    lst.write_text("\n  \n")
    _fails(["inbred", "--samples", str(lst), "-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "out"), "--refine"], tmp_path, monkeypatch)
    lst.write_text("%s\n%s\n" % (a, tmp_path / "missing.bed"))
    _fails(["inbred", "--samples", str(lst), "-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "out")], tmp_path, monkeypatch)
    _fails(["inbred", "--samples", str(tmp_path / "no_list.txt"), "-d", str(tmp_path / "db.npz")], tmp_path, monkeypatch)


def test_duplicate_prefixes(tmp_path, sample_inbred, monkeypatch):
    a, b = _bed_files(tmp_path, sample_inbred)
    lst = tmp_path / "list.txt"
    lst.write_text("%s\tsame\n%s\tsame\n" % (a, b))
    _fails(["inbred", "--samples", str(lst), "-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "out")], tmp_path, monkeypatch)
    os.makedirs(tmp_path / "d")
    c = str(tmp_path / "d" / "s0.other.bed")
    _write_bed(c, sample_inbred)
    lst.write_text("%s\n%s\n" % (a, c))                     # the same default prefix <out>.s0
    _fails(["inbred", "--samples", str(lst), "-d", str(tmp_path / "db.npz"), "-o", str(tmp_path / "out")], tmp_path, monkeypatch)


def test_launch_budget_from_shapes():
    from snpmatch_b200.core import snpmatch
    small = snpmatch.inbred_bytes_per_sample(50000, 1135, 36)
    assert 4 << 20 < small < 16 << 20
    assert snpmatch.inbred_bytes_per_sample(50000, 20000, 626) > 5 * small
    assert snpmatch.inbred_bytes_per_sample(50000, 1135, 36, chunk_size=100) > small
