"""Host side of `pairsnp --samples` without a GPU: the union of markers and the chromosome ranges, the GT-string classes, the
TSV writer's label rules and the command line's arguments."""
import os

import numpy as np
import pytest

import snpmatch_b200
from snpmatch_b200.core import snpmatch


def _key(cid, pos):
    return (np.asarray(cid, np.int64) << 32) | (np.asarray(pos, np.int64) + 2**31)


def test_union_columns_and_chromosome_ranges():
    # sample 0 lists chromosome 2 before chromosome 0; sample 2 is empty; chromosome 1 is nobody's
    k0 = np.concatenate([_key([2, 2], [5, 9]), _key([0, 0, 0], [-3, 7, 100])])
    k1 = _key([0, 0, 2, 3], [7, 8, 9, 1])
    k3 = _key([3], [1])
    keys = np.concatenate([k0, k1, k3])
    cls = np.arange(len(keys), dtype=np.uint8) % 3
    offsets, col, mcls, union = snpmatch.build_pair_columns(keys, [5, 4, 0, 1], cls, "cpu")
    want_union = np.sort(np.unique(keys))
    assert np.array_equal(union, want_union)
    assert offsets.tolist() == [0, 5, 9, 9, 10]
    for s, k in enumerate([k0, k1, np.zeros(0, np.int64), k3]):
        seg = slice(offsets[s], offsets[s + 1])
        assert np.all(np.diff(col[seg]) > 0)
        assert np.array_equal(union[col[seg]], np.sort(k))
        c = cls[sum(len(x) for x in [k0, k1, np.zeros(0), k3][:s]):][:len(k)]
        assert np.array_equal(mcls[seg], c[np.argsort(k)])
    chr_start = np.searchsorted(union >> 32, np.arange(5))
    assert chr_start.tolist() == [0, 4, 4, 6, 7]                # chromosome 1 has no column; each range is contiguous


def test_union_restricted_to_database_positions():
    keys = np.concatenate([_key([0, 0, 1], [1, 2, 3]), _key([0, 1], [2, 4])])
    cls = np.array([0, 1, 2, 1, 0], np.uint8)
    offsets, col, mcls, union = snpmatch.build_pair_columns(keys, [3, 2], cls, "cpu", restrict=lambda u: (u & 0xFFFFFFFF) - 2**31 != 3)
    assert ((union & 0xFFFFFFFF) - 2**31).tolist() == [1, 2, 4]
    assert offsets.tolist() == [0, 2, 4]
    assert col.tolist() == [0, 1, 1, 2] and mcls.tolist() == [0, 1, 1, 0]


def test_gt_classes():
    gts = np.array(["0/0", "1|1", "1/1", "./.", "0/0", "1|1", "0/1"])
    codes, uniq = snpmatch.gt_classes(gts)
    assert len(uniq) == 5 and np.array_equal(uniq[codes], gts)
    long = np.array(["0/0/1", "0/0", "0/0/1"])                  # wider than three characters: the pandas path
    codes, uniq = snpmatch.gt_classes(long)
    assert np.array_equal(uniq[codes], long)
    codes, uniq = snpmatch.gt_classes(np.array(["1", "11", "1"]))
    assert codes.tolist() == [0, 1, 0]


def test_tsv_writer_labels(tmp_path):
    pm = snpmatch.PairMatrix(np.array([[[3, 0], [0, 2]], [[1, 0], [0, 0]]]), np.array([[[3, 0], [0, 1]], [[0, 0], [0, 0]]]),
                             np.array(["1", "2"]), [np.array([0, 1]), np.array([0])], np.array([4, 2]), ["/d/a.bed", "/e/b.vcf"])
    out = str(tmp_path / "p")
    pm.write(out)
    rows = [line.split("\t") for line in open(out + ".identity.tsv").read().splitlines()]
    assert rows[0] == ["sample", "a.bed", "b.vcf"]
    assert rows[1][0] == "a.bed" and float(rows[1][1]) == 0.75 and rows[1][2] == "nan"
    assert rows[2][0] == "b.vcf" and float(rows[2][2]) == 0.5
    rows = [line.split("\t") for line in open(out + ".common.tsv").read().splitlines()]
    assert rows[1:] == [["a.bed", "4", "0"], ["b.vcf", "0", "2"]]
    assert not os.path.exists(out + ".pairs.jsonl")
    pm.write(out, labels=["x", "y"])
    assert open(out + ".common.tsv").readline() == "sample\tx\ty\n"
    for bad in (["x", "x"], ["x"], ["x\ty", "z"], ["", "z"]):
        with pytest.raises(ValueError):
            pm.write(out, labels=bad)
    same_base = snpmatch.PairMatrix(pm.common, pm.same, pm.chromosomes, pm._chr_ids, pm.n_markers, ["/d/a.bed", "/e/a.bed"])
    with pytest.raises(ValueError, match="same label"):
        same_base.write(out)


def test_pairsnp_samples_arguments(tmp_path):
    a, b = tmp_path / "a.bed", tmp_path / "b.bed"
    a.write_text("Chr1\t5\t0/0\n")
    b.write_text("Chr1\t5\t1/1\n")
    lst = tmp_path / "list.txt"
    lst.write_text("%s\n%s\tsecond\n" % (a, b))
    p = snpmatch_b200.get_options("t", "v")
    args = vars(p.parse_args(["pairsnp", "--samples", str(lst), "-o", "x", "--pairs_json"]))
    assert args["samples"] == str(lst) and args["pairs_json"] and args["inFile_1"] is None
    assert not vars(p.parse_args(["pairsnp", "-i", str(a), "-j", str(b)]))["pairs_json"]
    with pytest.raises(SystemExit):
        snpmatch_b200.main(["pairsnp", "--samples", str(lst), "-i", str(a)])
    assert snpmatch_b200.read_sample_list(str(lst), "x", default_name=os.path.basename) == [(str(a), "a.bed"), (str(b), "second")]
    dup = tmp_path / "dup.txt"
    dup.write_text("%s\n%s\ta.bed\n" % (a, b))
    with pytest.raises(SystemExit):
        snpmatch_b200.read_sample_list(str(dup), "x", default_name=os.path.basename)
    empty = tmp_path / "empty.txt"
    empty.write_text("\n")
    with pytest.raises(SystemExit):
        snpmatch_b200.read_sample_list(str(empty), "x", default_name=os.path.basename)


def test_refusals_before_device_work(tmp_path):
    from snpmatch_b200.core import parsers
    with pytest.raises(ValueError, match="empty"):
        snpmatch.pairwise_score_many([])

    def inp(chrs, pos, gt):
        x = parsers.ParseInputs("")
        x.load_snp_info(np.array(chrs), np.array(pos), np.array(gt), np.ones((len(pos), 3)), "NA")
        return x
    ok = inp(["1", "1"], [1, 2], ["0/0", "1/1"])
    with pytest.raises(ValueError, match=r"sample 1 \(dup\).*1:7 appears more than once"):
        snpmatch.pairwise_score_many([ok, inp(["Chr1", "2", "chr1"], [7, 3, 7], ["0/0"] * 3)], names=["ok", "dup"])
    nine = inp(["1"] * 9, np.arange(9), ["%d/%d" % (k, k) for k in range(9)])
    with pytest.raises(ValueError, match="9 distinct GT strings"):
        snpmatch.pairwise_score_many([ok, nine])
    with pytest.raises(ValueError, match="sample 0.*position 2147483647"):
        snpmatch.pairwise_score_many([inp(["1"], [2**31 - 1], ["0/0"])])
    from snpmatch_b200 import lib
    with pytest.raises(ValueError, match="at most %d" % lib.PAIR_MAX_SAMPLES):
        snpmatch.pairwise_score_many([ok] * (lib.PAIR_MAX_SAMPLES + 1))
