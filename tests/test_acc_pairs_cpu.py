"""`pairsnp --accessions` without a GPU: the arguments and their refusals, the accession list, PanelIdentity's close pairs and
its TSV files."""
import numpy as np
import pytest

import snpmatch_b200
from snpmatch_b200.core import snpmatch


class _Panel(object):
    """What accession_indices reads of a Genotype."""
    accessions = np.array(["6909", "6046", "9321", "1001"])


def _result():
    # accessions a..e: a = b (identity 1), c shares 4 rows with a at 0.75, d and e share nothing, e has no called row
    common = np.array([[10, 8, 4, 0, 0],
                       [8, 9, 4, 2, 0],
                       [4, 4, 6, 3, 0],
                       [0, 2, 3, 5, 0],
                       [0, 0, 0, 0, 0]], np.int32)
    same = np.array([[10, 8, 3, 0, 0],
                     [8, 9, 3, 2, 0],
                     [3, 3, 6, 0, 0],
                     [0, 2, 0, 5, 0],
                     [0, 0, 0, 0, 0]], np.int32)
    return snpmatch.PanelIdentity(common, same, np.array(["a", "b", "c", "d", "e"]))


def test_identity_and_close_pairs_order():
    r = _result()
    ident = r.identity()
    assert np.isnan(ident[4]).all() and np.isnan(ident[0, 3])
    assert ident[0, 2] == 0.75 and ident[2, 2] == 1.0
    # identity 1 three ways: ties go in (i, j) order; 0.75 twice, then 0 (c-d shares 3 rows, none equal)
    assert r.close_pairs(0.0) == [("a", "b", 1.0, 8, 8), ("b", "d", 1.0, 2, 2), ("a", "c", 0.75, 4, 3), ("b", "c", 0.75, 4, 3),
                                  ("c", "d", 0.0, 3, 0)]
    assert r.close_pairs(0.8) == [("a", "b", 1.0, 8, 8), ("b", "d", 1.0, 2, 2)]
    assert r.close_pairs(0.75)[-1] == ("b", "c", 0.75, 4, 3)
    assert r.close_pairs(1.01) == []


def test_tsv_files(tmp_path):
    r = _result()
    out = str(tmp_path / "p")
    r.write(out)
    rows = [line.split("\t") for line in open(out + ".identity.tsv").read().splitlines()]
    assert rows[0] == ["sample", "a", "b", "c", "d", "e"]
    assert [x[0] for x in rows[1:]] == ["a", "b", "c", "d", "e"]
    assert rows[1][1:] == ["1.0", "1.0", "0.75", "nan", "nan"]
    rows = [line.split("\t") for line in open(out + ".common.tsv").read().splitlines()]
    assert rows[3] == ["c", "4", "4", "6", "3", "0"]
    assert not (tmp_path / "p.close_pairs.tsv").exists()
    r.write(out, min_identity=0.75)
    lines = open(out + ".close_pairs.tsv").read().splitlines()
    assert lines == ["acc_1\tacc_2\tidentity\tcommon\tsame", "a\tb\t1.0\t8\t8", "b\td\t1.0\t2\t2", "a\tc\t0.75\t4\t3", "b\tc\t0.75\t4\t3"]
    # the writer of `pairsnp --samples` with the ids as labels
    snpmatch.write_matrix_tsv(str(tmp_path / "w.tsv"), ["a", "b", "c", "d", "e"], r.common)
    assert open(str(tmp_path / "w.tsv")).read() == open(out + ".common.tsv").read()
    bad = snpmatch.PanelIdentity(r.common[:2, :2], r.same[:2, :2], np.array(["a", "a"]))
    with pytest.raises(ValueError, match="same label"):
        bad.write(out)


def test_accession_selection():
    g = _Panel()
    assert snpmatch.accession_indices(g, None).tolist() == [0, 1, 2, 3]
    assert snpmatch.accession_indices(g, ["1001", 6909, "9321"]).tolist() == [3, 0, 2]
    with pytest.raises(ValueError, match="accession 777 is not in the database"):
        snpmatch.accession_indices(g, ["6909", "777"])
    with pytest.raises(ValueError, match=r"accession 6046 is listed twice \(entries 0 and 2\)"):
        snpmatch.accession_indices(g, ["6046", "6909", "6046"])
    with pytest.raises(ValueError, match="empty"):
        snpmatch.accession_indices(g, [])


def test_accession_list_file(tmp_path, capsys):
    f = tmp_path / "ids.txt"
    f.write_text("9321\n\n  6909 \n1001\n")
    assert snpmatch_b200.read_accession_list(str(f)) == ["9321", "6909", "1001"]
    f.write_text("9321\n6909\n9321\n")
    with pytest.raises(SystemExit) as e:
        snpmatch_b200.read_accession_list(str(f))
    err = capsys.readouterr().err
    assert e.value.code == 1 and "9321 is listed twice" in err and "lines 1 and 3" in err
    f.write_text("\n")
    with pytest.raises(SystemExit):
        snpmatch_b200.read_accession_list(str(f))


def test_command_line_arguments(tmp_path, capsys):
    p = snpmatch_b200.get_options("t", "v")
    args = vars(p.parse_args(["pairsnp", "-d", "db.npz", "--accessions", "all", "--skip_db_hets", "--min_identity", "0.99", "-o", "x"]))
    assert args["accessions"] == "all" and args["skip_db_hets"] and args["min_identity"] == 0.99 and args["hdf5File"] == "db.npz"
    args = vars(p.parse_args(["pairsnp", "-i", "a.bed", "-j", "b.bed"]))
    assert args["accessions"] is None and not args["skip_db_hets"] and args["min_identity"] is None
    a = tmp_path / "a.bed"
    a.write_text("Chr1\t5\t0/0\n")
    db = tmp_path / "db.npz"
    db.write_bytes(b"")
    lst = tmp_path / "list.txt"
    lst.write_text("%s\n" % a)
    cases = [
        (["pairsnp", "--accessions", "all", "-o", "x"], "give the database with -d"),
        (["pairsnp", "--accessions", "all", "-d", str(db), "-i", str(a)], "cannot be combined"),
        (["pairsnp", "--accessions", "all", "-d", str(db), "-j", str(a)], "cannot be combined"),
        (["pairsnp", "--accessions", "all", "-d", str(db), "--samples", str(lst)], "cannot be combined"),
        (["pairsnp", "--accessions", str(tmp_path / "missing.txt"), "-d", str(db)], "does not exist"),
        (["pairsnp", "-i", str(a), "-j", str(a), "--min_identity", "0.9"], "go with --accessions"),
        (["pairsnp", "--samples", str(lst), "--skip_db_hets"], "go with --accessions"),
    ]
    for argv, msg in cases:
        with pytest.raises(SystemExit) as e:
            snpmatch_b200.main(argv)
        assert e.value.code == 1, argv
        assert msg in capsys.readouterr().err, argv


def test_sharded_panel_is_refused():
    class Db(object):
        row0_global, n_rows = 100, 50

    class G(object):
        db = Db()
        accessions = _Panel.accessions
        global_chr_regions = np.array([[0, 150]])
    with pytest.raises(ValueError, match="shard"):
        snpmatch.panel_identity(G())
