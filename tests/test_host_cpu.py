"""CPU-side checks: the C-ABI library builds, loads and exports every declared symbol; host logic
(identity table, window geometry, marker preparation, parsers) against the oracle / golden facts."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT, load_golden
from oracle import snpmatch_oracle as orc
from snpmatch_b200 import synth


@pytest.fixture(scope="module")
def built_lib():
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib
    return lib


def test_library_exports_every_declared_symbol(built_lib):
    lib = built_lib
    header = open(os.path.join(ROOT, "include", "snpmatch_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(snpm_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 30
    handle = lib.load()
    for name in sorted(declared):
        assert hasattr(handle, name), "libsnpmatch_b200.so does not export %s" % name
    assert declared == set(lib.SIGNATURES), "lib.py binds %s" % sorted(declared ^ set(lib.SIGNATURES))
    assert handle.snpm_version() == 100


def test_no_device_is_a_loud_failure(built_lib):
    lib = built_lib
    if lib.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(lib.SnpmError):
        lib.Database(np.arange(1, 11, dtype=np.int32), np.array([[0, 10]]), 4)
    with pytest.raises(lib.SnpmError):
        lib.match_gts_accs(np.ones((2, 3)), np.zeros((2, 4), dtype=np.int8))


def test_identity_table_matches_bruteforce():
    from snpmatch_b200.core import snpmatch
    for e in (0.02, 0.0005, 0.1):
        fast = snpmatch.identity_kmax_table(1500, e)
        slow = orc.identity_kmax_table(1500, e)
        assert np.array_equal(fast[:1501], slow)
    g = load_golden("epilogue.npz")
    assert np.array_equal(snpmatch.np_test_identity(g["id_x"], g["id_n"], error_rate=0.02), g["id_e02"])
    assert np.array_equal(snpmatch.np_test_identity(g["id_xf"], g["id_n"], error_rate=0.02), g["id_e02_f"])
    assert np.array_equal(snpmatch.np_test_identity(g["id_x"], g["id_n"]), g["id_default"])


def test_window_geometry():
    from snpmatch_b200.core import genomes
    gen = genomes.Genome("athaliana_tair10")
    assert gen.chrs_ids.tolist() == ["1", "2", "3", "4", "5"]
    cnt, off, n, winds = gen.window_layout(np.array(["Chr1", "chr2", "3", "4", "5"]), 300000)
    assert n == 399 and cnt.tolist() == [102, 66, 79, 62, 90] and off.tolist() == [0, 102, 168, 247, 309]
    assert len(winds) == 399 and winds[0] == "1" and winds[-1] == "5"
    # a database that lists the chromosomes in another order, plus one the genome lacks (count 0)
    gen2 = genomes.Genome("athaliana_tair10")
    gen2.chrs_ids = np.array(["1", "2", "3", "4", "5", "c"])
    gen2.chrlen = np.append(gen2.chrlen, 1000)
    cnt, off, n, _ = gen2.window_layout(np.array(["5", "1", "C"]), 300000)
    assert cnt.tolist() == [90, 102, 1] and off.tolist() == [309, 0, 399] and n == 400
    # iterator API against a brute-force binning
    rng = np.random.default_rng(5)
    pos = np.sort(rng.choice(2_000_000, size=500, replace=False)) + 1
    bins = list(genomes.get_bins_echr(1_900_000, pos, 300000, 7))
    assert len(bins) == orc.num_windows(1_900_000, 300000) == 7
    for k, (bed, idx) in enumerate(bins):
        assert bed == [1 + k * 300000, (k + 1) * 300000]
        want = [i + 7 for i, p in enumerate(pos) if bed[0] <= p <= bed[1]]
        assert idx == want
    assert np.array_equal(orc.window_of(pos, 1_900_000, 300000) >= 0, pos <= 7 * 300000)


def test_prepare_markers_orders_like_the_reference_join():
    from snpmatch_b200.core import snp_genotype
    g = object.__new__(snp_genotype.Genotype)
    g.chrs = np.array(["Chr1", "Chr3", "chrC"])
    g._db_chr_norm = snp_genotype.normalize_chr_names(g.chrs)
    chrs = np.array(["1", "1", "1", "2", "2", "ChrM", "ChrM", "C", "C"])
    pos = np.array([9, 12, 13, 1, 2, 5, 6, 8, 9])
    order, cid, p = g.prepare_markers(chrs, pos)
    assert cid.tolist() == [0, 0, 0, 2, 2, -1, -1, -1, -1]
    assert order.tolist() == [0, 1, 2, 7, 8, 3, 4, 5, 6] and p.tolist() == [9, 12, 13, 8, 9, 1, 2, 5, 6]
    # unsorted chromosome -> sorted for the join; duplicates keep the first
    order, cid, p = g.prepare_markers(np.array(["1", "1", "1", "1"]), np.array([30, 10, 20, 10]))
    assert p[cid >= 0].tolist() == [10, 20, 30] and sorted(order.tolist()) == [0, 1, 2, 3]
    assert order[:3].tolist() == [1, 2, 0]


def test_synthetic_panel_is_block_addressable():
    a = synth.panel_codes(synth.SEED_PANEL, np.arange(100, 140), 70)
    b = synth.panel_codes_cols(synth.SEED_PANEL, np.arange(110, 120), np.arange(5, 50))
    assert np.array_equal(a[10:20, 5:50], b)
    pos, regions = synth.panel_positions(50000)
    for s, e in regions:
        assert np.all(np.diff(pos[s:e]) > 0)
    assert regions[-1, 1] == 50000


def test_pack_reference_layout():
    rng = np.random.default_rng(3)
    snps = rng.choice(np.array([-1, 0, 1, 2], dtype=np.int8), size=(5, 70))
    packed = orc.pack_2bit_words(snps)
    assert packed.shape == (5, 4) and packed.dtype == np.uint64     # 3 words padded to 4
    for r in range(5):
        for a in range(70):
            w = int(packed[r, a // 32])
            code = ((w >> (a % 32)) & 1) | ((((w >> 32) >> (a % 32)) & 1) << 1)
            assert code == (int(snps[r, a]) & 3)
    assert int(packed[0, 3]) == 2**64 - 1 and (int(packed[0, 2]) >> 6) & 1 == 1    # padding = missing


def _write_sample_vcf(path, g):
    """The kept records of the reference's sample file 701_501.filter.vcf, as the reference parsed them (golden
    vcf701_sample.npz), written back as VCF text: integer PL = -10 ln(wei) (exact for every record), INFO/DP and FORMAT
    GT:AD:DP:GQ:PL of that file.  After every third record a no-call record (three spellings) that the parser must drop.
    Returns the number of no-call records written."""
    with np.errstate(divide="ignore"):
        pl = np.rint(-10.0 * np.log(g["wei"])).astype(np.int64)
    dp = g["dp"].astype(np.int64)
    no_calls = ["./.:0,0:0:.:.", ".|.:.:.:.:.", "."]
    dropped = 0
    with open(path, "w") as fh:
        fh.write("##fileformat=VCFv4.2\n"
                 "##INFO=<ID=DP,Number=1,Type=Integer,Description=\"Approximate read depth\">\n"
                 "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">\n"
                 "##FORMAT=<ID=AD,Number=R,Type=Integer,Description=\"Allelic depths\">\n"
                 "##FORMAT=<ID=DP,Number=1,Type=Integer,Description=\"Read depth\">\n"
                 "##FORMAT=<ID=GQ,Number=1,Type=Integer,Description=\"Genotype quality\">\n"
                 "##FORMAT=<ID=PL,Number=G,Type=Integer,Description=\"Phred-scaled genotype likelihoods\">\n"
                 "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t701_501\n")
        n = len(g["pos"])
        for i in range(n):
            c, p = str(g["chrs"][i]), int(g["pos"][i])
            fh.write("%s\t%d\t.\tA\tT\t.\t.\tDP=%d\tGT:AD:DP:GQ:PL\t%s:.:%d:.:%d,%d,%d\n" % (c, p, dp[i], g["gt"][i], dp[i], *pl[i]))
            nxt = (str(g["chrs"][i + 1]), int(g["pos"][i + 1])) if i + 1 < n else None
            if i % 3 == 2 and nxt != (c, p + 1):
                fh.write("%s\t%d\t.\tA\tT\t.\t.\tDP=0\tGT:AD:DP:GQ:PL\t%s\n" % (c, p + 1, no_calls[dropped % 3]))
                dropped += 1
    return dropped


def test_parsers_on_the_reference_sample_files(tmp_path, golden_outputs):
    """VCF and BED readers on the records of the reference's sample file, against the reference's own parse of it."""
    from snpmatch_b200.core import parsers
    g = load_golden("vcf701_sample.npz")
    vcf = tmp_path / "701_501.filter.vcf"                                    # the parser writes next to its input
    bed = tmp_path / "701_501.filter.bed"
    assert _write_sample_vcf(str(vcf), g) > 2000
    v = parsers.ParseInputs(str(vcf))
    facts = golden_outputs["facts"]
    assert len(v.chrs) == 7545 == facts["vcf_kept"]                          # tests/test_inbred.py:9-12
    assert v.chrs[0] == "Chr1" and v.gt[0] == "0/0" and int(v.pos[0]) == 13226
    np.testing.assert_allclose(v.wei.sum(axis=0), [6582.58869952, 3247.44885746, 903.85454402], rtol=1e-9)
    np.testing.assert_allclose(v.wei[0], [1.0, 0.40656966, 1.66585811e-04], rtol=1e-7)
    assert np.array_equal(v.pos, g["pos"]) and np.array_equal(v.wei, g["wei"]) and np.array_equal(v.gt, g["gt"])
    assert np.array_equal(v.chrs, g["chrs"]) and np.array_equal(v.dp, g["dp"])
    np.testing.assert_allclose(parsers.mean_depth(v.dp), facts["vcf_dp_mean"], rtol=1e-12)
    # the same records as a three-column BED with bare chromosome numbers (the layout of the reference's 701_502.filter.bed)
    chrs = np.char.replace(g["chrs"], "Chr", "")
    with open(str(bed), "w") as fh:
        fh.writelines("%s\t%d\t%s\n" % r for r in zip(chrs, g["pos"], g["gt"]))
    b = parsers.ParseInputs(str(bed))
    assert len(b.chrs) == 7545 and b.chrs[0] == "1" and b.gt[0] == "0/0" and int(b.pos[1]) == 21006
    assert np.array_equal(b.chrs, chrs) and np.array_equal(b.pos, g["pos"]) and np.array_equal(b.gt, g["gt"])
    assert np.array_equal(b.wei, parsers.ParseInputs.get_wei_from_GT(g["gt"])) and b.wei.sum() == 7545
    assert os.path.isfile(str(bed) + ".snpmatch.npz") and os.path.isfile(str(bed) + ".snpmatch.stats.json")
    again = parsers.ParseInputs(str(bed))                                    # npz cache path
    assert np.array_equal(again.pos, b.pos) and np.array_equal(again.wei, b.wei)


def test_group_markers_host_preparation(built_lib):
    """snpm_group_markers (host code of the library): stable order by weight triple, one-byte chromosome ids, exact table."""
    lib = built_lib
    rng = np.random.default_rng(5)
    n0, n1 = 500, 300
    offs = np.array([0, n0, n0 + n1])
    chrom = np.concatenate([np.sort(rng.integers(-1, 5, size=n0)), np.sort(rng.integers(0, 5, size=n1))]).astype(np.int32)
    pos = np.arange(n0 + n1, dtype=np.int32) * 7 + 3
    menu = np.exp(-rng.integers(0, 40, size=(12, 3)) / 10.0)
    menu[:, 0] = 1.0
    wei = menu[rng.integers(0, 12, size=n0 + n1)]
    g = lib.group_markers(offs, chrom, pos, wei)
    assert g is not None and len(g.table) <= 12 and g.table.shape[1] == 3
    # table[gid] reproduces the weights bit for bit; markers of a sample stay inside it; order is (gid, input order)
    assert np.array_equal(g.table[g.gid], wei[g.order])
    assert np.array_equal(g.pos, pos[g.order])
    assert np.array_equal(g.chrom, np.where(chrom[g.order] < 0, 255, chrom[g.order]).astype(np.uint8))
    for s in range(2):
        lo, hi = offs[s], offs[s + 1]
        assert np.array_equal(np.sort(g.order[lo:hi]), np.arange(lo, hi))
        key = g.gid[lo:hi].astype(np.int64) * (n0 + n1) + g.order[lo:hi]
        assert np.all(np.diff(key) > 0)
    # chromosome id and position in one word; positions / ids that do not fit leave the unpacked form
    assert g.packed is not None and np.array_equal(g.packed >> 27, np.where(g.chrom == 255, 31, g.chrom))
    assert np.array_equal(g.packed & 0x7ffffff, g.pos)
    big = lib.group_markers(offs, chrom, pos + (1 << 27), wei)
    assert big is not None and big.packed is None and big.h2d_bytes > g.h2d_bytes
    assert lib.group_markers(offs, np.where(chrom >= 0, chrom + 40, chrom).astype(np.int32), pos, wei).packed is None
    # inputs the grouped kernel cannot take
    bad = wei.copy()
    bad[3, 1] = -0.5
    assert lib.group_markers(offs, chrom, pos, bad) is None
    bad[3, 1] = np.nan
    assert lib.group_markers(offs, chrom, pos, bad) is None
    assert lib.group_markers(offs, chrom, pos, rng.random((n0 + n1, 3)), table_cap=100) is None
    assert lib.group_markers(offs, np.full(n0 + n1, 300, np.int32), pos, wei) is None


def test_label_factorize_and_chromosome_names():
    """core/labels.py: per-marker strings reduced to codes + distinct values (run detection and the hash path) reproduce the
    per-element operations of the reference (parsers.py:161-163, genomes.py:75)."""
    from snpmatch_b200.core import genomes, labels, snp_genotype
    rng = np.random.default_rng(4)
    sorted_chrs = np.char.add("Chr", np.sort(rng.integers(1, 6, 5000)).astype(str))
    for arr in (sorted_chrs, sorted_chrs[rng.permutation(5000)], np.array(["chrC", "ChrM", "chrC", "1", "CHR1"]),
                np.array([b"2", b"2", b"10"]), np.array(["x"]), np.array([], dtype="U4")):
        codes, uniq = labels.factorize(arr)
        as_text = np.array([a.decode() if isinstance(a, bytes) else str(a) for a in arr], dtype="U8") if len(arr) else arr.astype("U")
        assert np.array_equal(uniq[codes] if len(arr) else uniq[:0], as_text)
        if len(arr):
            _, first = np.unique(as_text, return_index=True)
            assert uniq.tolist() == as_text[np.sort(first)].tolist()          # first-appearance order
        want = np.array([re.sub("chr", "", s, flags=re.IGNORECASE) for s in as_text], dtype="U8")
        assert np.array_equal(snp_genotype.normalize_chr_names(arr), want)
        assert np.array_equal(orc.normalize_chr_names(as_text), want)
        assert np.array_equal(genomes.genome_style_ids(arr), np.array([s.lower().replace("chr", "") for s in as_text], dtype="U8"))


def test_filter_chr_names_and_multi_sample_vcf(tmp_path):
    from snpmatch_b200.core import parsers
    inp = parsers.ParseInputs("")
    inp.load_snp_info(np.array(["Chr2", "Chr2", "chr1", "1", "ChrC"]), np.arange(5), np.repeat("0/0", 5), np.ones((5, 3)), "NA")
    inp.filter_chr_names()
    assert inp.g_chrs.tolist() == ["2", "2", "1", "1", "C"] and inp.g_chrs_ids.tolist() == ["2", "1", "C"]
    vcf = tmp_path / "pop.vcf"
    vcf.write_text("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tA\tB\tC\n"
                   "1\t100\t.\tA\tT\t9\tPASS\t.\tGT:DP\t0/0:3\t0|1:2\t./.:0\n"
                   "1\t250\t.\tG\tC\t9\tPASS\t.\tDP:GT\t4:1/1\t1:.\t2:1|0\n"
                   "Chr2\t7\t.\tG\tC\t9\tPASS\t.\tGT\t1/1\t0/0\n")
    v = parsers.import_vcf_file(str(vcf), samples_to_load=None)
    assert v["samples"].tolist() == ["A", "B", "C"] and v["chr"].tolist() == ["1", "1", "Chr2"] and v["pos"].tolist() == [100, 250, 7]
    assert v["gt"].tolist() == [["0/0", "0/1", "./."], ["1/1", "./.", "1/0"], ["1/1", "0/0", "./."]]    # phasing dropped, short rows padded
    assert parsers.parseGT(v["gt"].ravel()).reshape(3, 3).tolist() == [[0, 2, -1], [1, -1, 2], [1, 0, -1]]
    assert np.array_equal(parsers.parseGT(v["gt"].ravel()), orc.parse_gt(v["gt"].ravel()))


def test_grouped_samples_run_length_ids(built_lib):
    """GroupedSamples.pack (host code of the library + NumPy): packed chromosome/position words and the run-length form of the ids."""
    lib = built_lib
    rng = np.random.default_rng(8)
    n = [3000, 0, 1, 500]
    offs = np.concatenate([[0], np.cumsum(n)]).astype(np.int64)
    chrom = rng.integers(-1, 5, size=offs[-1]).astype(np.int32)
    pos = rng.integers(1, 30_000_000, size=offs[-1]).astype(np.int32)
    levels = np.exp(-np.arange(0, 40, 3) / 10.0)
    many = lib.group_markers(offs, chrom, pos, levels[rng.integers(0, len(levels), size=(offs[-1], 3))])
    assert many.packed is not None and many.run_gid is None               # ~2000 triples for 3500 markers: runs would be longer than the ids
    wei = levels[rng.integers(0, 4, size=(offs[-1], 3))]
    g = lib.group_markers(offs, chrom, pos, wei)
    assert g.packed is not None and g.run_gid is not None
    gid = np.repeat(g.run_gid, np.diff(np.concatenate([[0], g.run_end.astype(np.int64)])))
    assert np.array_equal(gid, g.gid) and int(g.run_end[-1]) == offs[-1] and np.all(np.diff(g.run_end.astype(np.int64)) > 0)
    assert np.array_equal(g.packed >> 27, np.where(g.chrom == 255, 31, g.chrom)) and np.array_equal(g.packed & 0x7FFFFFF, g.pos)
    assert np.array_equal(g.table[g.gid], wei[g.order])                     # the table reproduces every marker's weights bit for bit
    for s in range(len(n)):                                                 # inside a sample the ids ascend (that is what makes runs long)
        assert np.all(np.diff(g.gid[offs[s]:offs[s + 1]].astype(int)) >= 0)
    assert g.h2d_bytes < offs.nbytes + 6 * offs[-1] + len(g.table) * 32


def test_makedb_host_side(tmp_path):
    """`makedb` without bcftools / HDF5 (SURVEY 8(f)-2): the VCF -> CSV step (getCSV, makedb.py:34-62) and the CSV loader
    against the arrays the reference's pygwas loader builds (tests/golden/makedb_csv.npz)."""
    import json
    from snpmatch_b200.core import makedb
    g = load_golden("makedb_csv.npz")
    path = str(tmp_path / "db.csv")
    with open(path, "w") as fh:
        fh.write(str(g["csv"]))
    d = makedb.load_csv(path)
    assert np.array_equal(d["snps"], g["snps"]) and np.array_equal(d["positions"], g["positions"])
    assert d["chrs"].tolist() == g["chrs"].tolist() and np.array_equal(d["chr_regions"], g["chr_regions"])
    assert d["accessions"].astype("U").tolist() == g["accessions"].tolist()
    with open(str(tmp_path / "tabs.csv"), "w") as fh:
        fh.write(str(g["csv"]).replace(",", "\t").replace("Position", "Positions"))
    t = makedb.load_csv(str(tmp_path / "tabs.csv"))
    assert np.array_equal(t["snps"], g["snps"]) and np.array_equal(t["chr_regions"], g["chr_regions"])
    with open(str(tmp_path / "bad.csv"), "w") as fh:
        fh.write("chrom,pos,a\n1,2,0\n")
    with pytest.raises(Exception, match="First two columns"):
        makedb.load_csv(str(tmp_path / "bad.csv"))
    vcf = tmp_path / "strains.vcf"
    vcf.write_text("##fileformat=VCFv4.2\n##contig=<ID=Chr1,length=30427671>\n##contig=<ID=Chr2,length=19698289,assembly=x>\n"
                   "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t6909\t8236\t9999\n"
                   "Chr1\t10\t.\tA\tT\t.\t.\t.\tGT\t0/0\t1/1\t0/1\nChr1\t25\t.\tA\tT\t.\t.\t.\tGT:DP\t1|0:3\t./.:0\t1/2:4\n"
                   "Chr2\t7\t.\tA\tT\t.\t.\t.\tGT\t1/1\t0|0\t.\n")
    makedb.vcf_to_csv(str(vcf), str(tmp_path / "db2"))
    assert open(str(tmp_path / "db2.csv")).read() == "Chromosome,Position,6909,8236,9999\nChr1,10,0,1,2\nChr1,25,2,-1,-1\nChr2,7,1,0,-1\n"
    assert json.load(open(str(tmp_path / "db2.json"))) == {"ref_chrs": ["Chr1", "Chr2"], "ref_chrlen": [30427671, 19698289]}
    assert makedb.get_contigs(["##contig=<ID=1,length=5>", "##INFO=<ID=DP>"]) == {"ref_chrs": ["1"], "ref_chrlen": [5]}


def test_coded_samples_host_side():
    """lib.code_markers / CodedSamples.pack / ParseInputs.coded_weights: what crosses the bus reproduces the inputs bit for bit."""
    from snpmatch_b200 import lib, synth
    from snpmatch_b200.core import parsers
    pos, regions = synth.panel_positions(20000)
    s = synth.make_sample_fast(pos, regions, 50, 3, n_db=2000, n_extra=200, seed=5)
    n = len(s["pos"])
    cs = lib.code_markers(np.array([0, n]), s["chr_ix"], s["pos"], s["wei"])
    assert cs is not None and cs.codes.shape == (n, 3) and cs.codes.dtype == np.uint16
    assert np.array_equal(cs.wtable[cs.codes.astype(np.int64)].view(np.uint64), s["wei"].view(np.uint64))
    assert np.array_equal(cs.chrom_pos >> np.uint32(27), s["chr_ix"].astype(np.uint32))
    assert np.array_equal(cs.chrom_pos & np.uint32((1 << 27) - 1), s["pos"].astype(np.uint32))
    assert cs.codes32 is not None and cs.h2d_bytes < 8 * n + 8 * len(cs.wtable) + 64
    c32 = cs.codes32
    assert np.array_equal(c32 & 1023, cs.codes[:, 0]) and np.array_equal((c32 >> 10) & 1023, cs.codes[:, 1]) and np.array_equal(c32 >> 20, cs.codes[:, 2])
    # integer PLs as ready-made codes
    table = synth.pl_table(int(s["pl"].max()))
    assert np.array_equal(table[s["pl"]].view(np.uint64), s["wei"].view(np.uint64))
    cs2 = lib.code_markers(np.array([0, n]), s["chr_ix"], s["pos"], codes=s["pl"].astype(np.uint16), wtable=table)
    assert np.array_equal(cs2.wtable[cs2.codes.astype(np.int64)], s["wei"])
    # markers outside the panel's chromosomes, ids / positions that do not fit one word, weights that cannot be coded
    assert int(lib.pack_chrom_pos(np.array([-1, 2]), np.array([5, 6]))[0] >> 27) == 31
    assert lib.pack_chrom_pos(np.array([31]), np.array([5])) is None and lib.pack_chrom_pos(np.array([0]), np.array([1 << 27])) is None
    assert lib.code_markers(np.array([0, 1]), np.array([0]), np.array([1]), np.array([[-0.5, 0.0, 1.0]])) is None
    big = lib.CodedSamples(np.array([0, 1]), np.zeros(1, np.uint32), np.zeros((1, 3), np.uint16), np.arange(2000.0)).pack()
    assert big.codes32 is None                                   # more than 1024 weight values: three uint16 per marker
    inp = parsers.ParseInputs("")
    inp.load_snp_info(np.array(["Chr1"] * n), s["pos"], synth._gt_strings(s["code"]), s["wei"], s["dp"])
    codes, tab = inp.coded_weights()
    assert np.array_equal(tab[codes.astype(np.int64)].view(np.uint64), s["wei"].view(np.uint64))
    assert inp.coded_weights()[0] is codes                       # cached


def test_coded_batch_host_side(built_lib):
    """core.batch.coded_batch: what goes up for a list of ParseInputs reproduces every sample's markers and weights bit for bit
    whichever shortcut was taken (files already in the join's order, tables that are prefixes of one table) or not."""
    from snpmatch_b200 import lib, synth
    from snpmatch_b200.core import batch, parsers, snp_genotype
    pos, regions = synth.panel_positions(20000)
    g = object.__new__(snp_genotype.Genotype)
    g.chrs = np.array(synth.TAIR10_CHRS)
    g._db_chr_norm = snp_genotype.normalize_chr_names(g.chrs)
    names = np.array(["Chr" + c for c in synth.TAIR10_CHRS])

    def make(seed, shuffle_chromosomes, own_table):
        s = synth.make_sample_fast(pos, regions, 50, 3, n_db=1500, n_extra=150, seed=seed)
        chrs, p, wei, pl = names[s["chr_ix"]], s["pos"], s["wei"], s["pl"]
        if shuffle_chromosomes:                                  # chromosome blocks in another order than the database's
            blocks = [np.flatnonzero(s["chr_ix"] == c) for c in (3, 0, 4, 1, 2)]
            k = np.concatenate(blocks)
            chrs, p, wei, pl = chrs[k], p[k], wei[k], pl[k]
        inp = parsers.ParseInputs("")
        inp.load_snp_info(chrs, p, synth._gt_strings(s["code"]), wei, s["dp"])
        if not own_table:
            inp._coded = (pl.astype(np.uint16), synth.pl_table(int(pl.max())), inp.wei)
        return inp

    for case in ([(11, False, False), (12, False, False)],       # in order, prefix tables: no permutation, no remap
                 [(13, True, False), (14, False, False)],        # one sample permuted
                 [(15, False, True), (16, True, False)]):        # one sample with its own dictionary (np.unique order): union + remap
        inputs = [make(*c) for c in case]
        cs, offs, cid, p, wei = batch.coded_batch(g, inputs)
        assert cs is not None and cs.codes32 is not None
        cs_lazy = batch.coded_batch(g, inputs, with_weights=False)
        assert cs_lazy[4] is None and np.array_equal(cs_lazy[0].codes32, cs.codes32) and np.array_equal(cs_lazy[0].chrom_pos, cs.chrom_pos)
        for i, inp in enumerate(inputs):
            order, c_i, p_i = g.prepare_markers(inp.chrs, inp.pos)
            lo, hi = int(offs[i]), int(offs[i + 1])
            assert np.array_equal(cid[lo:hi], c_i) and np.array_equal(p[lo:hi], p_i)
            want = np.asarray(inp.wei)[order]
            assert np.array_equal(wei[lo:hi].view(np.uint64), want.view(np.uint64))
            assert np.array_equal(cs.wtable[cs.codes[lo:hi].astype(np.int64)].view(np.uint64), want.view(np.uint64))
            assert np.array_equal(cs.chrom_pos[lo:hi] >> np.uint32(27), np.where(c_i < 0, 31, c_i).astype(np.uint32))
            assert np.array_equal(cs.chrom_pos[lo:hi] & np.uint32((1 << 27) - 1), p_i.astype(np.uint32))
        c32 = cs.codes32
        assert np.array_equal(c32 & 1023, cs.codes[:, 0]) and np.array_equal((c32 >> 10) & 1023, cs.codes[:, 1]) and np.array_equal(c32 >> 20, cs.codes[:, 2])
    # the native packer refuses what does not fit the words
    assert lib.code_markers(np.array([0, 1]), np.array([31]), np.array([5]), codes=np.zeros((1, 3), np.uint16), wtable=np.ones(4)) is None
    assert lib.code_markers(np.array([0, 1]), np.array([0]), np.array([1 << 27]), codes=np.zeros((1, 3), np.uint16), wtable=np.ones(4)) is None
    assert lib.code_markers(np.array([0, 1]), np.array([0]), np.array([7]), codes=np.full((1, 3), 9, np.uint16), wtable=np.ones(4)) is None
    one = lib.code_markers(np.array([0, 2]), np.array([-1, 2]), np.array([5, 6]), codes=np.array([[0, 1, 2], [3, 2, 1]], np.uint16), wtable=np.arange(4.0))
    assert int(one.chrom_pos[0] >> 27) == 31 and int(one.chrom_pos[1]) == (2 << 27 | 6) and one.codes32.tolist() == [0 | 1 << 10 | 2 << 20, 3 | 2 << 10 | 1 << 20]


def test_bench_numa_binding_is_optional():
    """bench.py binds a rank to the cores next to its GPU when the topology can be read, and says why not otherwise
    (no NVML in the build container): never an exception, never an empty affinity mask."""
    import os
    import bench
    before = os.sched_getaffinity(0)
    info = bench.bind_to_gpu_numa_node(0)
    assert isinstance(info, dict) and "bound" in info
    assert info["bound"] or "why" in info
    assert len(os.sched_getaffinity(0)) >= 1
    os.sched_setaffinity(0, before)
