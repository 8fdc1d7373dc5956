"""BGZF `.vcf.gz` inflated on the device (csrc/inflate.cuh k_bgzf_inflate, lib.BgzfInflater, parsers.BgzfReader): thousands of
members of every DEFLATE block type in one call equal gzip.decompress; read_vcf_many, read_vcf_gt_codes and makeDB_from_vcf on
a BGZF file equal their results on the plain file whatever the chunking and wherever the member boundaries fall; the commands
write the same files; a corrupt member raises gzip.BadGzipFile naming its offset, and nothing is written."""
import gzip
import os
import zlib

import numpy as np
import pytest

from snpmatch_b200 import synth
from test_gpu_genotype_cross_vcf import _population, edge_vcf, golden, small_geno  # noqa: F401  (fixtures)
from test_gpu_vcf_samples import _same_inputs, e2e  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


def _raw(tmp_path, data, name="x.gz", **kw):
    p = str(tmp_path / name)
    synth.write_bgzf(p, data, **kw)
    return p


def test_inflater_mixed_members_in_one_call(lib, tmp_path):
    rng = np.random.default_rng(9)
    vcf = synth.multi_sample_vcf(3000, 20, seed=2)[0].encode()
    noise = rng.integers(0, 256, 1 << 20, dtype=np.uint8).tobytes()
    strategies = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_RLE, zlib.Z_HUFFMAN_ONLY, zlib.Z_FILTERED]
    parts, texts = [], []
    for i in range(2500):
        src = noise if i % 7 == 3 else vcf
        n = [0, 1, 65280, 65536, 300][i % 5] if i % 11 == 0 else int(rng.integers(0, 65281))
        a = int(rng.integers(0, len(src) - n + 1))
        t = src[a:a + n] if i % 13 else b"A" * n
        if src is noise and len(t) > 65000:
            t = t[:65000]
        p = _raw(tmp_path, t, "m.gz", level=i % 10, strategy=strategies[i % 5], member_bytes=[len(t)], eof=False)
        parts.append(open(p, "rb").read())
        texts.append(t)
    raw = b"".join(parts) + synth.BGZF_EOF
    want = b"".join(texts)
    assert gzip.decompress(raw) == want
    data = np.frombuffer(raw, np.uint8)
    off, isize = lib.bgzf_scan(data)
    assert len(isize) == 2501 and int(isize.sum()) == len(want)
    inf = lib.BgzfInflater(0, len(raw), len(want))
    out = np.empty(len(want), np.uint8)
    assert inf.inflate(data, off, out=out) == len(want)
    assert out.tobytes() == want and inf.text(0, len(want)) == want
    inf.close()
    path = str(tmp_path / "all.gz")
    open(path, "wb").write(raw)
    from snpmatch_b200.core import parsers
    r = parsers.BgzfReader.open(path, 0, batch_bytes=1 << 22)       # several batches
    got = b"".join(iter(lambda: r.read(1 << 20), b""))
    r.close()
    assert got == want


def _boundaries(text, member_bytes):
    """Member sizes of member_bytes that also cut once between a '\\r' and its '\\n' and once inside a line."""
    b = text.encode("utf-8") if isinstance(text, str) else text
    cuts = {i for i in range(member_bytes, len(b), member_bytes)}
    crlf = b.find(b"\r\n", len(b) // 3)
    if crlf > 0:
        cuts.add(crlf + 1)
    cuts.add(len(b) // 2 + 3)
    edges = [0] + sorted(c for c in cuts if 0 < c < len(b)) + [len(b)]
    return [y - x for x, y in zip(edges, edges[1:])]


def _write(path, text):
    with open(path, "w", encoding="utf-8", newline="") as fh:
        fh.write(text)


def _files(tmp_path, text, member_bytes, tag):
    plain = str(tmp_path / ("%s.vcf" % tag))
    _write(plain, text)
    gz = str(tmp_path / ("%s.vcf.gz" % tag))
    synth.write_bgzf(gz, text.encode("utf-8"), member_bytes=_boundaries(text, member_bytes))
    return plain, gz


def _longest(text):
    return max(len(x) for x in text.encode("utf-8").replace(b"\r\n", b"\n").replace(b"\r", b"\n").split(b"\n")) + 5


@pytest.mark.parametrize("member_bytes", [65280, 4099, 777])
@pytest.mark.parametrize("line_end", ["\n", "\r\n", ["\r\n", "\r", "\n"]])
def test_read_vcf_many_bgzf_equals_plain(lib, tmp_path, member_bytes, line_end):
    from snpmatch_b200.core import parsers
    text, _ = synth.multi_sample_vcf(600, 40, seed=3, line_end=line_end)
    plain, gz = _files(tmp_path, text, member_bytes, "many")
    ref = parsers.read_vcf_many(plain)
    for chunk in (_longest(text), 20000, parsers.VCF_CHUNK_BYTES):
        tm = {}
        got = parsers.read_vcf_many(gz, chunk_bytes=chunk, timings=tm)
        assert tm["inflate"] == "device" and tm["gz_bytes"] == os.path.getsize(gz)
        assert [n for n, _ in got] == [n for n, _ in ref]
        for (n, a), (_, b) in zip(got, ref):
            _same_inputs(a, b, (chunk, n))


def _same_codes(a, b):
    for k in ("samples", "chr", "pos", "gt_codes"):
        assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("member_bytes", [65280, 1500, 333])
def test_read_vcf_gt_codes_bgzf_equals_plain(lib, tmp_path, member_bytes):
    from snpmatch_b200.core import parsers
    for k, line_end in enumerate(["\n", "\r\n", ["\r\n", "\r", "\n"]]):
        text = edge_vcf(40, line_end=line_end, final_newline=k != 1)
        plain, gz = _files(tmp_path, text, member_bytes, "codes%d" % k)
        ref = parsers.read_vcf_gt_codes(plain)
        for chunk in (_longest(text), None):
            tm = {}
            got = parsers.read_vcf_gt_codes(gz, timings=tm, **({} if chunk is None else {"chunk_bytes": chunk}))
            assert tm["inflate"] == "device"
            _same_codes(got, ref)
    # the same text as a single-member gzip keeps the host route
    single = str(tmp_path / "single.vcf.gz")
    with gzip.open(single, "wb") as fh:
        fh.write(text.encode("utf-8"))
    tm = {}
    _same_codes(parsers.read_vcf_gt_codes(single, timings=tm), ref)
    assert tm["inflate"] == "host"
    tm = {}
    parsers.read_vcf_gt_codes(plain, timings=tm)
    assert tm["inflate"] is None


def _same_db(a, b):
    x, y = np.load(a + ".npz"), np.load(b + ".npz")
    assert sorted(x.files) == sorted(y.files)
    for k in x.files:
        assert x[k].dtype == y[k].dtype and np.array_equal(x[k], y[k]), k
    assert open(a + ".json", "rb").read() == open(b + ".json", "rb").read()


@pytest.mark.parametrize("member_bytes", [65280, 2000])
def test_makedb_bgzf_equals_plain(lib, tmp_path, member_bytes):
    import io
    from snpmatch_b200.core import makedb
    buf = io.BytesIO()
    synth.panel_vcf(buf, 3000, 70)
    text = buf.getvalue().decode().replace("\n", "\r\n")
    plain, gz = _files(tmp_path, text, member_bytes, "panel")
    makedb.makeDB_from_vcf(plain, str(tmp_path / "a")).close()
    for chunk in (_longest(text), None):
        tm = {}
        makedb.makeDB_from_vcf(gz, str(tmp_path / "b"), timings=tm, **({} if chunk is None else {"chunk_bytes": chunk})).close()
        assert tm["inflate"] == "device" and tm["inflate_ms"] > 0
        _same_db(str(tmp_path / "a"), str(tmp_path / "b"))


def test_cli_makedb_and_genotype_cross(lib, small_geno, golden, tmp_path):
    import io
    import snpmatch_b200
    buf = io.BytesIO()
    synth.panel_vcf(buf, 2000, 50)
    plain, gz = _files(tmp_path, buf.getvalue().decode(), 5000, "cli_panel")
    for p, o in ((plain, "p"), (gz, "g")):
        assert snpmatch_b200.main(["makedb", "-i", p, "-o", str(tmp_path / o), "--no_csv"]) == 0
    _same_db(str(tmp_path / "p"), str(tmp_path / "g"))
    c = golden["b1M_lr3"]
    db_path = str(tmp_path / "panel.npz")
    small_geno.save_packed(db_path)
    pop = str(tmp_path / "population.vcf")
    _population(pop)
    pop_gz = pop + ".gz"
    synth.write_bgzf(pop_gz, open(pop, "rb").read(), member_bytes=3000)
    outs = []
    for p in (pop, pop_gz):
        out = str(tmp_path / (os.path.basename(p) + ".csv"))
        assert snpmatch_b200.main(["genotype_cross", "-i", p, "-d", db_path, "-p", c["parents"], "-b", str(c["bin_len"]),
                                   "--lr_thres", str(c["lr_thres"]), "-o", out, "--gpu_parse"]) == 0
        outs.append(open(out, "rb").read())
    assert outs[0] == outs[1] and outs[0].decode().split("\n")[:-1] == c["lines"]


def _same_tree(a, b, names, exts):
    for name in names:
        for ext in exts:
            x, y = a + "." + name + ext, b + "." + name + ext
            assert os.path.exists(x) == os.path.exists(y), y
            if os.path.exists(x):
                assert open(x, "rb").read() == open(y, "rb").read(), y


def test_cli_samples_vcf_bgzf(lib, e2e, tmp_path, capsys):
    import snpmatch_b200
    gz = str(tmp_path / "population.vcf.gz")
    synth.write_bgzf(gz, open(e2e["vcf"], "rb").read(), member_bytes=7000)
    for p, o in ((e2e["vcf"], "p"), (gz, "g")):
        assert snpmatch_b200.main(["inbred", "--samples_vcf", p, "-d", e2e["db"], "-o", str(tmp_path / ("inbred_" + o))]) == 0
    _same_tree(str(tmp_path / "inbred_p"), str(tmp_path / "inbred_g"), e2e["names"], (".scores.txt", ".matches.json"))
    for p, o in ((e2e["vcf"], "p"), (gz, "g")):
        with pytest.raises(SystemExit) as e:         # "empty" names no chromosome of the genome: status 1 after the others
            snpmatch_b200.main(["cross", "--samples_vcf", p, "-d", e2e["db"], "-o", str(tmp_path / ("cross_" + o)), "-b", "300000"])
        assert e.value.code == 1
    capsys.readouterr()
    _same_tree(str(tmp_path / "cross_p"), str(tmp_path / "cross_g"), e2e["names"],
               (".scores.txt", ".windowscore.txt", ".scores.txt.matches.json", ".matches.json"))


def _corrupt(raw, off, which, kind):
    b = bytearray(raw)
    a, e = int(off[which]), int(off[which + 1])
    if kind == "crc":
        b[e - 8] ^= 0x5A
    elif kind == "isize":
        b[e - 4] ^= 0x01
    else:                                            # a payload byte of the member's DEFLATE stream
        b[a + 18 + (e - a - 26) // 2] ^= 0xFF
    return bytes(b)


@pytest.mark.parametrize("kind", ["crc", "isize", "payload"])
def test_corrupt_member_raises_and_writes_nothing(lib, tmp_path, kind):
    import io
    import snpmatch_b200
    from snpmatch_b200.core import parsers
    buf = io.BytesIO()
    synth.panel_vcf(buf, 3000, 40)
    good = _raw(tmp_path, buf.getvalue(), "good.vcf.gz", member_bytes=9000)
    raw = open(good, "rb").read()
    off, _ = lib.bgzf_scan(np.frombuffer(raw, np.uint8))
    which = len(off) // 2
    bad = str(tmp_path / "bad.vcf.gz")
    open(bad, "wb").write(_corrupt(raw, off, which, kind))
    reason = {"crc": "CRC-32", "isize": "ISIZE|DEFLATE", "payload": "DEFLATE|ISIZE|CRC"}[kind]
    for fn in (parsers.read_vcf_gt_codes, parsers.read_vcf_many):
        with pytest.raises(gzip.BadGzipFile, match=r"bad\.vcf\.gz: BGZF member at byte %d: .*(%s)" % (off[which], reason)):
            fn(bad)
    with pytest.raises(Exception):                   # the host route refuses the same file
        gzip.decompress(open(bad, "rb").read())
    out = str(tmp_path / "db")
    assert snpmatch_b200.main(["makedb", "-i", bad, "-o", out, "--no_csv"]) == 2
    assert not os.path.exists(out + ".npz") and not os.path.exists(out + ".json")
