"""BGZF without a device: synth.write_bgzf, the member scanner's verdicts (lib.bgzf_scan), and the DEFLATE decoder of
csrc/inflate.cuh compiled for the host and checked against zlib on a corpus and on seeded corruptions."""
import gzip
import io
import os
import shutil
import struct
import subprocess
import warnings
import zlib

import numpy as np
import pytest

from snpmatch_b200 import lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "snpmatch_b200", "csrc")
CAP = 65536


@pytest.fixture(scope="module")
def built():
    """The library holds the scanner (host code): build it, as a clean checkout has no libsnpmatch_b200.so."""
    import __graft_entry__ as ge
    ge.build()
    return lib


def test_write_bgzf_reads_back(built, tmp_path):
    text = (b"chr1\t%d\t.\tA\tT\n" * 20000) % tuple(range(20000))
    data = np.random.default_rng(3).integers(0, 256, 70000, dtype=np.uint8).tobytes() + text
    data2 = b"".join([data[:1], text[:65280], text[:65536]])
    p = tmp_path / "a.vcf.gz"
    synth.write_bgzf(p, data2, member_bytes=[0, 1, 65280, 65536])
    raw = p.read_bytes()
    assert gzip.decompress(raw) == data2
    assert raw.endswith(synth.BGZF_EOF)
    off, isize = lib.bgzf_scan(np.frombuffer(raw, np.uint8))
    assert isize.tolist() == [0, 1, 65280, 65536, 0] and off[-1] == len(raw)
    synth.write_bgzf(p, data, eof=False)                  # random bytes: stored blocks
    assert gzip.decompress(p.read_bytes()) == data
    with pytest.raises(ValueError):
        synth.write_bgzf(p, data[:65536], member_bytes=65536)    # 64 KiB of random bytes do not fit one member


def _member(text, extra=b"BC\x02\x00", bsize_delta=0, flg=4, isize=None):
    """One gzip member of text; extra = its extra field with the BC subfield's 2 value bytes left out (filled in here)."""
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    payload = c.compress(text) + c.flush()
    size = 12 + len(extra) + 2 + len(payload) + 8
    ex = extra.replace(b"BC\x02\x00", b"BC\x02\x00" + struct.pack("<H", size - 1 + bsize_delta))
    return (b"\x1f\x8b\x08" + bytes([flg]) + b"\0\0\0\0\0\xff" + struct.pack("<H", len(ex)) + ex + payload
            + struct.pack("<II", zlib.crc32(text), len(text) if isize is None else isize))


def _verdict(raw):
    r = lib.bgzf_scan(np.frombuffer(raw, np.uint8))
    return None if r is None else len(r[1])


def test_scanner_verdicts(built):
    a, b = b"chr1\t1\n" * 500, b"chr2\t2\n" * 300
    bgzf = _member(a) + _member(b)
    assert _verdict(bgzf) == 2
    assert _verdict(bgzf + synth.BGZF_EOF) == 3
    assert gzip.decompress(bgzf + synth.BGZF_EOF) == a + b
    # extra subfields besides BC, before and after it
    other = _member(a, extra=b"XY\x03\x00abc" + b"BC\x02\x00") + _member(b, extra=b"BC\x02\x00" + b"ZZ\x00\x00")
    assert gzip.decompress(other) == a + b and _verdict(other) == 2
    assert _verdict(gzip.compress(a)) is None             # single-member gzip: FLG 0, no BC
    assert _verdict(bgzf + gzip.compress(b)) is None      # BGZF followed by a plain gzip member
    with io.BytesIO() as buf:
        with gzip.GzipFile("x.vcf", "wb", fileobj=buf) as g:
            g.write(a)
        fname = buf.getvalue()                            # FNAME set, as `gzip file` writes
    assert fname[3] & 8 and _verdict(fname) is None
    assert _verdict(bgzf[:-5]) is None                    # truncated last member
    assert _verdict(bgzf + b"\0" * 16) is None            # trailing zero padding
    big = _member(b"x" * 70000)                           # ISIZE > 65536
    assert _verdict(big) is None
    assert _verdict(_member(a, isize=65537)) is None
    assert _verdict(_member(a, flg=5)) is None            # FTEXT besides FEXTRA
    assert _verdict(_member(a, bsize_delta=1)) is None    # BSIZE past the file's end
    assert _verdict(b"") is None


# ---- the decoder compiled for the host ------------------------------------------------------------------------------------
HARNESS = r'''
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "inflate.cuh"
// stdin: records [u32 n][n bytes], each a raw DEFLATE stream; stdout per record: [i32 status][u32 produced][the text]
int main() {
    uint32_t n;
    while (fread(&n, 4, 1, stdin) == 1) {
        uint8_t *in = (uint8_t *)malloc(n ? n : 1);       // exactly n bytes: the sanitizer sees any read past them
        if (n && fread(in, 1, n, stdin) != n) return 2;
        uint8_t *out = (uint8_t *)malloc(65536);
        BgzfTables *T = (BgzfTables *)malloc(sizeof(BgzfTables));
        memset(T, 0xA5, sizeof(BgzfTables));
        uint32_t produced = 0;
        int32_t st = bgzf_inflate_raw(in, n, out, 65536, &produced, *T, 0, 1);
        if (st != BGZF_OK) produced = 0;
        fwrite(&st, 4, 1, stdout);
        fwrite(&produced, 4, 1, stdout);
        fwrite(out, 1, produced, stdout);
        free(T);
        free(out);
        free(in);
    }
    return 0;
}
'''


# one flag per -Xcompiler: nvcc splits an -Xcompiler argument at its commas
SANITIZE = ["-Xcompiler", "-fsanitize=address", "-Xcompiler", "-fsanitize=undefined", "-Xcompiler", "-fno-sanitize-recover=all",
            "-lasan", "-lubsan"]


@pytest.fixture(scope="module")
def harness_build(tmp_path_factory):
    """(path of the harness, whether it carries AddressSanitizer and UBSan).  The sanitized build is the one expected; the plain
    build is taken only when the host toolchain cannot build even an empty program with the sanitizers, and then with a warning
    (test_harness_is_sanitized reports the skip)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not (os.path.isfile(nvcc) or shutil.which(nvcc)):
        pytest.skip("no nvcc")
    d = tmp_path_factory.mktemp("inflate_host")
    src = d / "harness.cu"
    src.write_text(HARNESS)
    exe = str(d / "harness")
    base = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O1", "-g", "-I", CSRC, "-o", exe, str(src)]
    r = subprocess.run(base + SANITIZE, capture_output=True, text=True)
    if r.returncode == 0:
        return exe, True
    probe = d / "probe.cu"
    probe.write_text("int main() { return 0; }\n")
    if subprocess.run([nvcc, "-o", str(d / "probe"), str(probe)] + SANITIZE, capture_output=True).returncode == 0:
        raise AssertionError("the sanitizers work on this host but the harness does not build with them:\n" + r.stderr[-3000:])
    warnings.warn("the host toolchain has no AddressSanitizer / UBSan runtime: the decoder harness is built without them")
    subprocess.run(base, check=True, capture_output=True)
    return exe, False


@pytest.fixture(scope="module")
def harness(harness_build):
    return harness_build[0]


def test_harness_is_sanitized(harness_build):
    exe, sanitized = harness_build
    if not sanitized:
        pytest.skip("decoder harness built WITHOUT AddressSanitizer / UBSan: the host toolchain has no sanitizer runtime")
    with open(exe, "rb") as fh:
        image = fh.read()
    assert b"__asan_init" in image and b"__ubsan_handle" in image


def _run(exe, payloads):
    recs = b"".join(struct.pack("<I", len(p)) + p for p in payloads)
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0:abort_on_error=0", UBSAN_OPTIONS="halt_on_error=1")
    r = subprocess.run([exe], input=recs, capture_output=True, env=env)
    assert r.returncode == 0, r.stderr.decode(errors="replace")[-3000:]
    out, at, res = r.stdout, 0, []
    for _ in payloads:
        st, n = struct.unpack_from("<iI", out, at)
        at += 8
        res.append((st, out[at:at + n]))
        at += n
    assert at == len(out)
    return res


def _zlib(p):
    """zlib's output when it accepts p as one whole raw DEFLATE stream of at most 64 KiB of text, else None."""
    d = zlib.decompressobj(-15)
    try:
        out = d.decompress(p, CAP + 1)
    except zlib.error:
        return None
    return out if d.eof and not d.unused_data and len(out) <= CAP else None


def _check(exe, payloads):
    for p, (st, got) in zip(payloads, _run(exe, payloads)):
        ref = _zlib(p)
        if st == 0:
            assert ref is not None and got == ref, "decoder accepts a stream zlib refuses or decodes it differently"
        else:
            assert st in (1, 2) and ref is None, "decoder refuses (status %d) a stream zlib accepts" % st


def _deflate(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    return c.compress(data) + c.flush()


def _corpus():
    rng = np.random.default_rng(17)
    vcf, _ = synth.multi_sample_vcf(400, 12, seed=5)
    buf = io.BytesIO()
    synth.panel_vcf(buf, 300, 40)
    texts = [vcf.encode()[:65280], buf.getvalue()[:65536], rng.integers(0, 256, 65280, dtype=np.uint8).tobytes(), b"",
             b"A", b"A" * 65536, bytes(range(256)) * 40, vcf.encode()[1000:1500]]
    out = []
    for t in texts:
        for level in range(10):
            out.append(_deflate(t, level))
        for strategy in (zlib.Z_FIXED, zlib.Z_RLE, zlib.Z_HUFFMAN_ONLY, zlib.Z_FILTERED):
            out.append(_deflate(t, 6, strategy))
    # several DEFLATE blocks of different types in one stream
    # several DEFLATE blocks of different types in one stream: sync-flushed (non-final, byte-aligned) parts, then a final one
    multi = b""
    for t, level, strategy in ((texts[0][:15000], 6, zlib.Z_DEFAULT_STRATEGY), (texts[2][:15000], 0, zlib.Z_DEFAULT_STRATEGY),
                               (texts[1][:9000], 9, zlib.Z_FIXED)):
        c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
        multi += c.compress(t) + c.flush(zlib.Z_SYNC_FLUSH)
    multi += _deflate(texts[0][20000:35000])
    out.append(multi)
    return out


def test_decoder_matches_zlib_on_corpus(harness):
    corpus = _corpus()
    res = _run(harness, corpus)
    for p, (st, got) in zip(corpus, res):
        assert st == 0 and got == _zlib(p)


class _Bits(object):
    def __init__(self):
        self.v, self.n = 0, 0

    def put(self, value, k):
        self.v |= (value & ((1 << k) - 1)) << self.n
        self.n += k

    def code(self, code, k):                              # Huffman codes go most significant bit first
        self.put(int(format(code, "0%db" % k)[::-1], 2) if k else 0, k)

    def bytes(self):
        return self.v.to_bytes((self.n + 7) // 8, "little")


def _canonical(lens):
    count = [0] * 16
    for L in lens:
        count[L] += 1
    count[0] = 0
    code, nxt = 0, [0] * 16
    for L in range(1, 16):
        code = (code + count[L - 1]) << 1
        nxt[L] = code
    codes = {}
    for s, L in enumerate(lens):
        if L:
            codes[s] = (nxt[L], L)
            nxt[L] += 1
    return codes


def _dynamic(lit, dist, symbols, hlit=None, hdist=None, cl=None, raw_cl_syms=None):
    """One final dynamic block: the literal/length and distance lengths sent with a code-length code of 4 bits for the lengths
    0..15 (or the given cl lengths), then symbols: ints (literal/length symbols, 257.. sent with zero extra bits) or ('d', s)
    distance symbols.  raw_cl_syms replaces the code-length symbols sent."""
    b = _Bits()
    b.put(1, 1)
    b.put(2, 2)
    hlit = len(lit) if hlit is None else hlit
    hdist = len(dist) if hdist is None else hdist
    b.put(hlit - 257, 5)
    b.put(hdist - 1, 5)
    order = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
    cl = cl if cl is not None else [4] * 16 + [0, 0, 0]
    b.put(19 - 4, 4)
    for s in order:
        b.put(cl[s], 3)
    clc = _canonical(cl)
    for s in (raw_cl_syms if raw_cl_syms is not None else list(lit) + list(dist)):
        if s in clc:
            b.code(*clc[s])
    lc, dc = _canonical(lit), _canonical(dist)
    for s in symbols:
        if isinstance(s, tuple):
            if s[1] in dc:
                b.code(*dc[s[1]])
            else:
                b.put(0, 5)
        elif s in lc:
            b.code(*lc[s])
            if 265 <= s < 285:
                b.put(0, (s - 261) // 4)
        else:
            b.put(0, 9)
    return b.bytes()


def _hand_built():
    lit_full = [9] * 256 + [5, 5] + [6] * 28             # complete over the 286 literal/length symbols
    dist_full = [4, 4] + [5] * 28                       # complete over the 30 distance symbols
    word = [ord(c) for c in "ACGT" * 5]
    cases = [
        _dynamic(lit_full, dist_full, word + [256]),                         # complete codes: accepted
        _dynamic(lit_full, dist_full, word + [257, ("d", 0), 256]),           # a match
        _dynamic(lit_full, dist_full, [257, ("d", 0), 256]),                  # a distance before the first byte
        _dynamic(lit_full, [0], word + [256]),                               # all-zero distance set, unused: accepted
        _dynamic(lit_full, [0], word + [257, ("d", 0), 256]),                # ... used
        _dynamic(lit_full, [1], word + [257, ("d", 0), 256]),                # single distance code of length 1
        _dynamic([0] * 256 + [1], [1], [256]),                               # single literal/length code (EOB) of length 1
        _dynamic([0] * 256 + [1, 1], [1], [256]),                            # two codes of length 1: complete
        _dynamic([0] * 256 + [2], [1], [256]),                               # single code of length 2: incomplete
        _dynamic([8] * 257 + [0] * 29, dist_full, [256]),                     # over-subscribed literal/length set
        _dynamic([8] * 128 + [0] * 128 + [8] + [0] * 29, dist_full, [256]),   # incomplete literal/length set
        _dynamic(lit_full, [4] * 17 + [0] * 13, [256]),                      # over-subscribed distance set
        _dynamic(lit_full, [5] * 20 + [0] * 10, [256]),                      # incomplete distance set
        _dynamic([8] * 256 + [0] + [8] * 29, dist_full, [0, 256]),            # no end-of-block code
        _dynamic(lit_full, dist_full, [256], cl=[4] * 16 + [4, 0, 0]),        # over-subscribed code-length code
        _dynamic(lit_full, dist_full, [256], cl=[5] * 16 + [0, 0, 0]),        # incomplete code-length code
        _dynamic(lit_full, dist_full, [256], cl=[0] * 19),                    # empty code-length code
        _dynamic(lit_full + [8, 8], dist_full, [256]),                        # HLIT 288
        _dynamic(lit_full, [5] * 32, [256]),                                 # HDIST 32
        _dynamic(lit_full, dist_full, [256], cl=[4] * 15 + [0, 4, 0, 0], raw_cl_syms=[16] + lit_full[1:] + dist_full),  # repeat first
    ]
    # stored blocks: LEN / NLEN agree, disagree; block type 3; fixed codes using symbols 286 / 287 and distances 30 / 31
    cases.append(b"\x01\x05\x00\xfa\xffhello")
    cases.append(b"\x01\x05\x00\xfa\xfehello")
    cases.append(b"\x07\x00")
    b = _Bits()
    b.put(1, 1)
    b.put(1, 2)
    b.code(0b11000110, 8)                                                # symbol 286
    cases.append(b.bytes() + b"\0")
    b = _Bits()
    b.put(1, 1)
    b.put(1, 2)
    b.code(0x30 + ord("A"), 8)
    b.code(0b0000001, 7)                                                 # symbol 257: length 3
    b.code(30, 5)                                                        # distance symbol 30
    cases.append(b.bytes() + b"\0")
    return cases


def test_decoder_hand_built_code_sets(harness):
    cases = _hand_built()
    res = _run(harness, cases)
    verdicts = [st == 0 for st, _ in res]
    accepted = {0, 1, 3, 5, 6, 7, 20}
    assert verdicts == [i in accepted for i in range(len(cases))]
    _check(harness, cases)


def test_decoder_fuzz(harness):
    rng = np.random.default_rng(2024)
    base = _corpus() + _hand_built()
    payloads = []
    for i in range(4000):
        p = bytearray(base[int(rng.integers(0, len(base)))])
        kind = i % 5
        if kind in (0, 1) and p:                           # bit flips
            for _ in range(int(rng.integers(1, 4))):
                k = int(rng.integers(0, len(p)))
                p[k] ^= 1 << int(rng.integers(0, 8))
        elif kind == 2 and p:                              # truncation
            p = p[:int(rng.integers(0, len(p)))]
        elif kind == 3:                                    # random payload
            p = bytearray(rng.integers(0, 256, int(rng.integers(0, 300)), dtype=np.uint8).tobytes())
        elif p:                                            # flips in the block header, where the code sets are
            k = int(rng.integers(0, min(len(p), 40)))
            p[k] ^= 1 << int(rng.integers(0, 8))
        payloads.append(bytes(p))
    _check(harness, payloads)
