"""
Sample parsing and PL -> weight preparation (host side; stays Python per the north star).

Mirrors the interface of the reference's `snpmatch/core/parsers.py` — `ParseInputs`
(parsers.py:59-175), `parseGT` (:12-35), `snp_binary_to_gt` (:37-44), `import_vcf_file`
(:178-213), `potatoParser` (:216-218) — and produces the buffers that cross the C ABI
(`chrs`, `pos`, `gt`, `wei` f64 [n,3], `dp`).

The reference delegates VCF reading to scikit-allel (parsers.py:184,189), which is not
available here; `read_vcf_minimal` is an in-repo reader that reproduces the fields the path
uses (first sample's GT and PL, CHROM, POS, INFO/DP).  It is validated against the golden
facts of the reference's sample files (SURVEY.md A.7).

Documented deviation (SURVEY.md A.8 Q5): BED inputs carry dp = "NA"; the reference crashes
in np.nanmean on the first parse (parsers.py:113) — here the depth statistic is nan instead.
"""
import gzip
import json
import locale
import logging
import mmap
import os
import re
import sys
import time

import numpy as np

log = logging.getLogger(__name__)

snp_thres = 4000   # snpmatch.py:18


def die(msg):
    sys.stderr.write('Error: ' + msg + '\n')
    sys.exit(1)


def parseGT(snpGT):
    """GT strings -> int8 codes: 1/1 -> 1, 0/1|1/0 -> 2, ./. -> -1, anything else 0.
    The separator is sniffed from the first element only (parsers.py:12-35)."""
    snpGT = np.asarray(snpGT)
    codes = np.zeros(len(snpGT), dtype="int8")
    if len(codes) == 0:
        return codes
    first = str(snpGT[0])
    if "|" in first:
        sep = "|"
    elif "/" in first:
        sep = "/"
    elif first.isdigit():
        return np.array(snpGT, dtype="int8")
    else:
        die("unable to parse the format of GT in vcf!")
    gt = snpGT.astype("str")
    codes[gt == "1" + sep + "1"] = 1
    codes[(gt == "0" + sep + "1") | (gt == "1" + sep + "0")] = 2
    codes[gt == "." + sep + "."] = -1
    return codes


def snp_binary_to_gt(snpBinary):
    """int8 codes -> GT byte strings (parsers.py:37-44)."""
    snpBinary = np.array(snpBinary, dtype="int8")
    table = {-1: b"./.", 0: b"0/0", 1: b"1/1", 2: b"0/1"}
    out = np.zeros(len(snpBinary), dtype="S8")
    for code, text in table.items():
        out[snpBinary == code] = text
    return out


def mean_depth(dp):
    """np.nanmean(dp) that yields nan instead of raising for the "NA" depth of BED inputs."""
    try:
        arr = np.asarray(dp, dtype=float)
    except (TypeError, ValueError):
        return float("nan")
    if arr.size == 0 or np.all(np.isnan(arr)):
        return float("nan")
    return float(np.nanmean(arr))


_DP_RE = re.compile(r"(?:^|;)DP=([^;]+)")


def vcf_record(f, sample_index=0):
    """What read_vcf_minimal takes from one record, f = the line's tab-separated fields: (chrom, pos, dp, gt, pl, has_pl) with
    dp = INFO/DP (-1 when absent or not an integer), gt rendered 'a/b', pl the first three PLs (-1 where missing) and has_pl
    whether FORMAT has a PL key; None when the line has fewer than 10 + sample_index fields."""
    if len(f) < 10 + sample_index:
        return None
    pos = int(f[1])
    m = _DP_RE.search(f[7])
    try:
        dp = int(m.group(1)) if m else -1
    except ValueError:
        dp = -1
    keys = f[8].split(":")
    vals = f[9 + sample_index].split(":")
    rec = dict(zip(keys, vals))
    alleles = re.split(r"[/|]", rec.get("GT", "."))
    if len(alleles) == 1:
        alleles = [alleles[0], "."] if alleles[0] != "." else [".", "."]
    gt = "/".join(a if a != "" else "." for a in alleles[:2])
    pl = [-1.0, -1.0, -1.0]
    if "PL" in rec:
        for i, v in enumerate(rec["PL"].split(",")[:3]):
            if v not in (".", ""):
                pl[i] = float(v)
    return f[0], pos, dp, gt, pl, "PL" in keys


def read_vcf_minimal(inFile, sample_index=0):
    """Minimal VCF reader: CHROM, POS, INFO/DP, and GT + PL of one sample.

    Output conventions follow what the reference receives from scikit-allel
    (parsers.py:191-206): GT rendered as 'a/b' with '.' for a missing allele (phasing is
    dropped by GenotypeArray.to_gt), PL as float [n,3] with -1 for missing entries,
    dp = INFO/DP (-1 when absent on a record) or an array of "NA" when the header declares
    no INFO DP field."""
    opener = gzip.open if str(inFile).endswith(".gz") else open
    chrom, pos, gts, pls, dps = [], [], [], [], []
    has_info_dp = False
    has_pl = False
    with opener(inFile, "rt") as fh:
        for line in fh:
            if line.startswith("##"):
                if line.startswith("##INFO=<ID=DP,"):
                    has_info_dp = True
                continue
            if line.startswith("#"):
                continue
            r = vcf_record(line.rstrip("\n").split("\t"), sample_index)
            if r is None:
                continue
            chrom.append(r[0])
            pos.append(r[1])
            dps.append(r[2])
            gts.append(r[3])
            pls.append(r[4])
            has_pl |= r[5]
    out = {
        "chr": np.array(chrom, dtype="str"),
        "pos": np.array(pos, dtype=np.int64),
        "gt": np.array(gts, dtype="str"),
    }
    if has_pl:
        out["wei"] = np.array(pls, dtype=float).reshape(-1, 3)
    out["dp"] = np.array(dps, dtype=np.int64) if has_info_dp else np.repeat("NA", len(pos))
    return out


def read_vcf_samples(inFile):
    """All samples of a VCF: 'samples' str[S], 'chr', 'pos', 'gt' str [n,S] rendered 'a/b' as scikit-allel's
    GenotypeArray.to_gt does for the reference (parsers.py:191-193).  Used by genotype_cross (genotype_cross.py:212)."""
    opener = gzip.open if str(inFile).endswith(".gz") else open
    samples, chrom, pos, rows = [], [], [], []
    with opener(inFile, "rt") as fh:
        for line in fh:
            if line.startswith("##"):
                continue
            f = line.rstrip("\n").split("\t")
            if line.startswith("#"):
                samples = f[9:]
                continue
            if len(f) < 10:
                continue
            chrom.append(f[0])
            pos.append(int(f[1]))
            gt_at = f[8].split(":").index("GT") if "GT" in f[8].split(":") else -1
            row = []
            for cell in f[9:9 + len(samples)]:
                v = cell.split(":")
                raw = v[gt_at] if 0 <= gt_at < len(v) else "."
                alleles = re.split(r"[/|]", raw)
                if len(alleles) == 1:
                    alleles = [alleles[0], "."] if alleles[0] != "." else [".", "."]
                row.append("/".join(a if a != "" else "." for a in alleles[:2]))
            row += ["./."] * (len(samples) - len(row))
            rows.append(row)
    return {"samples": np.array(samples, dtype="str"), "chr": np.array(chrom, dtype="str"), "pos": np.array(pos, dtype=np.int64),
            "gt": np.array(rows, dtype="str").reshape(len(pos), len(samples))}


def import_vcf_file(inFile, logDebug=False, samples_to_load=[0], add_fields=None):
    """Same role as parsers.py:178-213; returns dict with 'gt' [n,1], 'wei' [n,1,3], 'chr', 'pos', 'dp'.
    samples_to_load=None loads the genotypes of every sample ('samples', 'gt' [n,S]; genotype_cross.py:212)."""
    if samples_to_load is None:
        out = read_vcf_samples(inFile)
        out["dp"] = np.repeat("NA", len(out["pos"]))
        return out
    raw = read_vcf_minimal(inFile, sample_index=samples_to_load[0])
    snp_inputs = {"chr": raw["chr"], "pos": raw["pos"], "dp": raw["dp"], "gt": raw["gt"][:, None]}
    if "wei" in raw:
        snp_inputs["wei"] = raw["wei"][:, None, :]
    return snp_inputs


class ParseInputs(object):
    """VCF / BED / npz -> chrs, pos, gt, wei, dp (parsers.py:59-175)."""

    def __init__(self, inFile, logDebug=True, outFile="parser"):
        if outFile == "parser" or not outFile:
            outFile = inFile + ".snpmatch"
        if os.path.isfile(inFile + ".snpmatch.npz"):
            log.info("snpmatch parser dump found! loading %s", inFile + ".snpmatch.npz")
            snps = np.load(inFile + ".snpmatch.npz")
            self.load_snp_info(snps['chr'], snps['pos'], snps['gt'], snps['wei'], snps['dp'])
        elif os.path.isfile(inFile):
            _, inType = os.path.splitext(inFile)
            if inType == '.npz':
                snps = np.load(inFile)
                self.load_snp_info(snps['chr'], snps['pos'], snps['gt'], snps['wei'], snps['dp'])
            else:
                if inType == '.vcf' or os.path.basename(inFile).endswith(".vcf.gz"):
                    parsed = self.read_vcf(inFile, logDebug)
                elif inType == '.bed':
                    parsed = self.read_bed(inFile, logDebug)
                else:
                    die("input file type %s not supported" % inType)
                self.load_snp_info(*parsed)
                self.save_snp_info(outFile)
                self.case_interpret_inputs(outFile + ".stats.json")

    def load_snp_info(self, snpCHR, snpPOS, snpGT, snpWEI, DPmean):
        self.chrs = np.array(snpCHR, dtype="str")
        self.pos = np.array(snpPOS, dtype=int)
        self.gt = np.array(snpGT, dtype="str")
        self.wei = np.array(snpWEI, dtype=float)
        self.dp = DPmean
        pc = getattr(self, "_pl_codes", None)       # read_vcf: integer PLs as weight codes
        self._coded = (pc[0], pc[1], self.wei) if pc is not None and len(pc[0]) == len(self.wei) else None
        self._pl_codes = None

    def coded_weights(self):
        """(codes uint16 [n,3], table f64 [V]) with table[codes] == wei bit for bit, or None when the weights take more than
        65536 distinct values.  A VCF with integer PLs gives the codes for free (code = PL, table = exp(-PL/10): read_vcf keeps
        them); any other input is dictionary-coded once here and cached.  This is what crosses the PCIe bus in the batched path
        (lib.CodedSamples): 6 instead of 24 bytes per marker."""
        cached = getattr(self, "_coded", None)
        if cached is None or cached[2] is not self.wei:
            from .. import lib
            iw = lib.index_weights(self.wei)
            cached = (iw[0], iw[1], self.wei) if iw is not None else (None, None, self.wei)
            self._coded = cached
        return None if cached[0] is None else (cached[0], cached[1])

    def save_snp_info(self, outFile):
        np.savez(outFile, chr=self.chrs, pos=self.pos, gt=self.gt, wei=self.wei, dp=self.dp)

    def case_interpret_inputs(self, outFile):
        from . import snpmatch as _sm
        n = len(self.chrs)
        names, counts = np.unique(self.chrs, return_counts=True)
        stat = {
            "snps": dict((str(k), int(v)) for k, v in zip(names, counts)),
            "interpretation": {"case": 1, "text": "Attention: low number of SNPs provided"} if n < snp_thres
            else {"case": 0, "text": "Sufficient number of SNPs"},
            "num_of_snps": n,
            "depth": mean_depth(self.dp),
            "percent_heterozygosity": _sm.getHeterozygosity(self.gt),
        }
        with open(outFile, "w") as out_stats:
            out_stats.write(json.dumps(stat))

    @staticmethod
    def get_wei_from_GT(snpGT):
        """One-hot weights of the called genotype, columns (0/0, 0/1, 1/1) (parsers.py:132-139)."""
        codes = parseGT(snpGT)
        wei = np.zeros((len(codes), 3), dtype=float)
        wei[codes == 0, 0] = 1.0
        wei[codes == 2, 1] = 1.0
        wei[codes == 1, 2] = 1.0
        return wei

    @staticmethod
    def read_bed(inFile, logDebug):
        """Three whitespace-separated columns chr, pos, GT (parsers.py:118-130)."""
        chrs, pos, gt = [], [], []
        with open(inFile) as fh:
            for line in fh:
                f = line.split()
                if len(f) < 3:
                    continue
                chrs.append(f[0])
                pos.append(int(f[1]))
                gt.append(f[2])
        gt = np.array(gt)
        return (np.array(chrs, dtype="str"), np.array(pos, dtype=int), gt,
                ParseInputs.get_wei_from_GT(gt), "NA")

    def read_vcf(self, inFile, logDebug):
        """First sample; drop no-calls; wei = exp(-PL/10), GT one-hot where PL is absent
        (parsers.py:141-157)."""
        v = import_vcf_file(inFile, logDebug, samples_to_load=[0])
        parsed, self._pl_codes = vcf_called_inputs(v['chr'], v['pos'], v['gt'][:, 0], v['wei'][:, 0] if 'wei' in v else None, v['dp'])
        return parsed

    def filter_chr_names(self):
        """parsers.py:159-163: strip every 'chr' (any case); ids in first-appearance order."""
        from . import labels
        self.g_chrs, _, mapped = labels.map_labels(self.chrs, lambda c: re.sub("chr", "", c, flags=re.IGNORECASE))
        self.g_chrs_ids = labels.factorize(mapped)[1] if len(mapped) else self.g_chrs

    def save_to_bed(self, outFile):
        with open(outFile, "w") as fh:
            for c, p, g in zip(self.chrs, self.pos, self.gt):
                fh.write("%s\t%s\t%s\n" % (c, p, g))


def vcf_called_inputs(chrs, pos, gt_all, pl, dp):
    """The step of ParseInputs.read_vcf from one sample's VCF fields to (chrs, pos, gt, wei, dp): drop the no-calls; wei =
    exp(-PL/10), the called genotype's one-hot where a marker has no PL and everywhere when pl is None (no PL key in the file).
    pl: float [n,3] with -1 for a missing value, or None.  Returns (those five, pl_codes): pl_codes = (codes uint16 [m,3],
    table) when the PLs are integers, the dictionary codes of the weights that coded_weights() hands out, else None."""
    req = np.flatnonzero((gt_all != './.') & (gt_all != '.|.'))
    gt = gt_all[req]
    pl_codes = None
    if pl is not None:
        pl = pl[req]
        no_pl = np.all(pl == -1, axis=1)
        wei = np.exp(pl / (-10))
        wei[no_pl, ] = ParseInputs.get_wei_from_GT(gt[no_pl])
        # integer PLs are ready-made dictionary codes of the weights: table[k] = exp(k / -10), one extra entry for 0.0
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
        wei = ParseInputs.get_wei_from_GT(gt)
    return (chrs[req], pos[req], gt, wei, dp[req]), pl_codes


# ---- every sample column of one VCF, the genotype columns parsed on the device (`inbred/cross --samples_vcf`) ----------------
VCF_CHUNK_BYTES = 64 << 20
# allele codes of snpm_vcf_fetch: 0 '.', 1 + d for the digit d, 11 + 10x + y for the two digits xy; class = a1 * 111 + a2
_ALLELES = ["."] + [str(d) for d in range(10)] + ["%d%d" % (x, y) for x in range(10) for y in range(10)]
VCF_GT_TEXT = np.array([a + "/" + b for a in _ALLELES for b in _ALLELES])
VCF_GT_LEN = np.array([len(t) for t in VCF_GT_TEXT.tolist()])
_LINE_END = re.compile(rb"\r\n|\r|\n")


# text per device call of BgzfReader, chosen end to end: makeDB_from_vcf of 4.57 GB of text (NVIDIA B200, three alternating runs
# of each size; DESIGN.md section 6) took 5.5-6.4 s at 64 MB, 7.0-8.4 s at 256 MB and 5.7-6.6 s at 512 MB.  The kernel alone
# favours larger batches (111 / 42 / 35 ms: 1000 members do not fill the GPU); the host's reading of the text out of the pinned
# buffer favours smaller ones (read_s 2.7-3.0 / 4.0-4.8 / 3.2-3.8 s)
BGZF_BATCH_BYTES = 64 << 20


class BgzfReader(object):
    """A BGZF file read as its text, its members inflated on CUDA device `device` (lib.BgzfInflater), in batches of consecutive
    members of at most batch_bytes of text and batch_bytes // 4 compressed bytes whatever the caller's n.  read(n) returns at
    most n bytes of the current batch (b"" only at the end of the text).  A refused member raises gzip.BadGzipFile naming the
    path, its byte offset and the reason.  Counters: comp_bytes (compressed bytes inflated), inflate_s (wall time of the device
    calls, copies of the compressed bytes into pinned staging included) and ms (device ms of the copies up, the kernel and the
    copies down).  Made by BgzfReader.open."""

    def __init__(self, path, mm, member_off, isize, device, batch_bytes):
        from .. import lib
        self.path, self._mm, self._data = path, mm, np.frombuffer(mm, np.uint8)
        self._off = member_off
        text_end = np.concatenate([[0], np.cumsum(isize)])
        in_cap = max(batch_bytes // 4, 1 << 17)
        self._bounds, i, n = [], 0, len(isize)
        while i < n:
            j = min(int(np.searchsorted(text_end, text_end[i] + batch_bytes, "right")),
                    int(np.searchsorted(member_off, member_off[i] + in_cap, "right"))) - 1
            j = max(j, i + 1)
            self._bounds.append((i, j))
            i = j
        max_out = max(int(max(text_end[j] - text_end[i] for i, j in self._bounds)), 1)
        max_in = max(int(max(member_off[j] - member_off[i] for i, j in self._bounds)), 1)
        self._inf = lib.BgzfInflater(device, max_in, max_out)
        self._batch, self._at, self._end = 0, 0, 0
        self.comp_bytes, self.inflate_s = 0, 0.0

    @classmethod
    def open(cls, path, device, batch_bytes=None):
        """A reader of path when it is all BGZF (lib.bgzf_scan), else None; batch_bytes defaults to BGZF_BATCH_BYTES."""
        from .. import lib
        with open(path, "rb") as f:
            if os.fstat(f.fileno()).st_size == 0:
                return None
            mm = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)
        table = lib.bgzf_scan(np.frombuffer(mm, np.uint8))
        if table is None:
            mm.close()
            return None
        return cls(path, mm, table[0], table[1], device, batch_bytes or BGZF_BATCH_BYTES)

    @property
    def ms(self):
        return self._inf.ms

    def _next(self):
        while self._batch < len(self._bounds):
            i, j = self._bounds[self._batch]
            self._batch += 1
            a = int(self._off[i])
            t0 = time.perf_counter()
            self._end = self._inf.inflate(self._data[a:int(self._off[j])], self._off[i:j + 1] - a, path=self.path, base=a)
            self.inflate_s += time.perf_counter() - t0
            self.comp_bytes += int(self._off[j]) - a
            self._at = 0
            if self._end:
                return True
        return False

    def read(self, n=-1):
        if n is None or n < 0:
            parts = []
            while self._at < self._end or self._next():
                parts.append(self.read(self._end - self._at))
            return b"".join(parts)
        if n == 0 or (self._at == self._end and not self._next()):
            return b""
        k = min(n, self._end - self._at)
        out = self._inf.text(self._at, self._at + k)
        self._at += k
        return out

    def readable(self):
        return True

    def close(self):
        if self._mm is not None:
            self._inf.close()
            self._data = None
            try:
                self._mm.close()
            except BufferError:               # a traceback still holds a view of the mapping: it is unmapped when that goes
                pass
            self._mm = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def _open_binary(path, device=None):
    """path opened for binary reading of its text: a BgzfReader inflating on CUDA device `device` when device is given, the
    name ends in .gz and the file is all BGZF; gzip.open for any other .gz; open otherwise."""
    if not str(path).endswith(".gz"):
        return open(path, "rb")
    if device is not None:
        reader = BgzfReader.open(path, device)
        if reader is not None:
            return reader
    return gzip.open(path, "rb")


def _inflate_timings(fh, tm):
    """The decompression route of fh into tm: inflate = "device" (BgzfReader), "host" (gzip) or None (plain text); for .gz,
    gz_bytes = compressed bytes read; for the device route, inflate_s (wall time of the device calls, inside read_s) and the
    device times inflate_h2d_ms, inflate_ms (k_bgzf_inflate) and d2h_ms."""
    if isinstance(fh, BgzfReader):
        tm.update(inflate="device", gz_bytes=fh.comp_bytes, inflate_s=fh.inflate_s, inflate_h2d_ms=float(fh.ms[0]),
                  inflate_ms=float(fh.ms[1]), d2h_ms=float(fh.ms[2]))
    elif isinstance(fh, gzip.GzipFile):
        tm.update(inflate="host", gz_bytes=fh.fileobj.tell() if fh.fileobj is not None else 0)
    else:
        tm["inflate"] = None


def read_vcf_header(fh, block=1 << 20, meta_lines=None):
    """Header of a VCF opened in binary mode, read up to and including its #CHROM line with the universal-newline rule of the
    text-mode readers: returns (sample names, has_info_dp, lines read, the bytes read past the #CHROM line).  Raises ValueError
    when a record (10 fields or more) comes before the #CHROM line, or when there is no #CHROM line.  meta_lines (optional
    list) receives the '##' lines before the #CHROM line, without their line ends."""
    enc = locale.getpreferredencoding(False)
    buf, at, n, has_dp, eof = b"", 0, 0, False, False
    while True:
        m = _LINE_END.search(buf, at)
        if m is None or (m.group() == b"\r" and m.end() == len(buf) and not eof):
            if not eof:
                piece = fh.read(block)
                eof = not piece
                buf, at = buf[at:] + piece, 0
                continue
            if at == len(buf):
                raise ValueError("no #CHROM line")
            line, at = buf[at:], len(buf)
        else:
            line, at = buf[at:m.start()], m.end()
        n += 1
        text = line.decode(enc)
        if text.startswith("##"):
            has_dp |= text.startswith("##INFO=<ID=DP,")
            if meta_lines is not None:
                meta_lines.append(text)
        elif text.startswith("#"):
            return text.split("\t")[9:], has_dp, n, buf[at:]
        elif len(text.split("\t")) >= 10:
            raise ValueError("line %d is a record before the #CHROM line" % n)


def vcf_sample_names(path):
    """The sample columns of a VCF's #CHROM line."""
    with _open_binary(path) as fh:
        return read_vcf_header(fh)[0]


def _whole_lines(buf, limit, eof):
    """Bytes of buf[:limit] up to its last line end; a trailing '\r' counts only when the byte after it is known."""
    n = min(len(buf), limit)
    cut = buf.rfind(b"\n", 0, n) + 1
    r = buf.rfind(b"\r", cut, n)
    while r >= 0:
        if (r + 1 < len(buf) and buf[r + 1] != 10) or (r + 1 == len(buf) and eof):
            return r + 1
        r = buf.rfind(b"\r", cut, r)
    return cut


def vcf_chunks(fh, head, chunk_bytes, path, line_no, parse, tm):
    """The text after the #CHROM line of the VCF fh (binary; head = the bytes the header reader read past that line) in chunks of
    whole lines of at most chunk_bytes, a line end added after an unterminated last line; each chunk goes through parse (a
    lib.VcfParser method).  Yields (chunk, parse(chunk), lines of the file before the chunk), line_no counting the header's.  A
    line longer than chunk_bytes raises ValueError naming it.  Adds to tm: read_s (read and gunzip), device_s, h2d_ms,
    kernel_ms, h2d_bytes."""
    buf, eof = bytearray(head), False
    while True:
        t0 = time.perf_counter()
        while len(buf) < chunk_bytes and not eof:
            piece = fh.read(chunk_bytes - len(buf))
            eof = not piece
            buf += piece
        if eof and buf and buf[-1] not in (10, 13):
            buf += b"\n"
        tm["read_s"] += time.perf_counter() - t0
        if not buf:
            return
        cut = _whole_lines(buf, chunk_bytes, eof)
        if cut == 0:
            raise ValueError("%s: line %d is longer than the chunk of %d bytes" % (path, line_no + 1, chunk_bytes))
        chunk = bytes(memoryview(buf)[:cut])
        del buf[:cut]
        t0 = time.perf_counter()
        r = parse(chunk)
        tm["device_s"] += time.perf_counter() - t0
        tm["h2d_ms"] += r["h2d_ms"]
        tm["kernel_ms"] += r["kernel_ms"]
        tm["h2d_bytes"] += len(chunk)
        yield chunk, r, line_no
        line_no += r["n_lines"]


def read_vcf_many(path, device=0, chunk_bytes=VCF_CHUNK_BYTES, timings=None):
    """Every sample column of a VCF (plain or .vcf.gz): [(sample name, ParseInputs)], where sample s's ParseInputs has the
    chrs, pos, gt, wei, dp and coded_weights() of ParseInputs on a VCF of the same header, the 9 fixed columns and column s
    alone (read_vcf_minimal(path, sample_index=s) + ParseInputs.read_vcf).  The host reads (and decompresses) the text after
    the #CHROM line in chunks of whole lines of at most chunk_bytes; the genotype columns are parsed on CUDA device `device`
    (lib.VcfParser); records the device flags are re-parsed with vcf_record.  Nothing is written next to the VCF and no parser
    dump is loaded.  A line longer than chunk_bytes, a record before the #CHROM line and a VCF without sample columns raise
    ValueError.  A BGZF .vcf.gz is inflated on the same device (BgzfReader).  timings (optional dict) receives seconds and
    bytes of the stages, the decompression route (_inflate_timings) and, under "fallback", the indices of the records the
    Python code parsed."""
    from .. import lib
    enc = locale.getpreferredencoding(False)
    tm = timings if timings is not None else {}
    for k in ("read_s", "device_s", "host_chunk_s", "assemble_s", "h2d_ms", "kernel_ms", "h2d_bytes"):
        tm[k] = 0
    tm["fallback"] = []
    t0 = time.perf_counter()
    fh = _open_binary(path, device)
    try:
        names, has_info_dp, line_no, head = read_vcf_header(fh)
        if not names:
            raise ValueError("%s has no sample columns" % path)
        S = len(names)
        name_id, name_list = {}, []

        def chrom_id(text):
            if text not in name_id:
                name_id[text] = len(name_list)
                name_list.append(text)
            return name_id[text]
        rec = {k: [] for k in ("cid", "pos", "dp", "nsf", "has_pl")}
        chunks, fb = [], [[] for _ in range(S)]
        n_rec = 0
        tm["read_s"] += time.perf_counter() - t0
        parser = lib.VcfParser(device, S, chunk_bytes)
        try:
            for chunk, r, _ in vcf_chunks(fh, head, chunk_bytes, path, line_no, parser.parse, tm):
                t0 = time.perf_counter()
                if r["non_ascii"]:
                    chunk.decode(enc)                  # the text-mode readers fail on what does not decode
                has_info_dp |= r["info_dp_lines"] > 0
                flags, ls = r["flags"], r["line_start"]
                lines = np.flatnonzero(flags & lib.VcfParser.FLAG_RECORD)
                fl = flags[lines]
                pos, dp, nsf = r["pos"][lines].astype(np.int64), r["dp"][lines].astype(np.int64), r["nsf"][lines]
                has_pl = (fl & lib.VcfParser.FLAG_HAS_PL) != 0
                # CHROM: decoded where it may differ from the previous record's, carried forward elsewhere
                new = np.flatnonzero(fl & lib.VcfParser.FLAG_NEW_CHROM)
                ids = np.zeros(len(lines), np.int32)
                ids[new] = [chrom_id(chunk[ls[L]:ls[L] + r["chrom_len"][L]].decode(enc)) for L in lines[new].tolist()]
                src = np.zeros(len(lines), np.int64)
                src[new] = new
                cid = ids[np.maximum.accumulate(src)] if len(lines) else ids
                for k in np.flatnonzero(fl & lib.VcfParser.FLAG_FALLBACK).tolist():
                    L = int(lines[k])
                    f = chunk[ls[L]:ls[L + 1]].rstrip(b"\r\n").decode(enc).split("\t")
                    first = vcf_record(f, 0)
                    cid[k], pos[k], dp[k], has_pl[k] = chrom_id(first[0]), first[1], first[2], first[5]
                    for smp in range(min(int(nsf[k]), S)):
                        one = vcf_record(f, smp)
                        if one[3] not in ('./.', '.|.'):
                            fb[smp].append((n_rec + k, one[3], one[4]))
                    tm["fallback"].append(n_rec + k)
                for key, v in (("cid", cid), ("pos", pos), ("dp", dp), ("nsf", nsf), ("has_pl", has_pl)):
                    rec[key].append(v)
                rec_of_line = np.cumsum(flags & lib.VcfParser.FLAG_RECORD, dtype=np.int64) - 1 + n_rec
                chunks.append((r["sample_off"], rec_of_line[r["line"]], r["cls"], r["pl"]))
                n_rec += len(lines)
                tm["host_chunk_s"] += time.perf_counter() - t0
        finally:
            parser.close()
    finally:
        _inflate_timings(fh, tm)
        fh.close()
    t0 = time.perf_counter()
    rec = {k: (np.concatenate(v) if v else np.zeros(0)) for k, v in rec.items()}
    cid_all, pos_all, dp_all = rec["cid"].astype(np.int64), rec["pos"].astype(np.int64), rec["dp"].astype(np.int64)
    nsf_all = np.minimum(rec["nsf"].astype(np.int64), S)
    has_pl_all = rec["has_pl"].astype(bool)
    names_arr = np.array(name_list, dtype="str")
    # per sample, the records it has (nsf > s): whether any has a PL key, how many there are, the longest CHROM among them
    # (read_vcf_minimal's arrays are as wide as their longest entry)
    pl_upto = int(nsf_all[has_pl_all].max()) if has_pl_all.any() else 0
    has_rec = np.cumsum(np.bincount(nsf_all, minlength=S + 1)[::-1])[::-1] if len(nsf_all) else np.zeros(S + 1, np.int64)
    longest = np.zeros(S + 1, np.int64)
    if len(nsf_all):
        np.maximum.at(longest, nsf_all, np.array([len(c) for c in name_list], np.int64)[cid_all])
    longest = np.maximum.accumulate(longest[::-1])[::-1]
    out = []
    for smp in range(S):
        parts = [(c_rec[o[smp]:o[smp + 1]], c_cls[o[smp]:o[smp + 1]], c_pl[o[smp]:o[smp + 1]]) for o, c_rec, c_cls, c_pl in chunks]
        idx = np.concatenate([p[0] for p in parts]) if parts else np.zeros(0, np.int64)
        cls = np.concatenate([p[1] for p in parts]) if parts else np.zeros(0, np.uint16)
        gt = VCF_GT_TEXT[cls]
        pl = (np.concatenate([p[2] for p in parts]) if parts else np.zeros((0, 3), np.int32)).astype(np.float64)
        width = int(VCF_GT_LEN[cls].max()) if len(cls) else 3
        if fb[smp]:
            idx = np.concatenate([idx, np.array([e[0] for e in fb[smp]], np.int64)])
            gt = np.concatenate([gt, np.array([e[1] for e in fb[smp]], dtype="str")])
            pl = np.concatenate([pl, np.array([e[2] for e in fb[smp]], dtype=np.float64).reshape(-1, 3)])
            width = max(width, max(len(e[1]) for e in fb[smp]))
            order = np.argsort(idx, kind="stable")
            idx, gt, pl = idx[order], gt[order], pl[order]
        n_have = int(has_rec[smp + 1])
        gt = gt.astype("<U%d" % (max(width, 3) if n_have else 1))
        chrs = names_arr[cid_all[idx]].astype("<U%d" % max(int(longest[smp + 1]), 1))
        dp = dp_all[idx] if has_info_dp else np.repeat("NA", len(idx))
        parsed, pl_codes = vcf_called_inputs(chrs, pos_all[idx], gt, pl if smp < pl_upto else None, dp)
        inp = object.__new__(ParseInputs)
        inp._pl_codes = pl_codes
        inp.load_snp_info(*parsed)
        out.append((names[smp], inp))
    tm["assemble_s"] += time.perf_counter() - t0
    return out


def _population_header(fh, path):
    """read_vcf_header for read_vcf_gt_codes: (sample names, lines read, bytes past the #CHROM line); ValueError naming path when
    there is no #CHROM line, a record comes before it or it names no sample column."""
    try:
        names, _, line_no, head = read_vcf_header(fh)
    except ValueError as e:
        raise ValueError("%s: %s" % (path, e))
    if not names:
        raise ValueError("%s has no sample columns" % path)
    return names, line_no, head


def vcf_population_samples(path):
    """The sample names read_vcf_gt_codes(path) returns, or the ValueError of its header refusals; reads the header only and
    needs no device."""
    with _open_binary(path) as fh:
        return _population_header(fh, path)[0]


def read_vcf_gt_codes(path, device=0, chunk_bytes=VCF_CHUNK_BYTES, timings=None):
    """What genotype_cross takes from a multi-sample VCF (plain or .vcf.gz), its genotype columns parsed on CUDA device `device`:
    dict(samples str [S], chr str [n], pos int64 [n], gt_codes int8 [n, S]), equal to read_vcf_samples(path)'s samples, chr and
    pos and to parseGT of its gt.  The host reads (and decompresses) the text after the #CHROM line in chunks of whole lines of
    at most chunk_bytes; the device turns each chunk's records into rows of codes (lib.VcfParser.parse_gt_codes); the host decodes
    CHROM only where it may change and converts a POS that is not 1-9 plain digits with int().  Raises ValueError naming the line
    or value on the inputs read_vcf_samples gives no usable result for: a '#' line after the #CHROM line, a POS that int()
    rejects; and on no #CHROM line, a record before it, no sample columns and a line longer than chunk_bytes.  timings (optional
    dict) receives read_s, device_s, h2d_ms, kernel_ms, host_chunk_s, assemble_s (seconds, ms) and h2d_bytes, and the
    decompression route (_inflate_timings): a BGZF .vcf.gz is inflated on the same device (BgzfReader)."""
    from .. import lib
    chunk_bytes = int(chunk_bytes)
    enc = locale.getpreferredencoding(False)
    tm = timings if timings is not None else {}
    for k in ("read_s", "device_s", "host_chunk_s", "assemble_s", "h2d_ms", "kernel_ms", "h2d_bytes"):
        tm[k] = 0
    t0 = time.perf_counter()
    fh = _open_binary(path, device)
    try:
        names, line_no, head = _population_header(fh, path)
        S = len(names)
        name_id, name_list = {}, []

        def chrom_id(text):
            if text not in name_id:
                name_id[text] = len(name_list)
                name_list.append(text)
            return name_id[text]
        cids, positions, codes = [], [], []
        tm["read_s"] += time.perf_counter() - t0
        parser = lib.VcfParser(device, S, chunk_bytes)
        try:
            for chunk, r, line_no in vcf_chunks(fh, head, chunk_bytes, path, line_no, parser.parse_gt_codes, tm):
                t0 = time.perf_counter()
                if r["non_ascii"]:
                    chunk.decode(enc)                  # the text-mode reader fails on what does not decode
                flags, ls, clen = r["flags"], r["line_start"], r["chrom_len"]
                lines = np.flatnonzero(flags & lib.VcfParser.FLAG_RECORD)
                fl = flags[lines]
                refuse = []                           # (line in chunk, message): the earliest wins
                text = np.frombuffer(chunk, np.uint8)
                first = ls[:-1]
                hashes = np.flatnonzero((text[first] == 35) & (text[np.minimum(first + 1, len(text) - 1)] != 35))
                if len(hashes):
                    refuse.append((int(hashes[0]), "is a '#' line after the #CHROM line"))
                # POS: converted on the host where the device did not read 1-9 plain digits
                pos = r["pos"][lines].astype(np.int64)
                for k in np.flatnonzero(fl & lib.VcfParser.FLAG_FALLBACK).tolist():
                    L = int(lines[k])
                    p0 = int(ls[L] + clen[L] + 1)
                    v = chunk[p0:chunk.index(b"\t", p0)].decode(enc)
                    try:
                        pos[k] = int(v)
                    except (ValueError, OverflowError):
                        refuse.append((L, "has the POS %r, which does not read as an int64 integer" % v))
                        break
                if refuse:
                    L, msg = min(refuse)
                    raise ValueError("%s: line %d %s" % (path, line_no + L + 1, msg))
                # CHROM: decoded where it may differ from the previous record's, carried forward elsewhere
                new = np.flatnonzero(fl & lib.VcfParser.FLAG_NEW_CHROM)
                ids = np.zeros(len(lines), np.int32)
                ids[new] = [chrom_id(chunk[ls[L]:ls[L] + clen[L]].decode(enc)) for L in lines[new].tolist()]
                src = np.zeros(len(lines), np.int64)
                src[new] = new
                cids.append(ids[np.maximum.accumulate(src)] if len(lines) else ids)
                positions.append(pos)
                codes.append(r["codes"])
                tm["host_chunk_s"] += time.perf_counter() - t0
        finally:
            parser.close()
    finally:
        _inflate_timings(fh, tm)
        fh.close()
    t0 = time.perf_counter()
    cid = np.concatenate(cids) if cids else np.zeros(0, np.int32)
    out = {"samples": np.array(names, dtype="str"), "chr": np.array(name_list, dtype="str")[cid],
           "pos": np.concatenate(positions) if positions else np.zeros(0, np.int64),
           "gt_codes": np.concatenate(codes) if codes else np.zeros((0, S), np.int8)}
    tm["assemble_s"] += time.perf_counter() - t0
    return out


def potatoParser(inFile, logDebug, outFile="parser"):
    inputs = ParseInputs(inFile, logDebug, outFile)
    return (inputs.chrs, inputs.pos, inputs.gt, inputs.wei, inputs.dp)
