"""
Deterministic, block-addressable synthetic inputs (SURVEY.md section 8d).

The panel is a pure function of (seed, row, accession): the CUDA generator inside
`libsnpmatch_b200.so` (`snpm_db_fill_synthetic`, csrc/synth.cuh) and `panel_codes` below
compute the same integer hash, so a 10.7 M x 1135 (or x 20 000) panel can live only in HBM
while a CPU checker materialises just the rows it needs.  Integer arithmetic only — no
libm call whose last bit could differ between host and device.

Shapes follow the 1001 Genomes panel: TAIR10 chromosome lengths
(resources/genomes/athaliana_tair10.json), rows per chromosome proportional to length.
The sample recipe follows the reference's simulator (simulate.py:10-31) and the PL shape of
sample_files/701_501.filter.vcf (e.g. `0,9,87` at DP 3).
"""
import io
import struct
import zlib

import numpy as np

TAIR10_CHRS = ["1", "2", "3", "4", "5"]
TAIR10_CHRLEN = [30427671, 19698289, 23459830, 18585056, 26975502]

SEED_PANEL = 1001
SEED_SAMPLE = 501

MISS_THRESH = 3277      # of 65536 -> 5 % missing
HET_THRESH = 131        # of 65536 -> 0.2 % het

_M1 = np.uint64(0xBF58476D1CE4E5B9)
_M2 = np.uint64(0x94D049BB133111EB)
_GOLD = np.uint64(0x9E3779B97F4A7C15)


def mix64(key, seed):
    """splitmix64 finaliser of (key + (seed+1)*golden); uint64 in, uint64 out (wraps)."""
    with np.errstate(over="ignore"):
        z = np.asarray(key, dtype=np.uint64) + (np.uint64(seed) + np.uint64(1)) * _GOLD
        z = (z ^ (z >> np.uint64(30))) * _M1
        z = (z ^ (z >> np.uint64(27))) * _M2
        z = z ^ (z >> np.uint64(31))
    return z


def row_alt_threshold(seed, rows):
    """Per-row alternate-allele frequency as a 32-bit threshold: f = u^3 (mean 0.25,
    skewed towards rare variants), u uniform from the row hash."""
    z = mix64((np.asarray(rows, dtype=np.uint64) << np.uint64(20)) | np.uint64(0xFFFFF), seed ^ 0x5A5A)
    u = z >> np.uint64(32)
    return (((u * u) >> np.uint64(32)) * u) >> np.uint64(32)


def panel_codes_cols(seed, rows, cols):
    """int8 codes (0 ref, 1 alt, 2 het, -1 missing) for the given rows x accession columns."""
    rows = np.asarray(rows, dtype=np.uint64)
    cols = np.asarray(cols, dtype=np.uint64)
    z = mix64((rows[:, None] << np.uint64(20)) | cols[None, :], seed)
    thr = row_alt_threshold(seed, rows)[:, None]
    u = z >> np.uint64(32)
    miss = (z & np.uint64(0xFFFF)) < np.uint64(MISS_THRESH)
    het = ((z >> np.uint64(16)) & np.uint64(0xFFFF)) < np.uint64(HET_THRESH)
    code = np.where(u < thr, 1, 0).astype(np.int8)
    code[het] = 2
    code[miss] = -1
    return code


def panel_codes(seed, rows, n_acc):
    return panel_codes_cols(seed, rows, np.arange(n_acc))


def panel_layout(n_rows, chrlen=TAIR10_CHRLEN):
    """Rows per chromosome proportional to length -> chr_regions int64 [C,2]."""
    chrlen = np.asarray(chrlen, dtype=np.int64)
    share = np.floor(n_rows * chrlen / chrlen.sum()).astype(np.int64)
    share[0] += n_rows - share.sum()
    ends = np.cumsum(share)
    return np.stack([ends - share, ends], axis=1).astype(np.int64)


def panel_positions(n_rows, chrlen=TAIR10_CHRLEN, seed=SEED_PANEL):
    """Strictly increasing positions in [1, chrlen) per chromosome: an even grid plus a
    hashed jitter smaller than the grid step.  Returns (positions int32[N], chr_regions)."""
    regions = panel_layout(n_rows, chrlen)
    pos = np.empty(n_rows, dtype=np.int32)
    for c, (s, e) in enumerate(regions):
        nc = int(e - s)
        if nc == 0:
            continue
        span = int(chrlen[c]) - 2
        step = span // nc
        assert step >= 2, "panel too dense for chromosome %d" % c
        i = np.arange(nc, dtype=np.int64)
        base = (i * span) // nc
        jit = (mix64(i.astype(np.uint64) + np.uint64(s), seed ^ 0xC3C3) % np.uint64(step - 1 if step > 1 else 1)).astype(np.int64)
        pos[s:e] = (1 + base + jit).astype(np.int32)
    return pos, regions


def accession_ids(n_acc):
    return np.array([str(1000 + a) for a in range(n_acc)], dtype="S")


def _pl_weights(rng, gt_code, dp):
    """Integer PLs shaped like the sample VCF: called genotype 0, adjacent class 3*DP,
    opposite homozygote 30*DP (+-U{0..9}); order (0/0, 0/1, 1/1)."""
    n = len(gt_code)
    pl = np.zeros((n, 3), dtype=np.int64)
    adj = 3 * dp
    far = 30 * dp + rng.integers(0, 10, size=n)
    ref = gt_code == 0
    alt = gt_code == 1
    het = gt_code == 2
    pl[ref, 1] = adj[ref]
    pl[ref, 2] = far[ref]
    pl[alt, 1] = adj[alt]
    pl[alt, 0] = far[alt]
    pl[het, 0] = (10 * dp + rng.integers(0, 10, size=n))[het]
    pl[het, 2] = (10 * dp + rng.integers(0, 10, size=n))[het]
    return pl, np.exp(pl / -10.0)


def _gt_strings(gt_code):
    out = np.full(len(gt_code), "0/0", dtype="U3")
    out[gt_code == 1] = "1/1"
    out[gt_code == 2] = "0/1"
    return out


def hard_weights(gt_code):
    """One-hot weights of a called genotype (parsers.py:132-139)."""
    w = np.zeros((len(gt_code), 3), dtype=np.float64)
    w[gt_code == 0, 0] = 1.0
    w[gt_code == 2, 1] = 1.0
    w[gt_code == 1, 2] = 1.0
    return w


def make_sample(positions, chr_regions, chr_names, n_acc, true_acc=7, n_db=45000, n_extra=5000,
                seed=SEED_SAMPLE, panel_seed=SEED_PANEL, err=0.01, het=0.02, chr_prefix="Chr",
                mosaic=None, chrlen=TAIR10_CHRLEN):
    """One low-coverage sample.  Returns dict(chrs, pos, gt, wei, wei_hard, dp, rows) with
    markers sorted by (chromosome order of the panel, position).

    mosaic=(p1, p2, block_bp): genotype follows p1 / het(p1,p2) / p2 in alternating blocks
    (an F2-like sample for `cross`)."""
    rng = np.random.Generator(np.random.Philox(key=seed))
    n_rows = len(positions)
    n_db = min(n_db, n_rows)
    rows = np.sort(rng.choice(n_rows, size=n_db, replace=False))
    row_chr = np.searchsorted(chr_regions[:, 1], rows, side="right")
    if mosaic is None:
        code = panel_codes_cols(panel_seed, rows, [true_acc])[:, 0]
        code = np.where(code < 0, 0, code)
    else:
        p1, p2, block = mosaic
        cc = panel_codes_cols(panel_seed, rows, [p1, p2])
        c1 = np.where(cc[:, 0] < 0, 0, cc[:, 0])
        c2 = np.where(cc[:, 1] < 0, 0, cc[:, 1])
        phase = (positions[rows].astype(np.int64) // int(block)) % 3
        hetc = np.where(c1 == c2, c1, 2)
        code = np.where(phase == 0, c1, np.where(phase == 1, hetc, c2))
    flip = rng.random(n_db) < err
    code = np.where(flip & (code != 2), 1 - code, code).astype(np.int8)
    code = np.where(rng.random(n_db) < het, 2, code).astype(np.int8)
    # extra markers at positions absent from the panel
    ex_chr = rng.integers(0, len(chr_regions), size=n_extra)
    ex_pos = np.empty(n_extra, dtype=np.int64)
    for i in range(n_extra):
        ex_pos[i] = rng.integers(1, int(chrlen[ex_chr[i] % len(chrlen)]))
    s_chr_ix = np.concatenate([row_chr, ex_chr]).astype(np.int64)
    s_pos = np.concatenate([positions[rows].astype(np.int64), ex_pos])
    s_code = np.concatenate([code, rng.integers(0, 2, size=n_extra).astype(np.int8)])
    is_db = np.concatenate([np.ones(n_db, bool), np.zeros(n_extra, bool)])
    # drop extras colliding with a panel position or each other
    key = s_chr_ix * (1 << 32) + s_pos
    order = np.argsort(key, kind="stable")
    key, s_chr_ix, s_pos, s_code, is_db = key[order], s_chr_ix[order], s_pos[order], s_code[order], is_db[order]
    keep = np.ones(len(key), bool)
    keep[1:] = key[1:] != key[:-1]
    if n_extra:
        in_panel = np.zeros(len(key), bool)
        for c, (s, e) in enumerate(chr_regions):
            sel = np.flatnonzero(s_chr_ix == c)
            seg = positions[s:e]
            j = np.searchsorted(seg, s_pos[sel])
            j = np.minimum(j, max(len(seg) - 1, 0))
            in_panel[sel] = (seg[j] == s_pos[sel]) if len(seg) else False
        keep &= is_db | ~in_panel
    s_chr_ix, s_pos, s_code = s_chr_ix[keep], s_pos[keep], s_code[keep]
    n = len(s_pos)
    dp = 1 + rng.poisson(3, size=n)
    pl, wei = _pl_weights(rng, s_code, dp)
    chrs = np.array([chr_prefix + str(chr_names[i]) for i in s_chr_ix], dtype="str")
    return dict(chrs=chrs, pos=s_pos.astype(np.int64), gt=_gt_strings(s_code), wei=wei, wei_hard=hard_weights(s_code),
                dp=dp.astype(np.float64), pl=pl, chr_ix=s_chr_ix.astype(np.int32), code=s_code)


def small_panel(n_rows=6000, n_acc=40, seed=SEED_PANEL, chrlen=TAIR10_CHRLEN, chr_names=TAIR10_CHRS):
    """A fully materialised small panel for CPU tests and golden vectors."""
    pos, regions = panel_positions(n_rows, chrlen, seed)
    snps = panel_codes(seed, np.arange(n_rows), n_acc)
    return dict(snps=snps, positions=pos, chr_regions=regions, chrs=np.array(chr_names, dtype="str"),
                accessions=accession_ids(n_acc))


def make_sample_fast(positions, chr_regions, n_acc, true_acc, n_db=45000, n_extra=5000, seed=SEED_SAMPLE,
                     panel_seed=SEED_PANEL, err=0.01, het=0.02, chrlen=TAIR10_CHRLEN):
    """Vectorised variant of make_sample for large panels (no per-marker Python loop, no name strings):
    returns dict(chr_ix int32, pos int32, wei f64[n,3], code int8, rows int64) sorted by (chromosome, position).
    Extra markers sit at positions absent from the panel."""
    rng = np.random.Generator(np.random.Philox(key=seed))
    n_rows = len(positions)
    rows = np.unique(rng.integers(0, n_rows, size=int(n_db * 1.05) + 16))
    if len(rows) > n_db:
        rows = np.sort(rng.choice(rows, size=n_db, replace=False))
    code = panel_codes_cols(panel_seed, rows, [true_acc])[:, 0]
    code = np.where(code < 0, 0, code)
    flip = rng.random(len(rows)) < err
    code = np.where(flip & (code != 2), 1 - code, code)
    code = np.where(rng.random(len(rows)) < het, 2, code).astype(np.int8)
    row_chr = np.searchsorted(chr_regions[:, 1], rows, side="right")
    ex_chr = rng.integers(0, len(chr_regions), size=n_extra)
    ex_pos = (rng.random(n_extra) * (np.asarray(chrlen)[ex_chr] - 2)).astype(np.int64) + 1
    key_db = row_chr.astype(np.int64) * (1 << 32) + positions[rows].astype(np.int64)
    key_ex = np.unique(ex_chr.astype(np.int64) * (1 << 32) + ex_pos)
    # drop extras that collide with a panel position
    ec, ep = key_ex >> 32, key_ex & 0xFFFFFFFF
    hit = np.zeros(len(key_ex), bool)
    for c, (s, e) in enumerate(chr_regions):
        sel = np.flatnonzero(ec == c)
        seg = positions[s:e]
        if len(seg) and len(sel):
            j = np.minimum(np.searchsorted(seg, ep[sel]), len(seg) - 1)
            hit[sel] = seg[j] == ep[sel]
    key_ex = key_ex[~hit]
    key = np.concatenate([key_db, key_ex])
    s_code = np.concatenate([code, rng.integers(0, 2, size=len(key_ex)).astype(np.int8)])
    s_rows = np.concatenate([rows, np.full(len(key_ex), -1, dtype=np.int64)])
    o = np.argsort(key, kind="stable")
    key, s_code, s_rows = key[o], s_code[o], s_rows[o]
    dp = 1 + rng.poisson(3, size=len(key))
    pl, wei = _pl_weights(rng, s_code, dp)
    return dict(chr_ix=(key >> 32).astype(np.int32), pos=(key & 0xFFFFFFFF).astype(np.int32), wei=wei, code=s_code,
                rows=s_rows, dp=dp.astype(np.float64), pl=pl)


def pl_table(max_pl):
    """exp(-PL/10) for PL = 0..max_pl, computed as parsers.py:147-148 computes it per marker (PL / -10, then exp): the weight
    of a marker IS table[PL], bit for bit, so integer PLs are ready-made dictionary codes of the weights."""
    return np.exp(np.arange(int(max_pl) + 1) / -10.0)


# ---- multi-sample VCF text (tests and measurement of parsers.read_vcf_many) -----------------------------------------------
def multi_sample_vcf(n_records, n_samples, seed=7, line_end="\n", info_dp_header=True, late_info_dp=False, edge_cases=True,
                     hash_lines=True):
    """Seeded text of a VCF with n_samples sample columns.  With edge_cases, the records mix every GT form read_vcf_minimal
    renders (phased, single alleles, '.', empty, multi-digit, more than two alleles, GT missing from FORMAT or from the cell,
    PL before GT), PL forms (missing key, '.', fewer or more than three values, 3.5, 1e2), INFO DP forms (present, absent,
    DP=x, DP=1_0, ADP=, an empty DP= before a real one), cells with fewer subfields than FORMAT, records with fewer sample
    columns than the header (one with exactly 32), '##' and '#' lines, blank and short lines among the records and a non-ASCII chromosome name.
    late_info_dp puts a '##INFO=<ID=DP,' line among the records; without hash_lines its '#' lines among the records become '##'
    lines (the same text otherwise).  line_end may also be a list of line ends to cycle through.  Returns (text, fallback): fallback = the 0-based indices of
    the records the device parser cannot reproduce (lib.VcfParser.FLAG_FALLBACK), i.e. the ones it hands to the Python code."""
    rng = np.random.default_rng(seed)
    ends = line_end if isinstance(line_end, (list, tuple)) else [line_end]
    lines = ["##fileformat=VCFv4.2"]
    if info_dp_header:
        lines.append('##INFO=<ID=DP,Number=1,Type=Integer,Description="depth">')
    lines.append("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join("smp%d" % i for i in range(n_samples)))
    plain_gt = ["0/0", "0|1", "1/0", "1/1", "./.", ".", "0", "./1", "2/3", "0/0/1", "", "1|1", "10/1", "01/1", "./0", "1"]
    chroms = ["Chr1", "Chr2", "chr3", "Chr4", "Chr5"]
    fallback = []
    pos = 100
    for r in range(n_records):
        fb = False
        if late_info_dp and r == n_records // 2:
            lines.append('##INFO=<ID=DP,Number=1,Type=Integer,Description="depth">')
        if edge_cases and rng.random() < 0.03:
            extra = ["##INFO=<ID=XX,Number=1>", "#comment", "", "Chr1\t5\t.\tA\tT", "##contig=<ID=Chr1>"][rng.integers(0, 5)]
            lines.append(extra if hash_lines or extra != "#comment" else "#" + extra)
        chrom = chroms[min(r * len(chroms) // max(n_records, 1), len(chroms) - 1)]
        if edge_cases and r % 97 == 13:
            chrom, fb = "Chrü", True
        pos += int(rng.integers(1, 400))
        pos_text = str(pos)
        if edge_cases and r % 89 == 5:
            pos_text, fb = "+" + pos_text, True
        info = "DP=%d" % rng.integers(0, 99)
        if edge_cases:
            k = rng.integers(0, 10)
            info = ["DP=%d" % rng.integers(0, 99), "AC=1;DP=%d;MQ=4" % rng.integers(0, 99), "ADP=3", "ADP=3;DP=9", ".", "DP=;DP=4",
                    "DP=12", "AC=2", "DP=x", "DP=1_0"][k]
            fb |= k >= 8
        fmt = ["GT", "PL"]
        if edge_cases:
            k = rng.integers(0, 9)
            fmt = [["GT", "PL"], ["PL", "GT"], ["GT"], ["GT", "AD", "PL"], ["AD", "DP"], ["GT", "PL"], ["GT", "PL"], ["GT", "GT"],
                   ["GT", "PL", "PL"]][k]
            fb |= k >= 7
        n_fields = n_samples
        if edge_cases and rng.random() < 0.08:
            n_fields = int(rng.integers(1, n_samples + 1))
        if edge_cases and r % 61 == 7:
            n_fields = min(32, n_samples)              # the last field closes a full warp's batch of cells
        cells = []
        for s in range(n_fields):
            gt = plain_gt[rng.integers(0, len(plain_gt))] if edge_cases else ["0/0", "0/1", "1/1", "./."][rng.integers(0, 4)]
            bad_gt = edge_cases and rng.random() < 0.002
            if bad_gt:
                gt = "A/1"
            pl = ",".join(str(v) for v in rng.integers(0, 255, 3))
            bad_pl = False
            if edge_cases:
                k = rng.integers(0, 12)
                pl = [pl, pl, pl, pl, ".", "5,3", "1,2,3,4,5,6", "", ".,.,.", "0,.,7", "3.5,1,2", "1e2,0,3"][k]
                bad_pl = k >= 10
            vals = {"GT": gt, "PL": pl, "AD": "3,4", "DP": "7"}
            sub = [vals[k] for k in fmt]
            keep = len(sub)
            if edge_cases and rng.random() < 0.05:
                keep = int(rng.integers(0, len(sub)))
            sub = sub[:keep]
            cells.append(":".join(sub))
            if s < n_samples and len(set(fmt)) == len(fmt):
                if bad_gt and "GT" in fmt[:keep]:
                    fb = True
                if bad_pl and "PL" in fmt[:keep]:
                    fb = True
        lines.append("\t".join([chrom, pos_text, ".", "A", "T", ".", "PASS", info, ":".join(fmt)] + cells))
        if fb:
            fallback.append(r)
    text = "".join(line + ends[i % len(ends)] for i, line in enumerate(lines))
    return text, fallback


def split_vcf_column(text, s):
    """The single-sample VCF of column s of a multi-sample VCF's text: every header and '#' line, and every other line cut to
    its 9 fixed fields and field 9 + s (to its first 9 fields when it has no field 9 + s)."""
    out = []
    for line in io.StringIO(text, newline=None):
        f = line.rstrip("\n").split("\t")
        if line.startswith("##"):
            out.append(line.rstrip("\n"))
        elif line.startswith("#") or len(f) >= 10 + s:
            out.append("\t".join(f[:9] + f[9 + s:10 + s]))
        else:
            out.append("\t".join(f[:9]))
    return "".join(x + "\n" for x in out)


_GT_TOKEN = np.array([b"./.", b"0/0", b"1/1", b"0/1"])      # index code + 1


def panel_vcf(fh, n_rows, n_acc, seed=SEED_PANEL, block=4096):
    """A GT-only multi-sample VCF of the synthetic panel, written to the binary file fh: record r is row r at
    panel_positions(n_rows) on chromosome TAIR10_CHRS[c], sample a (named accession_ids) calls panel_codes(seed, r, a) as
    0/0, 1/1, 0/1 or ./. (missing).  Built from these codes, `makedb` gives the panel load_int8 would.  Returns (positions,
    chr_regions)."""
    positions, regions = panel_positions(n_rows)
    fh.write(b"##fileformat=VCFv4.2\n")
    for c, n in zip(TAIR10_CHRS, TAIR10_CHRLEN):
        fh.write(b"##contig=<ID=%s,length=%d>\n" % (c.encode(), n))
    fh.write(b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + b"\t".join(accession_ids(n_acc).tolist()) + b"\n")
    chrom = np.searchsorted(regions[:, 1], np.arange(n_rows), side="right")
    token = np.frombuffer(b"".join(t + b"\t" for t in _GT_TOKEN.tolist()), np.uint8).reshape(4, 4)
    for r0 in range(0, n_rows, block):
        rows = np.arange(r0, min(r0 + block, n_rows))
        cells = token[panel_codes(seed, rows, n_acc).astype(np.int64) + 1].reshape(len(rows), 4 * n_acc)
        cells[:, -1] = 10
        fh.write(b"".join(b"%s\t%d\t.\tA\tT\t.\tPASS\t.\tGT\t" % (TAIR10_CHRS[c].encode(), p) + line.tobytes()
                          for c, p, line in zip(chrom[rows].tolist(), positions[rows].tolist(), cells)))
    return positions, regions


POPULATION_GT = ["0/0", "1/1", "0/1", "1/0", "./.", "0|1", "1|1", ".", "0", "1/.", "./1", "2/2", "1/1/0", "", "1|", "10/1", "A/1"]


def population_vcf(fh, chrs, positions, n_samples, seed=11, edge_forms=True, block=4096):
    """A seeded population VCF for `genotype_cross`, written to the binary file fh: record r at chrs[r], positions[r], FORMAT GT
    or GT:DP, n_samples columns whose GT is drawn from POPULATION_GT (edge_forms) or from 0/0, 1/1, 0/1, ./. alone."""
    rng = np.random.default_rng(seed)
    forms = POPULATION_GT if edge_forms else POPULATION_GT[:3] + POPULATION_GT[4:5]
    fh.write(b"##fileformat=VCFv4.2\n")
    fh.write(b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join("p%d" % i for i in range(n_samples)).encode() + b"\n")
    gts = np.array([g.encode() for g in forms], dtype=object)
    for r0 in range(0, len(positions), block):
        rows = range(r0, min(r0 + block, len(positions)))
        pick = rng.integers(0, len(forms), size=(len(rows), n_samples))
        dp = rng.random(len(rows)) < 0.3
        out = []
        for k, r in enumerate(rows):
            cells = gts[pick[k]]
            if dp[k]:
                out.append(b"%s\t%d\t.\tA\tT\t.\tPASS\t.\tGT:DP\t" % (str(chrs[r]).encode(), positions[r]) + b"\t".join(c + b":5" for c in cells))
            else:
                out.append(b"%s\t%d\t.\tA\tT\t.\tPASS\t.\tGT\t" % (str(chrs[r]).encode(), positions[r]) + b"\t".join(cells))
        fh.write(b"\n".join(out) + b"\n")


BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def write_bgzf(path, data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, member_bytes=65280, eof=True):
    """Write data as BGZF (bgzip's format: gzip members with a BC extra subfield holding the member's size - 1), each member
    the raw DEFLATE stream of zlib.compressobj(level, wbits=-15, strategy).  member_bytes: text per member (65280, bgzip's
    default), or a list of the sizes of the members in order (they must sum to len(data); 0 gives an empty member).  eof
    appends the 28-byte EOF member.  Raises ValueError when a member would exceed 65536 bytes."""
    data = bytes(data)
    if isinstance(member_bytes, int):
        sizes = [min(member_bytes, len(data) - a) for a in range(0, len(data), member_bytes)]
    else:
        sizes = list(member_bytes)
        if sum(sizes) != len(data):
            raise ValueError("member sizes sum to %d, not %d" % (sum(sizes), len(data)))
    with open(path, "wb") as fh:
        at = 0
        for n in sizes:
            piece = data[at:at + n]
            at += n
            c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
            payload = c.compress(piece) + c.flush()
            size = 26 + len(payload)
            if n > 65536 or size > 65536:
                raise ValueError("a member of %d bytes of text takes %d bytes" % (n, size))
            fh.write(b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", size - 1) + payload
                     + struct.pack("<II", zlib.crc32(piece), n))
        if eof:
            fh.write(BGZF_EOF)
