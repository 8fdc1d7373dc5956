"""
`snpmatch makedb` — build the database this package matches against (SURVEY 8(f)-2).

Mirrors the steps of `snpmatch/core/makedb.py` without its external tools: the reference shells out to bcftools + sed to turn
a multi-sample VCF into `Chromosome,Position,<accession>...` rows of 0 / 1 / 2 / -1 (`getCSV`, makedb.py:34-62), parses that
CSV into per-chromosome lists (`pygwas/genotype.py:29-105`) and writes two HDF5 files, one chunked by row and one by column
(`makeHDF5s`, makedb.py:83-90).  Here the VCF is read directly (`vcf_to_csv`), the CSV is parsed with one vectorised read
(`load_csv`), and the matrix goes to the GPU once, where it is packed to 2 bits per call (`k_pack_int8`); the packed words are
written as ONE native file (`<db_id>.npz`, `Genotype.save_packed`) that serves row and column access and is what
`-d` of every other sub-command loads.  The genome JSON of the contig lengths (`<db_id>.json`) is written as in the reference.

`makedb --no_csv` (makeDB_from_vcf) builds the same .npz and .json without the CSV: the VCF text goes to the GPU in chunks
and comes back as packed panel rows (lib.VcfParser.parse_gt_packed), with the CSV route's rules for every cell, CHROM and POS.

Departure: genotype calls other than 0/0, 1/1, 0/1, 1/0, ./. (e.g. a third allele) pass through the reference's sed chain
unchanged and then break its CSV parser; here they are stored as missing (-1) and counted in the log.
"""
import gzip
import io
import json
import locale
import logging
import os.path
import re
import sys

import numpy as np
import pandas as pd

from . import parsers, snp_genotype

log = logging.getLogger(__name__)

_GT_CODE = {"0/0": "0", "0|0": "0", "1/1": "1", "1|1": "1", "0/1": "2", "0|1": "2", "1/0": "2", "1|0": "2", "./.": "-1", ".|.": "-1", ".": "-1"}


def die(msg):
    sys.stderr.write('Error: ' + msg + '\n')
    sys.exit(1)


def get_contigs(vcf_header):
    """Chromosome names and lengths from the ##contig lines of a VCF header (makedb.py:25-32)."""
    chr_names, chr_len = [], []
    for eh in vcf_header:
        if eh[0:8] == '##contig':
            body = eh.replace(">", "").replace("<", "")
            chr_names.append(body.split("ID=")[1].split(",")[0])
            chr_len.append(int(body.split("length=")[1].split(",")[0]))
    return {"ref_chrs": chr_names, "ref_chrlen": chr_len}


def vcf_to_csv(inVCF, outFile):
    """What getCSV (makedb.py:34-62) produces with bcftools + sed, read straight from the VCF: `<outFile>.csv` with the header
    `Chromosome,Position,<samples>` and one row of 0 / 1 / 2 / -1 per record, and `<outFile>.json` with the contigs."""
    opener = gzip.open if str(inVCF).endswith(".gz") else open
    header, other = [], 0
    with opener(inVCF, "rt") as fh, open(outFile + ".csv", "w") as out:
        for line in fh:
            if line.startswith("##"):
                header.append(line.rstrip("\n"))
                continue
            f = line.rstrip("\n").split("\t")
            if line.startswith("#"):
                out.write("Chromosome,Position" + "".join("," + s for s in f[9:]) + "\n")
                with open(outFile + ".json", "w") as js:
                    js.write(json.dumps(get_contigs(header), sort_keys=True, indent=4))
                continue
            if len(f) < 10:
                continue
            keys = f[8].split(":")
            at = keys.index("GT") if "GT" in keys else -1
            codes = []
            for cell in f[9:]:
                v = cell.split(":")
                code = _GT_CODE.get(v[at] if 0 <= at < len(v) else ".")
                if code is None:
                    code = "-1"
                    other += 1
                codes.append(code)
            out.write(f[0] + "," + f[1] + "".join("," + c for c in codes) + "\n")
    if other:
        log.warning("%s genotype calls are neither 0/0, 1/1, 0/1 nor ./. and were stored as missing", other)
    log.info("Number of contigs found: %s", len(get_contigs(header)["ref_chrs"]))


def _sniff(csvFile):
    with open(csvFile) as fh:
        head = fh.readline().rstrip("\n")
    sep = "\t" if ("\t" in head and "," not in head) else ","
    cols = [c.strip() for c in head.split(sep)]
    if len(cols) < 2 or cols[0] != 'Chromosome' or cols[1] not in ('Positions', 'Position'):
        raise Exception('First two columns must be in form  Chromosome, Positions')
    return sep, cols


def _index_columns(csvFile, sep):
    """The first two columns of the CSV as the CSV route reads them, one entry per row: labels (pandas dtype=str, so NA-like
    text such as 'NA' becomes 'nan') and positions (int() of the text, wrapped to int32)."""
    idx = pd.read_csv(csvFile, sep=sep, usecols=[0, 1], dtype=str)
    return idx.iloc[:, 0].to_numpy().astype("U"), idx.iloc[:, 1].to_numpy().astype(np.int64).astype(np.int32)


def _runs(keys):
    """First row of every run of equal keys in file order, and the runs' row ranges int64 [C, 2]."""
    n = len(keys)
    starts = np.concatenate([[0], np.flatnonzero(keys[1:] != keys[:-1]) + 1]) if n else np.zeros(0, dtype=np.int64)
    ends = np.concatenate([starts[1:], [n]]) if n else starts
    regions = np.stack([starts, ends], axis=1).astype(np.int64) if n else np.zeros((0, 2), dtype=np.int64)
    return starts, regions


def _index_arrays(csvFile, sep):
    """(chrs, chr_regions, positions) of pygwas' `load_csv_genotype_data` (pygwas/genotype.py:29-105): a chromosome entry per run
    of equal labels in file order, `chr_regions` the row ranges of the runs.  Reads the first two columns only."""
    labels, positions = _index_columns(csvFile, sep)
    starts, regions = _runs(labels)
    return (labels[starts] if len(labels) else labels), regions, positions


def load_csv(csvFile):
    """All arrays of the CSV in memory (small files, tests): snps int8 [N,A], positions, chrs, chr_regions, accessions (bytes)."""
    sep, cols = _sniff(csvFile)
    chrs, regions, positions = _index_arrays(csvFile, sep)
    geno = pd.read_csv(csvFile, sep=sep, usecols=range(2, len(cols)), dtype=np.int8) if len(cols) > 2 else pd.DataFrame(index=range(len(positions)))
    return {"snps": np.ascontiguousarray(geno.to_numpy(dtype=np.int8)).reshape(len(positions), len(cols) - 2), "positions": positions,
            "chrs": chrs, "chr_regions": regions, "accessions": np.array(cols[2:], dtype="S")}


def makeDB(csvFile, outFile, device=0, chunk_rows=200000):
    """CSV -> resident 2-bit panel -> `<outFile>.npz` (replaces makeHDF5s, makedb.py:83-90: one native file instead of the
    row-chunked and the column-chunked HDF5).  The genotype columns are streamed to the GPU `chunk_rows` rows at a time, so
    the int8 matrix (12 GB for the 1001-genomes panel) never sits in host memory.  Returns the open Genotype."""
    from .. import lib
    sep, cols = _sniff(csvFile)
    chrs, regions, positions = _index_arrays(csvFile, sep)
    n_acc = len(cols) - 2
    assert n_acc > 0, "the CSV holds no accession columns"
    log.info("packing %s SNPs x %s accessions on the GPU", len(positions), n_acc)
    db = lib.Database(positions, regions, n_acc, device=device)
    row0 = 0
    for block in pd.read_csv(csvFile, sep=sep, usecols=range(2, len(cols)), dtype=np.int8, chunksize=int(chunk_rows)):
        codes = np.ascontiguousarray(block.to_numpy(dtype=np.int8))
        db.load_int8(codes, row0=row0)
        row0 += len(codes)
    assert row0 == len(positions), "the CSV changed while it was read"
    g = object.__new__(snp_genotype.Genotype)
    g._finish(db, positions, chrs, regions, np.array(cols[2:], dtype="S"))
    g.save_packed(outFile + ".npz")
    log.info("wrote %s.npz", outFile)
    return g


def _csv_read(values, what):
    """Texts of one CSV column (CHROM or POS, none holding ',' or '"') as the CSV route reads them back (_index_columns): U
    labels for what == 'CHROM', int32 positions for 'POS'.  Returns (result, None), or (None, i) when it fails on values[i]."""
    def table(vals):
        col = "Chromosome,Position\n" + "".join(("%s,1\n" if what == "CHROM" else "x,%s\n") % v for v in vals)
        return _index_columns(io.StringIO(col), ",")[0 if what == "CHROM" else 1]
    try:
        return table(values), None
    except (ValueError, OverflowError):
        for i, v in enumerate(values):
            try:
                table([v])
            except (ValueError, OverflowError):
                return None, i
        raise


def makeDB_from_vcf(inVCF, outFile, device=0, chunk_bytes=parsers.VCF_CHUNK_BYTES, timings=None):
    """VCF (plain or .vcf.gz) -> `<outFile>.npz` and `<outFile>.json`, the files vcf_to_csv + makeDB write, without the CSV: the
    host reads (and decompresses) the text after the #CHROM line in chunks of whole lines of at most chunk_bytes
    (64 MB by default), CUDA device `device` turns each chunk's records into rows of the packed panel
    (lib.VcfParser.parse_gt_packed) and the host keeps only those rows, the positions and one chromosome id per record.  The
    arrays of the .npz, the .json and the warning about calls other than 0/0, 1/1, 0/1, ./. equal the CSV route's.  The inputs
    the CSV route fails on raise ValueError naming the line or value, before any file is written: a record whose number of
    sample fields differs from the #CHROM line's, a '#' line after the #CHROM line, a POS that does not read as an integer, a
    CHROM or sample name holding ',' or '"', a non-ASCII sample name, no sample columns, no #CHROM line or a record before it;
    so does a line longer than chunk_bytes.  timings (optional dict) receives seconds of the stages (read_s: read and gunzip,
    device_s with h2d_ms / kernel_ms, host_chunk_s, assemble_s, write_s), h2d_bytes, and under "flagged" the indices of the
    records whose POS text the host converted; a BGZF .vcf.gz is inflated on the device (parsers.BgzfReader) and the route
    goes to timings as parsers._inflate_timings records it.  Returns the open Genotype."""
    import time
    from .. import lib
    chunk_bytes = int(chunk_bytes)
    enc = locale.getpreferredencoding(False)
    tm = timings if timings is not None else {}
    for k in ("read_s", "device_s", "host_chunk_s", "assemble_s", "write_s", "h2d_ms", "kernel_ms", "h2d_bytes"):
        tm[k] = 0
    tm["flagged"] = []
    t0 = time.perf_counter()
    fh = parsers._open_binary(inVCF, device)
    try:
        meta = []
        try:
            names, _, line_no, head = parsers.read_vcf_header(fh, meta_lines=meta)
        except ValueError as e:
            raise ValueError("%s: %s" % (inVCF, e))
        if not names:
            raise ValueError("%s has no sample columns" % inVCF)
        for i, name in enumerate(names):
            if "," in name or '"' in name:
                raise ValueError("sample column %d of %s has the name %r: ',' and '\"' do not fit the CSV" % (i + 1, inVCF, name))
        try:
            accessions = np.array([n.strip() for n in names], dtype="S")
        except UnicodeEncodeError:
            raise ValueError("%s: a sample name is not ASCII, which the database's accession ids must be" % inVCF)
        contigs = get_contigs(meta)
        S = len(names)
        label_of, label_id = {}, {}               # CHROM text -> id of the label the CSV route reads from it; label -> id
        ids, positions, rows = [], [], []
        n_rec, other = 0, 0
        tm["read_s"] += time.perf_counter() - t0
        parser = lib.VcfParser(device, S, chunk_bytes)
        try:
            for chunk, r, line_no in parsers.vcf_chunks(fh, head, chunk_bytes, inVCF, line_no, parser.parse_gt_packed, tm):
                t0 = time.perf_counter()
                if r["non_ascii"]:
                    chunk.decode(enc)                  # the text-mode reader fails on what does not decode
                flags, ls, nsf, clen = r["flags"], r["line_start"], r["nsf"], r["chrom_len"]
                lines = np.flatnonzero(flags & lib.VcfParser.FLAG_RECORD)
                fl = flags[lines]
                refuse = []                           # (line in chunk, message): the first of each kind, the earliest wins
                wrong = lines[nsf[lines] != S]
                if len(wrong):
                    refuse.append((int(wrong[0]), "has %d sample fields, the #CHROM line names %d" % (nsf[wrong[0]], S)))
                text = np.frombuffer(chunk, np.uint8)
                first = ls[:-1]
                hashes = np.flatnonzero((text[first] == 35) & (text[np.minimum(first + 1, len(text) - 1)] != 35))
                if len(hashes):
                    refuse.append((int(hashes[0]), "is a '#' line after the #CHROM line, a second header row of the CSV"))
                # CHROM: read where it may differ from the previous record's, carried forward elsewhere
                new = np.flatnonzero(fl & lib.VcfParser.FLAG_NEW_CHROM)
                raw = [chunk[ls[L]:ls[L] + clen[L]].decode(enc) for L in lines[new].tolist()]
                fresh = []
                for k, c in zip(new.tolist(), raw):
                    if c not in label_of and c not in fresh:
                        if "," in c or '"' in c:
                            refuse.append((int(lines[k]), "has the CHROM %r: ',' and '\"' do not fit the CSV" % c))
                            break
                        fresh.append(c)
                # POS: converted on the host where the device did not read 1-9 plain digits
                fb = np.flatnonzero(fl & lib.VcfParser.FLAG_FALLBACK)
                pos = r["pos"][lines]
                pos_text = []
                for k in fb.tolist():
                    p0 = int(ls[lines[k]] + clen[lines[k]] + 1)
                    v = chunk[p0:chunk.index(b"\t", p0)].decode(enc)
                    if "," in v or '"' in v:
                        refuse.append((int(lines[k]), "has the POS %r: ',' and '\"' do not fit the CSV" % v))
                        break
                    pos_text.append(v)
                if len(pos_text) == len(fb) > 0:
                    conv, bad = _csv_read(pos_text, "POS")
                    if bad is not None:
                        refuse.append((int(lines[fb[bad]]), "has the POS %r, which does not read as an integer" % pos_text[bad]))
                if refuse:
                    L, msg = min(refuse)
                    raise ValueError("%s: line %d %s" % (inVCF, line_no + L + 1, msg))
                if len(fb):
                    pos[fb] = conv
                    tm["flagged"].extend((n_rec + fb).tolist())
                if fresh:
                    for c, lab in zip(fresh, _csv_read(fresh, "CHROM")[0].tolist()):
                        label_of[c] = label_id.setdefault(lab, len(label_id))
                cid = np.zeros(len(lines), np.int32)
                cid[new] = [label_of[c] for c in raw]
                src = np.zeros(len(lines), np.int64)
                src[new] = new
                ids.append(cid[np.maximum.accumulate(src)] if len(lines) else cid)
                positions.append(pos.astype(np.int32))
                rows.append(r["packed"])
                other += r["other_calls"]
                n_rec += len(lines)
                tm["host_chunk_s"] += time.perf_counter() - t0
        finally:
            parser.close()
    finally:
        parsers._inflate_timings(fh, tm)
        fh.close()
    t0 = time.perf_counter()
    ids = np.concatenate(ids) if ids else np.zeros(0, np.int32)
    positions = np.concatenate(positions) if positions else np.zeros(0, np.int32)
    starts, regions = _runs(ids)
    chrs = np.array(list(label_id), dtype="U")[ids[starts]]
    if other:
        log.warning("%s genotype calls are neither 0/0, 1/1, 0/1 nor ./. and were stored as missing", other)
    log.info("Number of contigs found: %s", len(contigs["ref_chrs"]))
    log.info("packing %s SNPs x %s accessions on the GPU", len(positions), S)
    db = lib.Database(positions, regions, S, device=device)
    row0 = 0
    while rows:                                   # each chunk's rows leave host memory once they are on the device
        block = rows.pop(0)
        db.load_packed(block, row0=row0)
        row0 += len(block)
    g = object.__new__(snp_genotype.Genotype)
    g._finish(db, positions, chrs, regions, accessions)
    tm["assemble_s"] += time.perf_counter() - t0
    t0 = time.perf_counter()
    g.save_packed(outFile + ".npz")
    with open(outFile + ".json", "w") as js:
        js.write(json.dumps(contigs, sort_keys=True, indent=4))
    tm["write_s"] += time.perf_counter() - t0
    log.info("wrote %s.npz", outFile)
    return g


def makedb_from_vcf(args):
    _, inType = os.path.splitext(args['inFile'])
    if inType == '.vcf' or len(re.compile(".vcf.gz$").findall(os.path.basename(args['inFile']))) > 0:
        if args.get('no_csv'):
            log.info("VCF -> %s.npz", args['db_id'])
            try:
                makeDB_from_vcf(args['inFile'], args['db_id']).close()
            except ValueError as e:
                die(str(e))
            return
        log.info("VCF -> %s.csv", args['db_id'])
        vcf_to_csv(args['inFile'], args['db_id'])
        makeDB(args['db_id'] + '.csv', args['db_id']).close()
    elif args.get('no_csv'):
        die("--no_csv builds the database from a VCF; %s is not one" % args['inFile'])
    elif inType == '.csv':
        makeDB(args['inFile'], args['db_id']).close()
    else:
        die("please provide either a VCF file or a CSV!")
