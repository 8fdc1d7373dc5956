"""BGZF `.vcf.gz` inflated on the device (parsers.BgzfReader, k_bgzf_inflate) against the host's gunzip, for the three device VCF
readers.  Seeded GT-only VCFs, each written as BGZF (synth.write_bgzf, level 6 as bgzip writes it, members compressed in host
threads) and as single-member gzip at level 6, in a temporary directory:
  - makedb: synth.panel_vcf, --acc accessions x --records records, through makedb.makeDB_from_vcf;
  - genotype_cross: synth.panel_vcf, --samples samples x --records records, through parsers.read_vcf_gt_codes;
  - read_vcf_many: synth.population_vcf, --many_samples samples x --many_records records.
Per reader and file, one JSON line with the stages its timings report (host read, with the device inflate calls inside it:
inflate_s, and their CUDA-event times inflate_h2d_ms, inflate_ms, d2h_ms; the parser's device call; the host's per-chunk work;
the assembly), GB/s of text out of k_bgzf_inflate, the end-to-end seconds, and whether the outputs of the two files are equal.
Also: the member scanner on this file and on a file of 700 k members; makeDB_from_vcf at batches of 64 / 256 / 512 MB of text, alternating, three runs of each; and, for context
only, zlib over the same members in os.cpu_count() host threads.  Every line carries the card name and power limit.
    python scripts/measure_bgzf.py [--records 1000000] [--out profiles/bgzf_measure.jsonl]"""
import argparse
import concurrent.futures as cf
import gzip
import json
import mmap
import os
import shutil
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return out or None
    except (OSError, subprocess.SubprocessError):
        return None


def write_both(plain, gz_bgzf, gz_single, piece=64 << 20):
    """plain -> BGZF (pieces compressed in threads, concatenated) and single-member gzip, both at level 6; seconds."""
    from snpmatch_b200 import synth
    t0 = time.perf_counter()
    d = os.path.dirname(plain)
    with open(plain, "rb") as src:
        texts = iter(lambda: src.read(piece), b"")

        def one(k_t):
            k, t = k_t
            p = os.path.join(d, "piece%06d.gz" % k)
            synth.write_bgzf(p, t, level=6, eof=False)
            return p
        with cf.ThreadPoolExecutor(os.cpu_count()) as ex, open(gz_bgzf, "wb") as dst:
            for p in ex.map(one, enumerate(texts)):
                with open(p, "rb") as fh:
                    shutil.copyfileobj(fh, dst, 64 << 20)
                os.remove(p)
            dst.write(synth.BGZF_EOF)
    t1 = time.perf_counter()
    with open(plain, "rb") as src, gzip.open(gz_single, "wb", compresslevel=6) as dst:
        shutil.copyfileobj(src, dst, 64 << 20)
    return round(t1 - t0, 1), round(time.perf_counter() - t1, 1)


def stages(tm, total):
    keys = ("read_s", "inflate_s", "device_s", "host_chunk_s", "assemble_s", "write_s")
    out = {k: round(tm[k], 3) for k in keys if k in tm}
    for k in ("inflate_h2d_ms", "inflate_ms", "d2h_ms", "h2d_ms", "kernel_ms"):
        if k in tm:
            out[k] = round(tm[k], 1)
    out.update(inflate=tm.get("inflate"), gz_bytes=tm.get("gz_bytes"), text_bytes=int(tm["h2d_bytes"]), total_s=round(total, 3))
    if tm.get("inflate_ms"):
        out["inflate_GBps_text_out"] = round(tm["h2d_bytes"] / (tm["inflate_ms"] / 1e3) / 1e9, 1)
    return out


def scan_s(path):
    from snpmatch_b200 import lib
    with open(path, "rb") as f:
        mm = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)
    t0 = time.perf_counter()
    off, _ = lib.bgzf_scan(np.frombuffer(mm, np.uint8))
    s = time.perf_counter() - t0
    n = len(off) - 1
    del off
    mm.close()
    return n, round(s, 4)


def host_threads_s(path):
    """zlib over every member in os.cpu_count() threads (context only): seconds."""
    from snpmatch_b200 import lib
    raw = open(path, "rb").read()
    off, _ = lib.bgzf_scan(np.frombuffer(raw, np.uint8))
    off = off.tolist()

    def one(k):
        a, b = off[k], off[k + 1]
        x = raw[a + 10] | raw[a + 11] << 8
        return len(zlib.decompress(raw[a + 12 + x:b - 8], -15))
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(os.cpu_count()) as ex:
        n = sum(ex.map(one, range(len(off) - 1), chunksize=256))
    return n, round(time.perf_counter() - t0, 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=1000000)
    ap.add_argument("--acc", type=int, default=1135)
    ap.add_argument("--samples", type=int, default=384)
    ap.add_argument("--many_samples", type=int, default=256)
    ap.add_argument("--many_records", type=int, default=200000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bgzf_measure.jsonl"))
    args = ap.parse_args()
    from snpmatch_b200 import lib, synth
    from snpmatch_b200.core import makedb, parsers
    card = dict(device=lib.device_info(0)["name"], power_limit=power_limit(), cpus=os.cpu_count())
    lines = []

    def emit(rec):
        rec = dict(card, **rec)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    with tempfile.TemporaryDirectory() as d:
        # the scanner on 700 k members: tiny members of 100 bytes of text
        tiny = os.path.join(d, "tiny.gz")
        synth.write_bgzf(tiny, b"x" * (700000 * 100), member_bytes=100)
        n, s = scan_s(tiny)
        emit(dict(what="scanner", members=n, scan_s=s))
        os.remove(tiny)
        R = args.records
        for work in ("makedb", "genotype_cross", "read_vcf_many"):
            plain, bg, single = (os.path.join(d, work + x) for x in (".vcf", ".bgzf.vcf.gz", ".single.vcf.gz"))
            t0 = time.perf_counter()
            with open(plain, "wb") as fh:
                if work == "makedb":
                    synth.panel_vcf(fh, R, args.acc)
                elif work == "genotype_cross":
                    synth.panel_vcf(fh, R, args.samples)
                else:
                    pos, regions = synth.panel_positions(args.many_records)
                    chrom = np.array(synth.TAIR10_CHRS)[np.searchsorted(regions[:, 1], np.arange(args.many_records), side="right")]
                    synth.population_vcf(fh, chrom, pos, args.many_samples, seed=5, edge_forms=False)
            gen_s = round(time.perf_counter() - t0, 1)
            bgzf_s, single_s = write_both(plain, bg, single)
            n, s = scan_s(bg)
            base = dict(what=work, gen_s=gen_s, write_bgzf_s=bgzf_s, write_gzip_s=single_s, text_bytes=os.path.getsize(plain),
                        bgzf_bytes=os.path.getsize(bg), gzip_bytes=os.path.getsize(single), members=n, scan_s=s)
            os.remove(plain)
            results = {}
            for path, route in ((single, "host"), (bg, "device"), (single, "host"), (bg, "device")):   # each twice, alternating
                tm = {}
                t0 = time.perf_counter()
                if work == "makedb":
                    out = os.path.join(d, "db_" + route)
                    makedb.makeDB_from_vcf(path, out, timings=tm).close()
                    z = np.load(out + ".npz")
                    res = {k: z[k] for k in z.files}
                    res["json"] = open(out + ".json").read()
                elif work == "genotype_cross":
                    res = parsers.read_vcf_gt_codes(path, timings=tm)
                else:
                    res = parsers.read_vcf_many(path, timings=tm)
                total = time.perf_counter() - t0
                assert tm["inflate"] == route, (tm["inflate"], route)
                results[route] = res
                emit(dict(base, route=route, file=os.path.basename(path), **stages(tm, total),
                          **({"batch_bytes": parsers.BGZF_BATCH_BYTES} if route == "device" else {})))
            a, b = results["host"], results["device"]
            if work == "read_vcf_many":
                same = [n for n, _ in a] == [n for n, _ in b] and all(
                    all(np.array_equal(getattr(x, k), getattr(y, k)) for k in ("chrs", "pos", "gt", "wei", "dp")) for (_, x), (_, y) in zip(a, b))
            else:
                same = sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) if k != "json" else a[k] == b[k] for k in a)
            emit(dict(what=work, outputs_equal=bool(same)))
            del results, a, b
            if work == "makedb":
                default_batch = parsers.BGZF_BATCH_BYTES
                for batch in (64 << 20, 256 << 20, 512 << 20) * 3:          # alternating, three runs of each size
                    parsers.BGZF_BATCH_BYTES = batch
                    tm = {}
                    t0 = time.perf_counter()
                    makedb.makeDB_from_vcf(bg, os.path.join(d, "db_b"), timings=tm).close()
                    emit(dict(what="makedb_batch", batch_bytes=batch, **stages(tm, time.perf_counter() - t0)))
                parsers.BGZF_BATCH_BYTES = default_batch
            n, s = host_threads_s(bg)
            emit(dict(what=work + "_zlib_host_threads", threads=os.cpu_count(), text_bytes=n, seconds=s, note="context only, not shipped"))
            for p in (bg, single):
                os.remove(p)
    with open(args.out, "w") as fh:
        fh.write("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
