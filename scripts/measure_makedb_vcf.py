"""`makedb --no_csv` end to end: where the time goes when a strains VCF becomes the packed panel on the device
(makedb.makeDB_from_vcf), against the CSV route (vcf_to_csv + makeDB).  Seeded GT-only VCFs of the synthetic panel (synth.panel_vcf,
1135 accessions, R records), plain and gzip, written to a temporary directory.  Per file, one JSON line with:
  - the stages as makeDB_from_vcf's timings report them: host read (+ gunzip), the device call (with the CUDA-event time of the
    copies up and of the kernels), the host's per-chunk work, the assembly (device panel + load), the writing of .npz / .json;
    the end-to-end seconds, and GB/s of VCF text through the device stage (bytes copied up over h2d + kernel time);
  - the CSV route timed on the first --csv_records records of the same panel and extrapolated to R;
  - the card name and power limit, read in the same run.
A plain file is skipped (and says so) when the temporary directory has no room for it.
    python scripts/measure_makedb_vcf.py [--records 1000000[,4000000]] [--out profiles/makedb_vcf_measure.jsonl]"""
import argparse
import gzip
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return out or None
    except (OSError, subprocess.SubprocessError):
        return None


def device_route(path, out):
    from snpmatch_b200.core import makedb
    tm = {}
    t0 = time.perf_counter()
    makedb.makeDB_from_vcf(path, out, timings=tm).close()
    total = time.perf_counter() - t0
    dev_s = (tm["h2d_ms"] + tm["kernel_ms"]) / 1e3
    return dict(read_s=round(tm["read_s"], 3), device_call_s=round(tm["device_s"], 3), h2d_ms=round(tm["h2d_ms"], 1),
                kernel_ms=round(tm["kernel_ms"], 1), h2d_bytes=int(tm["h2d_bytes"]), host_chunk_s=round(tm["host_chunk_s"], 3),
                assemble_s=round(tm["assemble_s"], 3), write_s=round(tm["write_s"], 3), flagged_records=len(tm["flagged"]),
                total_s=round(total, 3), device_GBps=round(tm["h2d_bytes"] / dev_s / 1e9, 1) if dev_s else None,
                kernel_GBps=round(tm["h2d_bytes"] / (tm["kernel_ms"] / 1e3) / 1e9, 1) if tm["kernel_ms"] else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", default="1000000", help="record counts, comma-separated")
    ap.add_argument("--acc", type=int, default=1135)
    ap.add_argument("--csv_records", type=int, default=50000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "makedb_vcf_measure.jsonl"))
    args = ap.parse_args()
    from snpmatch_b200 import lib, synth
    from snpmatch_b200.core import makedb
    card = dict(device=lib.device_info(0)["name"], power_limit=power_limit())
    A = args.acc
    lines = []
    with tempfile.TemporaryDirectory() as d:
        # the CSV route on a slice: seconds per record
        sl = os.path.join(d, "slice.vcf")
        with open(sl, "wb") as fh:
            synth.panel_vcf(fh, args.csv_records, A)
        t0 = time.perf_counter()
        makedb.vcf_to_csv(sl, os.path.join(d, "slice"))
        t1 = time.perf_counter()
        makedb.makeDB(os.path.join(d, "slice.csv"), os.path.join(d, "slice")).close()
        t2 = time.perf_counter()
        csv_rec_s = (t1 - t0) / args.csv_records, (t2 - t1) / args.csv_records
        csv_bytes = os.path.getsize(os.path.join(d, "slice.csv")) / args.csv_records
        dev = device_route(sl, os.path.join(d, "slice_dev"))
        for ext in ("csv", "npz", "json", "vcf"):
            os.remove(os.path.join(d, "slice." + ext))
        for R in (int(x) for x in args.records.split(",")):
            plain, gz = os.path.join(d, "p%d.vcf" % R), os.path.join(d, "p%d.vcf.gz" % R)
            need = R * (4 * A + 40) * 1.1
            room = shutil.disk_usage(d).free
            t0 = time.perf_counter()
            if room > need:
                with open(plain, "wb") as fh:
                    synth.panel_vcf(fh, R, A)
                with open(plain, "rb") as src, gzip.open(gz, "wb", compresslevel=1) as dst:
                    shutil.copyfileobj(src, dst, 64 << 20)
            else:
                with gzip.open(gz, "wb", compresslevel=1) as dst:
                    synth.panel_vcf(dst, R, A)
            gen_s = time.perf_counter() - t0
            for path in (plain, gz):
                base = dict(card, accessions=A, records=R, file=os.path.basename(path), gen_s=round(gen_s, 1))
                if not os.path.exists(path):
                    rec = dict(base, skipped="not measured: %d bytes free, %d needed" % (room, need))
                else:
                    rec = dict(base, file_bytes=os.path.getsize(path), **device_route(path, os.path.join(d, "out")))
                    rec.update(csv_route_extrapolated_s=dict(vcf_to_csv=round(csv_rec_s[0] * R, 1), makeDB=round(csv_rec_s[1] * R, 1)),
                               csv_bytes_extrapolated=int(csv_bytes * R), csv_slice_records=args.csv_records,
                               slice_device_route_s=dev["total_s"])
                    for ext in ("npz", "json"):
                        os.remove(os.path.join(d, "out." + ext))
                    os.remove(path)
                print(json.dumps(rec), flush=True)
                lines.append(rec)
    with open(args.out, "w") as fh:
        fh.write("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
