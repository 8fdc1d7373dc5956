"""`genotype_cross --gpu_parse` end to end: where the time goes when a population VCF's genotype columns are parsed on the device
(parsers.read_vcf_gt_codes) before the window calls, against the text route (read_vcf_samples + parseGT).  A seeded GT-only VCF
of the synthetic panel (synth.panel_vcf: R records x S samples at the panel's positions), plain and gzip, written to a temporary
directory; the parents are two accessions of the same synthetic panel (synth.small_panel, same positions).  Per file, one JSON
line with:
  - read_vcf_gt_codes by stage, as its timings report them: host read (+ gunzip), the device call (with the CUDA-event time of
    the copies up and of the kernels), the host's per-chunk work, the assembly; GB/s of VCF text through the kernels;
  - genotype_cross(..., gpu_parse=True) plus the writing of the output file, end to end, in a run of its own;
  - the card name and power limit, read in the same run.
Then one line for the text route, which cannot hold R x S in memory: both routes on the first --prefix records of the same file,
their output files compared byte for byte, and the text route's seconds extrapolated to R records (labelled as such).
    python scripts/measure_genotype_cross_vcf.py [--records 1000000] [--samples 384] [--out profiles/genotype_cross_vcf_measure.jsonl]"""
import argparse
import filecmp
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


def read_stages(path):
    from snpmatch_b200.core import parsers
    tm = {}
    t0 = time.perf_counter()
    r = parsers.read_vcf_gt_codes(path, timings=tm)
    total = time.perf_counter() - t0
    return dict(read_s=round(tm["read_s"], 3), device_call_s=round(tm["device_s"], 3), h2d_ms=round(tm["h2d_ms"], 1),
                kernel_ms=round(tm["kernel_ms"], 1), h2d_bytes=int(tm["h2d_bytes"]), host_chunk_s=round(tm["host_chunk_s"], 3),
                assemble_s=round(tm["assemble_s"], 3), reader_total_s=round(total, 3),
                kernel_GBps=round(tm["h2d_bytes"] / (tm["kernel_ms"] / 1e3) / 1e9, 1) if tm["kernel_ms"] else None,
                codes_shape=list(r["gt_codes"].shape))


def end_to_end(x, path, out, gpu_parse):
    t0 = time.perf_counter()
    lines = x.genotype_cross(path, 1.5, gpu_parse=gpu_parse)
    t1 = time.perf_counter()
    x.write_output_genotype_cross(lines, out)
    t2 = time.perf_counter()
    return dict(genotype_cross_s=round(t1 - t0, 3), write_s=round(t2 - t1, 3), total_s=round(t2 - t0, 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=1000000)
    ap.add_argument("--samples", type=int, default=384)
    ap.add_argument("--prefix", type=int, default=20000)
    ap.add_argument("--bin_len", type=int, default=200000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "genotype_cross_vcf_measure.jsonl"))
    args = ap.parse_args()
    import logging
    logging.disable(logging.INFO)
    from snpmatch_b200 import lib, synth
    from snpmatch_b200.core import genotype_cross as gc, snp_genotype
    card = dict(device=lib.device_info(0)["name"], power_limit=power_limit())
    R, S = args.records, args.samples
    p = synth.small_panel(n_rows=R, n_acc=8)
    g = snp_genotype.Genotype.from_arrays(p["snps"], p["positions"], p["chrs"], p["chr_regions"], p["accessions"])
    parents = "%sx%s" % (p["accessions"][0].decode(), p["accessions"][1].decode())
    x = gc.GenotypeCross(g, parents, args.bin_len, None, False, genome_id="athaliana_tair10")
    lines = []
    with tempfile.TemporaryDirectory() as d:
        plain, gz = os.path.join(d, "pop.vcf"), os.path.join(d, "pop.vcf.gz")
        t0 = time.perf_counter()
        with open(plain, "wb") as fh:
            synth.panel_vcf(fh, R, S)
        with open(plain, "rb") as src, gzip.open(gz, "wb", compresslevel=1) as dst:
            shutil.copyfileobj(src, dst, 64 << 20)
        gen_s = time.perf_counter() - t0
        # the first --prefix records, for the text route
        pre = os.path.join(d, "prefix.vcf")
        with open(plain, "rb") as src, open(pre, "wb") as dst:
            n_rec = 0
            for line in src:
                dst.write(line)
                if not line.startswith(b"#"):
                    n_rec += 1
                    if n_rec == args.prefix:
                        break
        for path in (plain, gz):
            base = dict(card, samples=S, records=R, segregating_markers=len(x.commonSNPsPOS), bin_len=args.bin_len,
                        file=os.path.basename(path), file_bytes=os.path.getsize(path), gen_s=round(gen_s, 1))
            rec = dict(base, **read_stages(path))
            rec["end_to_end"] = end_to_end(x, path, os.path.join(d, "out.csv"), True)
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        dev = end_to_end(x, pre, os.path.join(d, "prefix_dev.csv"), True)
        txt = end_to_end(x, pre, os.path.join(d, "prefix_txt.csv"), False)
        same = filecmp.cmp(os.path.join(d, "prefix_dev.csv"), os.path.join(d, "prefix_txt.csv"), shallow=False)
        rec = dict(card, samples=S, prefix_records=args.prefix, file="prefix of " + os.path.basename(plain),
                   file_bytes=os.path.getsize(pre), device_route=dev, text_route=txt, output_files_equal=same,
                   text_route_extrapolated_to_records=R, text_route_extrapolated_s=round(txt["total_s"] * R / args.prefix, 1),
                   note="text_route_extrapolated_s is extrapolated linearly from the prefix, not measured")
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    g.close()
    with open(args.out, "w") as fh:
        fh.write("".join(json.dumps(r) + "\n" for r in lines))
    if not same:
        sys.exit("the two routes wrote different files on the prefix")


if __name__ == "__main__":
    main()
