"""`inbred --samples_vcf` end to end: where the time goes when every sample column of one VCF is parsed on the device
(parsers.read_vcf_many) and scored against the full synthetic panel (1135 accessions x 10.7 M rows, fill_synthetic) by
snpmatch.inbred_identify_many.  Seeded GT:PL VCFs (plain and gz, written to a temporary directory) with S sample columns and
R records at panel positions.  Per file, one JSON line with:
  - host read (+ gzip decompression) seconds, bytes copied up and the device time of the copies and of the parser kernels
    (CUDA events), the host's per-chunk work, the assembly of the S ParseInputs, the many-sample call (which writes every
    sample's files) and the whole run;
  - the baseline: read_vcf_minimal + ParseInputs.read_vcf of one sample column, timed on --baseline_samples columns and
    extrapolated to S (the text-mode reader splits every column of every line to read one);
  - the card name and power limit, read in the same run.
    python scripts/measure_vcf_samples.py [--sizes 64:250000,256:64000,1024:16000] [--out profiles/vcf_samples_measure.jsonl]"""
import argparse
import gzip
import json
import os
import subprocess
import sys
import tempfile
import time

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


def write_vcf(path, positions, regions, chr_names, S, R, seed):
    """R records at sorted random panel rows; cells 'a/b:p0,p1,p2' drawn from 4096 seeded ones (GT 0/0, 0/1, 1/1 or ./., PLs
    0-254), written in blocks."""
    rng = np.random.default_rng(seed)
    rows = np.sort(rng.choice(len(positions), size=R, replace=False))
    chrom = np.searchsorted(regions[:, 1], rows, side="right")
    gts = ["0/0", "0/1", "1/1", "./."]
    vocab = np.array(["%s:%d,%d,%d" % ((gts[k % 4],) + tuple(rng.integers(0, 255, 3))) for k in range(4096)], dtype=object)
    with open(path, "w") as fh:
        fh.write('##fileformat=VCFv4.2\n##INFO=<ID=DP,Number=1,Type=Integer,Description="depth">\n')
        fh.write("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join("s%d" % i for i in range(S)) + "\n")
        for b0 in range(0, R, 4096):
            n = min(4096, R - b0)
            cells = vocab[rng.integers(0, len(vocab), (n, S))].tolist()
            fixed = ["Chr%s\t%d\t.\tA\tT\t.\tPASS\tDP=%d\tGT:PL\t" % (chr_names[c], positions[r], r % 60)
                     for c, r in zip(chrom[b0:b0 + n], rows[b0:b0 + n])]
            fh.write("".join(f + "\t".join(c) + "\n" for f, c in zip(fixed, cells)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="64:250000,256:64000,1024:16000", help="S:R pairs")
    ap.add_argument("--rows", type=int, default=10_700_000)
    ap.add_argument("--acc", type=int, default=1135)
    ap.add_argument("--baseline_samples", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "vcf_samples_measure.jsonl"))
    args = ap.parse_args()
    from snpmatch_b200 import lib, synth
    from snpmatch_b200.core import parsers, snp_genotype, snpmatch
    card = dict(device=lib.device_info(0)["name"], power_limit=power_limit())
    g = snp_genotype.Genotype.synthetic(args.rows, args.acc)
    positions, regions = synth.panel_positions(args.rows)
    chr_names = [str(c).replace("Chr", "") for c in g.chrs]
    lines = []
    with tempfile.TemporaryDirectory() as d:
        for spec in args.sizes.split(","):
            S, R = (int(x) for x in spec.split(":"))
            plain = os.path.join(d, "m%d.vcf" % S)
            t0 = time.perf_counter()
            write_vcf(plain, positions, regions, chr_names, S, R, seed=S)
            gz = plain + ".gz"
            with open(plain, "rb") as src, gzip.open(gz, "wb", compresslevel=1) as dst:
                while True:
                    block = src.read(64 << 20)
                    if not block:
                        break
                    dst.write(block)
            gen_s = time.perf_counter() - t0
            for path in (plain, gz):
                tm = {}
                t0 = time.perf_counter()
                parsed = parsers.read_vcf_many(path, timings=tm)
                parse_s = time.perf_counter() - t0
                out = os.path.join(d, "out")
                os.makedirs(out, exist_ok=True)
                t1 = time.perf_counter()
                snpmatch.inbred_identify_many([p for _, p in parsed], g, [os.path.join(out, n) for n, _ in parsed])
                many_s = time.perf_counter() - t1
                n_markers = int(sum(len(p.pos) for _, p in parsed))
                del parsed
                # baseline: the text-mode reader, one column at a time
                t2 = time.perf_counter()
                for s in range(args.baseline_samples):
                    v = parsers.read_vcf_minimal(path, sample_index=s * (S // max(args.baseline_samples, 1)))
                    parsers.vcf_called_inputs(v["chr"], v["pos"], v["gt"], v.get("wei"), v["dp"])
                base_one = (time.perf_counter() - t2) / args.baseline_samples
                rec = dict(card, S=S, records=R, file=os.path.basename(path), file_bytes=os.path.getsize(path), gen_s=round(gen_s, 2),
                           read_s=round(tm["read_s"], 3), h2d_bytes=int(tm["h2d_bytes"]), h2d_ms=round(tm["h2d_ms"], 2),
                           kernel_ms=round(tm["kernel_ms"], 2), device_call_s=round(tm["device_s"], 3),
                           host_chunk_s=round(tm["host_chunk_s"], 3), assemble_s=round(tm["assemble_s"], 3),
                           read_vcf_many_s=round(parse_s, 3), fallback_records=len(tm["fallback"]), called_markers=n_markers,
                           inbred_identify_many_s=round(many_s, 3), total_s=round(parse_s + many_s, 3),
                           baseline_one_sample_s=round(base_one, 3), baseline_extrapolated_s=round(base_one * S, 1))
                print(json.dumps(rec), flush=True)
                lines.append(rec)
                for f in os.listdir(out):
                    os.remove(os.path.join(out, f))
            os.remove(plain)
            os.remove(gz)
    g.close()
    with open(args.out, "w") as fh:
        fh.write("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
