"""Many-sample `cross` against the sample-by-sample loop on the full synthetic panel (1135 accessions x 10.7 M rows,
fill_synthetic), PL samples from synth.make_sample_fast with varied true accessions and seeds.  For S in --sizes:
  (a) the single-sample device sequence looped over the samples: run_windows -> epilogue -> fetch -> fetch_window_rows ->
      f1_pairs on a one-sample batch;
  (b) the batched sequence on one S-sample batch (one upload, one windows run, one F1 pass);
device ms (CUDA events on the library's stream around the whole sequence), host-call ms (wall clock, every sequence ends in
a synchronise), samples/s, kernel launches per batch, and an exact comparison of (a) and (b) on every sample.  The public call
csmatch.cross_identify_many (pandas tables and files included) is timed on its own, next to CrossIdentifier looped over the
first samples.  A torch.profiler pass of (b) at the largest S gives the kernel busy time and the single-CTA row-offset scan.
Prints one JSON line with the device name and power limit.
    python scripts/measure_cross_many.py [--sizes 1,8,64,256] [--reps 3] [--out cross_many.json]"""
import argparse
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,8,64,256")
    ap.add_argument("--rows", type=int, default=10_700_000)
    ap.add_argument("--accessions", type=int, default=1135)
    ap.add_argument("--markers", type=int, default=45000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--public-single", type=int, default=8, help="samples of the CrossIdentifier loop timed next to the public call")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import __graft_entry__ as ge
    ge.build()
    import torch
    from snpmatch_b200 import lib, synth
    from snpmatch_b200.core import csmatch, genomes, parsers, snp_genotype, snpmatch
    assert lib.device_count() > 0, "measure_cross_many.py needs a CUDA device"
    sizes = [int(x) for x in args.sizes.split(",")]
    S_max = max(sizes)
    name = torch.cuda.get_device_name(0)
    g = snp_genotype.Genotype.synthetic(args.rows, args.accessions, device=0)
    stream = torch.cuda.Stream()
    g.db.set_stream(stream.cuda_stream)
    positions, regions = g.g.positions, g.g.chr_regions
    t0 = time.time()
    ss = [synth.make_sample_fast(positions, regions, args.accessions, (97 * i + 7) % args.accessions, n_db=args.markers,
                                 n_extra=args.markers // 9, seed=7000 + i) for i in range(S_max)]
    gen_s = time.time() - t0
    cnt, off, n_w, _ = genomes.Genome("athaliana_tair10").window_layout(g.g.chrs, 300000)
    binLen = 300000
    n_max = max(int(np.unique(s["chr_ix"].astype(np.int64) * (1 << 32) + (s["pos"].astype(np.int64) - 1) // binLen,
                              return_counts=True)[1].max()) for s in ss)
    kmax = snpmatch.identity_kmax_table(n_max, 0.02)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    one = lib.Batch(g.db, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3)))
    many = lib.Batch(g.db, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3)))

    def loop(sub):
        res, launches = [], 0
        for s in sub:
            one.upload([0, len(s["pos"])], s["chr_ix"], s["pos"], s["wei"])
            one.run_windows(False, binLen, cnt, off, n_w, kmax)
            one.epilogue()
            tot = one.fetch()
            rows = one.fetch_window_rows()
            top = np.argsort(-tot["prob"][0])[0:10]
            f1 = one.f1_pairs(top)
            launches += one.timings()["launches"]
            res.append((tot, rows, f1))
        return res, launches

    def batched(sub):
        offs = np.concatenate([[0], np.cumsum([len(s["pos"]) for s in sub])]).astype(np.int64)
        many.upload(offs, np.concatenate([s["chr_ix"] for s in sub]), np.concatenate([s["pos"] for s in sub]),
                    np.concatenate([s["wei"] for s in sub]))
        many.run_windows(False, binLen, cnt, off, n_w, kmax)
        many.epilogue()
        tot = many.fetch()
        rows = many.fetch_window_rows()
        if len(sub) == 1:
            rows = [rows]
        tops = np.stack([np.argsort(-tot["prob"][i])[0:10] for i in range(len(sub))])
        f1 = many.f1_pairs(tops)
        return (tot, rows, f1, offs), many.timings()["launches"]

    def timed(fn, sub):
        best = None
        with torch.cuda.stream(stream):
            fn(sub)                                               # warm-up: module load, buffers at their final size
            for _ in range(args.reps):
                torch.cuda.synchronize()
                t = time.perf_counter()
                ev0.record(stream)
                out, launches = fn(sub)
                ev1.record(stream)
                ev1.synchronize()
                host = (time.perf_counter() - t) * 1e3
                dev = ev0.elapsed_time(ev1)
                if best is None or host < best[1]:
                    best = (dev, host, out, launches)
        return best

    def agree(a, b):
        loop_res = a
        tot, rows, f1, offs = b
        for i, (t1, r1, f11) in enumerate(loop_res):
            for k in ("score", "matches", "ninfo", "m", "prob", "L", "LR"):
                if not np.array_equal(tot[k][i], t1[k][0], equal_nan=k in ("prob", "L", "LR")):
                    return False
            for k, v in r1.items():
                want = v + offs[i] if k == "matched_s_idx" else v
                if not np.array_equal(rows[i][k], want, equal_nan=(k == "L")):
                    return False
            if not (np.array_equal(f1[0][i], f11[0]) and np.array_equal(f1[1][i], f11[1])):
                return False
        return True

    rows_out = []
    all_agree = True
    for S in sizes:
        sub = ss[:S]
        a_dev, a_host, a_out, a_l = timed(loop, sub)
        b_dev, b_host, b_out, b_l = timed(batched, sub)
        ok = agree(a_out, b_out)
        all_agree &= ok
        rows_out.append({"S": S, "loop_device_ms": round(a_dev, 3), "loop_host_ms": round(a_host, 3),
                         "loop_samples_per_s": round(S / a_host * 1e3, 1), "loop_launches": a_l,
                         "batched_device_ms": round(b_dev, 3), "batched_host_ms": round(b_host, 3),
                         "batched_samples_per_s": round(S / b_host * 1e3, 1), "batched_launches": b_l,
                         "host_speedup": round(a_host / b_host, 2), "exact": bool(ok)})
        print(json.dumps(rows_out[-1]), flush=True)

    # kernel busy time of (b) at the largest S, and the single-CTA scan of the row offsets over S*W windows
    from torch.profiler import ProfilerActivity, profile
    with torch.cuda.stream(stream):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            batched(ss[:S_max])
            torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        if "snpm" in e.key:                                       # the library's kernels (copies and memsets excluded)
            key = e.key.split("(")[0].replace("void ", "")
            kern[key] = kern.get(key, 0.0) + e.device_time_total / 1e3
    busy = sum(kern.values())
    row_off = sum(v for k, v in kern.items() if "k_window_row_offsets" in k)
    prof_rec = {"S": S_max, "kernel_busy_ms": round(busy, 3), "row_offsets_ms": round(row_off, 4),
                "row_offsets_share": round(row_off / busy, 5) if busy else None,
                "top_kernels_ms": {k: round(v, 3) for k, v in sorted(kern.items(), key=lambda kv: -kv[1])[:8]}}
    print(json.dumps(prof_rec), flush=True)

    # the public call: tables and files included
    def inputs(s):
        inp = parsers.ParseInputs("")
        chrs = np.array(["Chr" + synth.TAIR10_CHRS[c] for c in s["chr_ix"]])
        inp.load_snp_info(chrs, s["pos"].astype(np.int64), synth._gt_strings(s["code"]), s["wei"], s["dp"])
        return inp
    public = []
    with tempfile.TemporaryDirectory() as tmp, torch.cuda.stream(stream):
        csmatch.cross_identify_many([inputs(s) for s in ss[:2]], g, "athaliana_tair10", binLen,
                                    [os.path.join(tmp, "w%d" % i) for i in range(2)])
        for S in sizes:
            ins = [inputs(s) for s in ss[:S]]
            t = time.perf_counter()
            csmatch.cross_identify_many(ins, g, "athaliana_tair10", binLen, [os.path.join(tmp, "m%d" % i) for i in range(S)])
            public.append({"S": S, "cross_identify_many_ms": round((time.perf_counter() - t) * 1e3, 1)})
        k = min(args.public_single, S_max)
        ins = [inputs(s) for s in ss[:k]]
        t = time.perf_counter()
        for i, inp in enumerate(ins):
            csmatch.CrossIdentifier(inp, g, "athaliana_tair10", binLen, os.path.join(tmp, "s%d" % i))
        single_ms = (time.perf_counter() - t) * 1e3
    print(json.dumps({"public": public, "crossidentifier_loop": {"S": k, "ms": round(single_ms, 1)}}), flush=True)
    one.close()
    many.close()
    line = {"metric": "cross_many", "device": name, "power_limit": power_limit(), "panel": "%d x %d (fill_synthetic)" % (args.rows, args.accessions),
            "samples": "make_sample_fast, %d panel markers + %d extra each, PL weights" % (args.markers, args.markers // 9),
            "windows_per_sample": int(n_w), "exact_all": bool(all_agree), "rows": rows_out, "profile": prof_rec,
            "public": public, "crossidentifier_loop": {"S": k, "ms": round(single_ms, 1)}, "sample_gen_s": round(gen_s, 1)}
    print(json.dumps(line), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(line) + "\n")
    g.close()
    return 0 if all_agree else 1


if __name__ == "__main__":
    sys.exit(main())
