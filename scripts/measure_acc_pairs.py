"""Accession against accession (`pairsnp --accessions`, lib.Database.acc_pairs) at the sizes users run, against NumPy.

Cases (synthetic panels generated in HBM, every accession selected, calls as they are and with --skip_db_hets):
  1135 accessions x 10.7 M rows   the full panel: one output block, 18 x 5 = 90 GEMM tiles per chunk
  20 000 accessions x --rows20k   three output blocks of 8192, six block pairs, 3.2 GB of int32 output
Reported per case: the library's device times (operand expansion, GEMMs, whole call with the copies of the two [n,n] outputs
to the host), the GEMMs' int8 operations as executed (padded tiles, 2 * 128 * 256 * 128 per tile and k-block) and their
rate, the algorithmic pair-row comparisons n(n-1)/2 * rows per second of the whole call, and a NumPy baseline (float64
BLAS products of the called and one-hot matrices) timed on a row subset and EXTRAPOLATED linearly to all rows.
The median of --reps calls is kept after one warm-up call.  The card's name and power limit are read in the same run.
Output: one JSON line per case on stdout, and all of them in --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    from snpmatch_b200 import lib
    info = lib.device_info(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                      # the figure is recorded as missing, not guessed
        q = "nvidia-smi unavailable: %s" % e
    return {"device": info["name"], "n_sm": info["n_sm"], "nvidia_smi": q}


def executed_ops(n, rows, block=8192, chunk_bytes=1 << 30):
    """int8 operations the GEMMs execute (tiles padded to 64 x 256 accessions, k-blocks to 32 rows), over the block pairs
    bi <= bj, with the library's default chunking (SNPM_PAIR_CHUNK_BYTES of operand tiles per chunk)."""
    kb_bytes = -(-n // 64) * 128 * 128 + -(-n // 256) * 256 * 128
    step = max(1, chunk_bytes // kb_bytes) * 32
    kbs = sum(-(-min(step, rows - r0) // 32) for r0 in range(0, rows, step))
    sizes = [min(block, n - b0) for b0 in range(0, n, block)]
    tiles = sum(-(-sizes[i] // 64) * -(-sizes[j] // 256) for i in range(len(sizes)) for j in range(i, len(sizes)))
    return 2.0 * 128 * 256 * 128 * tiles * kbs, tiles


def numpy_seconds(snps, skip_hets):
    """The oracle of tests/test_gpu_acc_pairs.py on int8 rows [r, n]: both counts of every pair."""
    t0 = time.perf_counter()
    called = (snps >= 0) & (snps <= (1 if skip_hets else 2))
    P = called.astype(np.float64)
    P.T @ P
    for c in range(3):
        H = (called & (snps == c)).astype(np.float64)
        H.T @ H
    return time.perf_counter() - t0


def run_case(n, rows, np_rows, reps, info):
    from snpmatch_b200.core import snp_genotype
    g = snp_genotype.Genotype.synthetic(rows, n)
    out = []
    try:
        g.db.acc_pairs(np.arange(min(n, 300)))                         # warm-up: module load, GEMM attributes
        sub = g.db.read_rows(np.arange(min(np_rows, rows)))
        ops, tiles = executed_ops(n, rows)
        pair_rows = n * (n - 1) / 2.0 * rows
        for skip in (False, True):
            calls = []
            for _ in range(reps):
                t0 = time.perf_counter()
                common, same, ms = g.db.acc_pairs(skip_db_hets=skip)
                calls.append((time.perf_counter() - t0, ms))
                del common, same
            calls.sort(key=lambda c: c[1][2])
            wall, ms = calls[len(calls) // 2]
            np_s = numpy_seconds(sub, skip)
            r = {"accessions": n, "rows": rows, "skip_db_hets": skip, "reps": reps, "gemm_tiles_per_chunk": tiles,
                 "device_ms": {"expand": ms[0], "gemm": ms[1], "call": ms[2]},
                 "host_call_s": wall,
                 "gemm_int8_ops_executed": ops, "gemm_pops": ops / (ms[1] * 1e-3) / 1e15 if ms[1] > 0 else None,
                 "pair_rows": pair_rows, "pair_rows_per_s_call": pair_rows / (ms[2] * 1e-3),
                 "numpy_baseline": {"rows_timed": int(len(sub)), "seconds_timed": np_s,
                                    "seconds_extrapolated": np_s * rows / len(sub)},
                 "card": info}
            print(json.dumps(r), flush=True)
            out.append(r)
    finally:
        g.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows1135", type=int, default=10_700_000)
    ap.add_argument("--rows20k", type=int, default=200_000)
    ap.add_argument("--np_rows1135", type=int, default=50_000)
    ap.add_argument("--np_rows20k", type=int, default=500)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    info = card()
    print(json.dumps(info), flush=True)
    results = run_case(1135, a.rows1135, a.np_rows1135, a.reps, info)
    results += run_case(20000, a.rows20k, a.np_rows20k, a.reps, info)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            for r in results:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
