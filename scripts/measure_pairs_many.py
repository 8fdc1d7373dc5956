"""All-against-all `pairsnp` (core.snpmatch.pairwise_score_many) at user sizes, against the per-pair loops it replaces.

Workload: the full synthetic 1135 x 10.7 M panel as the database; S samples of 50 k markers each, in two regimes:
  targeted  every sample draws from one shared 200 k-row target set (union ~200 k columns, pairs share ~12.5 k markers);
  sparse    every sample draws from the whole panel (union of millions of columns, pairs share ~230 markers).
Reported per (regime, S): the library's device times (operand expansion + memsets, GEMMs, whole call), the GEMMs' int8 op rate
from shapes (2 * 2S * S_pad * slots * K, S_pad = S rounded up to 256), the host seconds of every stage of the call, and two
baselines timed on random pairs and EXTRAPOLATED to S(S-1)/2 pairs: pairwiseScore looped over files (resident database), and
the fairer loop over pre-parsed, database-restricted inputs (get_common_positions + lib.pair_match_counts per pair).
Samples are handed over in memory; parsing is timed on files of a subset and extrapolated (the `parse` row).
The card's name and power limit are read in the same run.  Output: one JSON line per case, and all of them in --out."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

GTS = np.array(["0/0", "1/1", "0/1", "./."])


def card():
    from snpmatch_b200 import lib
    info = lib.device_info(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                      # the figure is recorded as missing, not guessed
        q = "nvidia-smi unavailable: %s" % e
    return {"device": info["name"], "n_sm": info["n_sm"], "nvidia_smi": q}


def make_samples(rng, S, n, regime, positions, chr_of_row, target):
    from snpmatch_b200.core import parsers
    out = []
    for _ in range(S):
        pool = target if regime == "targeted" else None
        if pool is None:
            rows = np.unique(rng.integers(0, len(positions), size=int(n * 1.01)))[:n]
        else:
            rows = np.sort(rng.choice(pool, size=n, replace=False))
        x = parsers.ParseInputs("")
        x.load_snp_info(chr_of_row[rows], positions[rows], GTS[rng.integers(0, 4, size=len(rows))], np.ones((len(rows), 3)), "NA")
        out.append(x)
    return out


def baselines(g, samples, n_pairs, rng, tmp):
    from snpmatch_b200 import lib
    from snpmatch_b200.core import snp_genotype, snpmatch, labels
    S = len(samples)
    pairs = [tuple(rng.choice(S, size=2, replace=False)) for _ in range(n_pairs)]
    files = {}
    for i in sorted({k for p in pairs for k in p}):
        f = os.path.join(tmp, "b%d.npz" % i)
        x = samples[i]
        np.savez(f, chr=x.chrs, pos=x.pos, gt=x.gt, wei=x.wei, dp=np.ones(len(x.pos)))
        files[i] = f
    t0 = time.perf_counter()
    for i, j in pairs:
        snpmatch.pairwiseScore(files[i], files[j], False, hdf5File=g)
    loop = (time.perf_counter() - t0) / n_pairs
    # the fairer loop: every sample parsed and restricted to the database once (not timed), then per pair the join and the
    # device count of pairwiseScore
    used = sorted({k for p in pairs for k in p})
    pre = {}
    for i in used:
        x = samples[i]
        s_idx = np.sort(g.get_positions_idxs(x.chrs, x.pos)[1])
        x.filter_chr_names()
        pre[i] = (x.chrs[s_idx], x.pos[s_idx], x.gt[s_idx].astype("U"))
    t0 = time.perf_counter()
    for i, j in pairs:
        c1, p1, g1 = pre[i]
        c2, p2, g2 = pre[j]
        i1, i2 = snp_genotype.Genotype.get_common_positions(c1, p1, c2, p2)
        ids = labels.factorize(np.concatenate([g1, g2]))[0]
        lib.pair_match_counts(i1, i2, np.zeros(len(c1), np.int32), ids[:len(c1)], ids[len(c1):], 1)
    fair = (time.perf_counter() - t0) / n_pairs
    t0 = time.perf_counter()
    for i in used[:16]:
        from snpmatch_b200.core import parsers
        parsers.ParseInputs(files[i], logDebug=False)
    parse_per_sample = (time.perf_counter() - t0) / min(16, len(used))
    return loop, fair, parse_per_sample


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="64,256,1024,4096")
    ap.add_argument("--regimes", default="targeted,sparse")
    ap.add_argument("--markers", type=int, default=50000)
    ap.add_argument("--rows", type=int, default=10_700_000)
    ap.add_argument("--pairs", type=int, default=20, help="pairs timed for each baseline")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from snpmatch_b200 import synth
    from snpmatch_b200.core import snp_genotype, snpmatch
    info = card()
    print(json.dumps(info), flush=True)
    g = snp_genotype.Genotype.synthetic(a.rows, 1135)
    positions, regions = synth.panel_positions(a.rows)
    chr_of_row = np.repeat(np.char.add("Chr", np.array(synth.TAIR10_CHRS)), np.diff(regions, axis=1).ravel())
    rng = np.random.default_rng(7)
    target = np.sort(rng.choice(a.rows, size=200_000, replace=False))
    # warm-up: module load, torch's CUDA context, the database join
    snpmatch.pairwise_score_many(make_samples(rng, 4, 1000, "targeted", positions, chr_of_row, target), hdf5File=g)
    results = []
    with tempfile.TemporaryDirectory() as tmp:
        for regime in a.regimes.split(","):
            for S in [int(x) for x in a.sizes.split(",")]:
                samples = make_samples(rng, S, a.markers, regime, positions, chr_of_row, target)
                t0 = time.perf_counter()
                pm = snpmatch.pairwise_score_many(samples, hdf5File=g)
                call = time.perf_counter() - t0
                t = pm.timings
                pm.write(os.path.join(tmp, "m"), pairs_json=False)
                slots = 4 if pm.n_classes <= 4 else 8
                s_pad = -(-S // 256) * 256
                ops = 2.0 * (2 * S) * s_pad * slots * pm.n_columns
                loop, fair, parse = baselines(g, samples, a.pairs, rng, tmp)
                n_pairs = S * (S - 1) // 2
                r = {"regime": regime, "S": S, "markers": a.markers, "union_columns": pm.n_columns, "classes": pm.n_classes,
                     "mean_common_pair": float(pm.common.sum(0)[np.triu_indices(S, 1)].mean()) if S > 1 else 0.0,
                     "device_ms": {"expand": t["expand_ms"], "gemm": t["gemm_ms"], "call": t["device_ms"]},
                     "gemm_int8_ops": ops, "gemm_pops": ops / (t["gemm_ms"] * 1e-3) / 1e15 if t["gemm_ms"] > 0 else None,
                     "host_s": {"parse_extrapolated": parse * S, "prepare": t["prepare"], "union_and_db_join": t["union"],
                                "device_call": t["device"], "matrix_build": t["build"], "write": pm.timings["write"],
                                "pairwise_score_many_in_memory": call},
                     "baseline_extrapolated_s": {"pairwiseScore_loop": loop * n_pairs, "preparsed_join_and_count_loop": fair * n_pairs,
                                                 "pairs_timed": a.pairs, "per_pair_s": [loop, fair]},
                     "card": info}
                print(json.dumps(r), flush=True)
                results.append(r)
                del samples, pm
    g.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            for r in results:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
