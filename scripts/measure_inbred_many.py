"""Many-sample `inbred` against the sample-by-sample loop on the full synthetic panel (1135 accessions x 10.7 M rows,
fill_synthetic), 50 k-marker PL samples from synth.make_sample_fast with varied true accessions.  For S in --sizes:
  (a) public calls: Genotyper (+ filter_tophits with --refine) looped over the samples against snpmatch.inbred_identify_many,
      without and with refine: host-call ms (wall clock; both end in a synchronise), the device event span on the library's
      stream, and `==` on every file of every sample;
  (b) the refine stage on its own, through snpmatch._refine_scores (what the public call runs), with top-hit sets of 2, 4 and
      16 accessions (the synthetic panel's accessions are independent, so its samples rarely refine): the single path's
      per-sample full-panel scan (identify_segregating_snps: scan, 10.7 MB read-back, flatnonzero) plus the filtered join
      and scoring, against one batch with the pair filter; results compared with `==`;
  (c) a torch.profiler pass of (b) at the largest S: k_segregating_pairs device time and the bytes it moves (one 32-byte
      sector per touched word and matched marker, plus match_row), next to k_segregating_rows of the single path;
  (d) host waits of one inbred_identify_many launch, counted per synchronising library call.
Prints one JSON line with the device name and power limit.
    python scripts/measure_inbred_many.py [--sizes 1,8,64,256] [--out inbred_many.json]"""
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


def same_files(a, b, exts=(".scores.txt", ".matches.json", ".refined.scores.txt")):
    for ext in exts:
        if os.path.exists(a + ext) != os.path.exists(b + ext):
            return False
        if os.path.exists(a + ext) and open(a + ext, "rb").read() != open(b + ext, "rb").read():
            return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,8,64,256")
    ap.add_argument("--rows", type=int, default=10_700_000)
    ap.add_argument("--accessions", type=int, default=1135)
    ap.add_argument("--markers", type=int, default=45000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import __graft_entry__ as ge
    ge.build()
    import torch
    from snpmatch_b200 import lib, synth
    from snpmatch_b200.core import parsers, snp_genotype, snpmatch
    assert lib.device_count() > 0, "measure_inbred_many.py needs a CUDA device"
    sizes = [int(x) for x in args.sizes.split(",")]
    S_max = max(sizes)
    A = args.accessions
    name = torch.cuda.get_device_name(0)
    g = snp_genotype.Genotype.synthetic(args.rows, A, device=0)
    stream = torch.cuda.Stream()
    g.db.set_stream(stream.cuda_stream)
    positions, regions = g.g.positions, g.g.chr_regions
    t0 = time.time()
    ss = [synth.make_sample_fast(positions, regions, A, (97 * i + 7) % A, n_db=args.markers, n_extra=args.markers // 9,
                                 seed=7000 + i) for i in range(S_max)]
    gen_s = time.time() - t0

    def inputs(s):
        inp = parsers.ParseInputs("")
        chrs = np.array(["Chr" + synth.TAIR10_CHRS[c] for c in s["chr_ix"]])
        inp.load_snp_info(chrs, s["pos"].astype(np.int64), synth._gt_strings(s["code"]), s["wei"], s["dp"])
        return inp
    ins = [inputs(s) for s in ss]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def span(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        ev0.record(stream)
        out = fn()
        ev1.record(stream)
        ev1.synchronize()
        return out, (time.perf_counter() - t) * 1e3, ev0.elapsed_time(ev1)

    # ---- (a) public calls ----------------------------------------------------------------------------------------------
    public, all_equal = [], True
    with tempfile.TemporaryDirectory() as tmp, torch.cuda.stream(stream):
        snpmatch.inbred_identify_many(ins[:2], g, [os.path.join(tmp, "w%d" % i) for i in range(2)], refine=True)    # warm-up
        snpmatch.Genotyper(ins[0], g, os.path.join(tmp, "w")).filter_tophits()
        for refine in (False, True):
            for S in sizes:
                def loop():
                    for i in range(S):
                        gt = snpmatch.Genotyper(ins[i], g, os.path.join(tmp, "l%d" % i), run_genotyper=not refine)
                        if refine:
                            gt.filter_tophits()
                _, l_host, l_dev = span(loop)
                gts, b_host, b_dev = span(lambda: snpmatch.inbred_identify_many(ins[:S], g, [os.path.join(tmp, "b%d" % i) for i in range(S)],
                                                                                refine=refine))
                eq = all(same_files(os.path.join(tmp, "l%d" % i), os.path.join(tmp, "b%d" % i)) for i in range(S))
                all_equal &= eq
                public.append({"S": S, "refine": refine, "loop_host_ms": round(l_host, 1), "loop_device_span_ms": round(l_dev, 2),
                               "batched_host_ms": round(b_host, 1), "batched_device_span_ms": round(b_dev, 2),
                               "host_speedup": round(l_host / b_host, 2), "refined_samples": sum(hasattr(x, "result_fine") for x in gts),
                               "files_equal": bool(eq)})
                print(json.dumps(public[-1]), flush=True)
                for f in os.listdir(tmp):
                    os.remove(os.path.join(tmp, f))

    # ---- (b) the refine stage on its own -------------------------------------------------------------------------------
    rng = np.random.default_rng(11)
    prepared = [g.prepare_markers(inp.chrs, inp.pos) for inp in ins]
    single = lib.Batch(g.db, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3)))
    many = lib.Batch(g.db, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 3)))
    stage = []

    def single_refine(sub, tops):
        out = []
        for i, top in zip(sub, tops):
            seg = snpmatch.identify_segregating_snps(g, top)
            order, cid, pos = prepared[i]
            single.upload([0, len(pos)], cid, pos, np.asarray(ins[i].wei, dtype=np.float64)[order])
            single.set_row_filter(seg)
            single.run(False)
            single.epilogue()
            out.append(single.fetch())
        single.set_row_filter(None)
        return out

    def batched_refine(sub, tops):
        return snpmatch._refine_scores(g, many, [ins[i] for i in sub], [prepared[i] for i in sub], tops, False)

    with torch.cuda.stream(stream):
        for k in (2, 4, 16):
            for S in sizes:
                sub = list(range(S))
                tops = [np.sort(rng.choice(A, size=k, replace=False)) for _ in sub]
                single_refine(sub[:1], tops[:1])
                batched_refine(sub, tops)
                best = {}
                for _ in range(args.reps):
                    a, a_host, a_dev = span(lambda: single_refine(sub, tops))
                    b, b_host, b_dev = span(lambda: batched_refine(sub, tops))
                    if "a" not in best or a_host < best["a"][0]:
                        best["a"] = (a_host, a_dev)
                    if "b" not in best or b_host < best["b"][0]:
                        best["b"] = (b_host, b_dev)
                eq = all(np.array_equal(b[key][j], a[j][key][0]) for j in range(S) for key in ("score", "ninfo", "m"))
                all_equal &= eq
                stage.append({"top_hits": k, "S": S, "scan_loop_host_ms": round(best["a"][0], 2), "scan_loop_device_span_ms": round(best["a"][1], 2),
                              "pair_filter_host_ms": round(best["b"][0], 2), "pair_filter_device_span_ms": round(best["b"][1], 2),
                              "host_speedup": round(best["a"][0] / best["b"][0], 1), "refined_pairs": int(np.sum(b["m"])), "equal": bool(eq)})
                print(json.dumps(stage[-1]), flush=True)

        # ---- (c) the pair filter in the profiler -----------------------------------------------------------------------
        from torch.profiler import ProfilerActivity, profile
        sub = list(range(S_max))
        tops = [np.sort(rng.choice(A, size=16, replace=False)) for _ in sub]
        offs = np.concatenate([[0], np.cumsum([len(prepared[i][2]) for i in sub])]).astype(np.int64)
        many.upload(offs, np.concatenate([prepared[i][1] for i in sub]), np.concatenate([prepared[i][2] for i in sub]),
                    np.concatenate([np.asarray(ins[i].wei, dtype=np.float64)[prepared[i][0]] for i in sub]))
        many.run(False)
        many.epilogue()
        matched = many.fetch()["m"]                                # pairs before the filter
        batched_refine(sub, tops)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            batched_refine(sub, tops)
            single_refine(sub[:8], tops[:8])
            torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        if "k_segregating" in e.key or "k_join" in e.key:
            key = e.key.split("(")[0].replace("void ", "").replace("snpm::", "")
            kern[key] = (kern.get(key, (0.0, 0))[0] + e.device_time_total / 1e3, kern.get(key, (0.0, 0))[1] + e.count)
    words = [len(np.unique(t >> 5)) for t in tops]
    n_up = int(offs[-1])
    bytes_moved = int(sum(int(m) * w * 32 for m, w in zip(matched, words)) + n_up * 8 + S_max * 8)
    pairs_ms = kern.get("k_segregating_pairs", (0.0, 0))[0]
    rows_ms, rows_n = kern.get("k_segregating_rows", (0.0, 0))
    prof_rec = {"S": S_max, "top_hits": 16, "markers": n_up, "matched_pairs": int(np.sum(matched)),
                "k_segregating_pairs_ms": round(pairs_ms, 4), "k_segregating_pairs_bytes": bytes_moved,
                "k_segregating_pairs_GBps": round(bytes_moved / (pairs_ms * 1e6), 1) if pairs_ms else None,
                "k_segregating_rows_ms_per_sample": round(rows_ms / max(rows_n, 1), 4),
                "k_segregating_rows_bytes_per_sample": int(args.rows) * g.db.row_words * 8,
                "kernels_ms": {k: round(v[0], 4) for k, v in kern.items()}}
    print(json.dumps(prof_rec), flush=True)

    # ---- (d) host waits of one launch --------------------------------------------------------------------------------
    waits = {}
    patched = [(lib.Batch, n) for n in ("fetch", "count_flagged_pairs", "guard_counts", "set_segregation_filter", "fetch_pairs", "set_row_filter")]
    patched += [(lib, "calculate_likelihoods"), (lib, "calculate_likelihoods_many"), (lib.Database, "segregating_rows"), (lib.Database, "intersect")]
    saved = []
    for obj, n in patched:
        fn = getattr(obj, n)
        saved.append((obj, n, fn))

        def counted(*a, _fn=fn, _n=n, **k):
            waits[_n] = waits.get(_n, 0) + 1
            return _fn(*a, **k)
        setattr(obj, n, counted)
    S_w = min(64, S_max)
    tops_w = {}
    with tempfile.TemporaryDirectory() as tmp, torch.cuda.stream(stream):
        gts = snpmatch.inbred_identify_many(ins[:S_w], g, [os.path.join(tmp, "c%d" % i) for i in range(S_w)], refine=True)
        tops_w = sum(hasattr(x, "result_fine") for x in gts)
    for obj, n, fn in saved:
        setattr(obj, n, fn)
    wait_rec = {"S": S_w, "launches": 1, "refined_samples": int(tops_w), "waits_by_call": waits, "waits_total": int(sum(waits.values()))}
    print(json.dumps(wait_rec), flush=True)

    single.close()
    many.close()
    line = {"metric": "inbred_many", "device": name, "power_limit": power_limit(), "panel": "%d x %d (fill_synthetic)" % (args.rows, A),
            "samples": "make_sample_fast, %d panel markers + %d extra each, PL weights" % (args.markers, args.markers // 9),
            "equal_all": bool(all_equal), "public": public, "refine_stage": stage, "pair_filter_profile": prof_rec, "waits": wait_rec,
            "sample_gen_s": round(gen_s, 1)}
    print(json.dumps(line), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(line) + "\n")
    g.close()
    return 0 if all_equal else 1


if __name__ == "__main__":
    sys.exit(main())
