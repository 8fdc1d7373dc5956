#!/usr/bin/env python
"""
bench.py — SNP x accession comparisons/s of the genotype-matching hot path (BASELINE.json metric).

Headline workload (config.workload): BASELINE configs[1] — the synthetic 1001-Genomes-shaped panel (1135 accessions x 10.7 M
SNPs, generated in HBM) scored against low-coverage samples with PL weights (~50 k markers each, ~45 k of them in the panel).
One step = one pass of the hot path over one batch of `--samples` independent samples, each scored on its own exactly as
separate `snpmatch inbred` runs would, FROM WHAT A PARSER HANDS OVER: markers in position order as (chromosome, position)
words + integer PLs as weight codes + the table exp(-PL/10).  Everything per marker happens on the device inside the step:
expansion, (chrom, pos) join, compaction, grouping of the matched pairs by weight triple (sort), change masks, counting
kernel, totals, truncation guard, likelihood epilogue.

  value      comparisons/s with the coded batch already resident in HBM (device-timed, CUDA events on the stream the kernels
             run on, max over ranks);
  e2e        the same through the host-buffer API: per step the H2D copy of the coded samples from pinned memory and the D2H
             read of scores / counts / likelihoods are inside the timed region (three batches in a software pipeline);
  e2e_api    (N = 1) `core.batch.genotype_many` on ParseInputs objects: chromosome-name mapping, marker ordering, upload, run,
             fetch, GenotyperOutput construction — the call a user of the Python mirror makes;
  roofline   the scoring kernel k_score_grouped2: SURVEY 8(d) algorithmic bytes per launch / its CUDA-event time;
  cpu_baseline  the CPU oracle (a NumPy restatement of the reference path) on one sample, one core, with `parity`: the
             oracle's integers == the GPU's for that sample (at N > 1: one sample finished by rank 0 and one by the last rank).

Sub-records of the same line: the order-exact fp64 kernel, called genotypes, `cross` (configs[2]), the 20 000-accession panel
(configs[4], STRONG scaling of a fixed batch), the tensor-core batched mode (configs[3]).

N > 1 (torchrun): the panel is sharded by SNP-row ranges, every rank gets the slice of every sample's markers that can match
its rows, per-GPU partial totals are summed with one reduce-scatter, then every rank finishes (truncation guard, epilogue) and
reads back its share of the samples.  The exchange is NCCL's on its own stream, begun after a step's combine and waited for by
that step's epilogue only: two resident batches alternate, so it runs next to the join and grouping kernels of the next step
(every step's work, the last epilogue included, is inside the timed region; `--reduce p2p` is the hand-written one-kernel pull
over peer memory, on the compute stream).  The headline batch grows with N (samples = N x --samples: "scaling": "weak"); the
configs[4] sub-record keeps its batch fixed.  Every rank runs on the host cores next to its GPU.

`--impl reference` times the reference's own CPU path (oracle port; one process per sample on all host cores, the way the
reference is deployed) for the same metric and config.

`--dump-outputs DIR` writes what the headline's last timed step computed, the arrays a caller of the path receives
(Batch.fetch() and the per-sample guard counts), as DIR/<name>.npy in float64; the inputs are a function of the arguments
only, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the benchmark leaves the tree as it found it (no __pycache__ next to the sources)

N_ROWS = 10_700_000
N_ACC = 1135
N_ACC_WIDE = 20_000
N_DB_MARKERS = 45_000
N_EXTRA_MARKERS = 5_000
E2E_DEPTH = 3            # batch objects rotating in the end-to-end arm
METRIC = "snp_accession_comparisons_per_sec"
UNIT = "comparisons/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--samples", type=int, default=64, help="samples per step and per GPU (headline, weak scaling)")
    ap.add_argument("--wide-samples", type=int, default=64, help="samples of the 20 000-accession sub-record (fixed: strong scaling)")
    ap.add_argument("--rows", type=int, default=N_ROWS)
    ap.add_argument("--accessions", type=int, default=N_ACC)
    ap.add_argument("--markers", type=int, default=N_DB_MARKERS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip the sub-records (development runs)")
    ap.add_argument("--group-chunk", type=int, default=320, help="rows per segment of the counting kernel")
    ap.add_argument("--wide-group-chunk", type=int, default=496, help="the same for the 20 000-accession sub-record (the library's choice for wide panels)")
    ap.add_argument("--reduce", default="auto", choices=["auto", "p2p", "nccl", "none"],
                    help="cross-GPU sum of the per-sample totals: p2p = one-shot reduce over peer memory (CUDA IPC over NVLink, flag barrier + "
                         "pulls in one kernel), nccl = NCCL reduce-scatter on its own stream, overlapped with the next step's join and "
                         "grouping kernels, auto = what was measured faster (nccl: 0.558 against 0.589 ms per step with the peer kernel on "
                         "2 GPUs, and NCCL reduces inside the NVSwitch beyond), none = timing experiment only (totals stay per rank)")
    ap.add_argument("--cpu-markers", type=int, default=0, help="bound the CPU sample (0 = one whole sample)")
    ap.add_argument("--no-numa-bind", action="store_true", help="leave the process on whatever cores it was started on (default: the cores next to its GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline's results of its last timed step as DIR/<name>.npy (float64: score, matches, ninfo, m, prob, L, "
                         "LR, guard; sample_index = the samples they belong to, a fixed seeded subset when all would exceed 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 arm")
    if args.reduce == "auto":
        args.reduce = "nccl"
    return args


def workload_config(args, n_gpus, n_samples):
    return {
        "workload": "configs[1]: inbred scoring of %d low-coverage PL samples (~%d markers each, %d in the panel) against the "
                    "synthetic 1001G-shaped panel %d accessions x %d SNPs" % (
                        n_samples, args.markers + N_EXTRA_MARKERS, args.markers, args.accessions, args.rows),
        "panel_rows": args.rows, "accessions": args.accessions, "samples_per_step": n_samples,
        "markers_per_sample": args.markers + N_EXTRA_MARKERS, "weights": "PL (exp(-PL/10), f64)",
        "kernel": "counting kernel k_score_grouped2 on pairs grouped by weight triple ON THE DEVICE (join -> key sort -> change masks -> scoring, every step)",
        "sharding": "single GPU" if n_gpus == 1 else "SNP-row ranges over %d GPUs + one reduce-scatter of the per-accession partials per step (%s; every rank finishes and reads back its share of the samples)" % (
            n_gpus, "one kernel over peer memory: flag barrier + 16-byte pulls through NVLink, no collective library on the path" if args.reduce == "p2p" else "NCCL"),
        "cache": "inputs larger than L2: each step gathers %.0f MB of distinct panel rows" % (
            n_samples * args.markers * ((args.accessions + 63) // 64 * 16) / 1e6),
    }


def make_samples(positions, regions, n_acc, n_samples, n_markers, first_seed=5000):
    from snpmatch_b200 import synth
    out = []
    for i in range(n_samples):
        out.append(synth.make_sample_fast(positions, regions, n_acc, true_acc=(7 + 13 * i) % n_acc, n_db=n_markers,
                                          n_extra=N_EXTRA_MARKERS, seed=first_seed + i))
    return out


# ------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path, one sample
# ------------------------------------------------------------------------------------------------------
def cpu_prepare_sample(sample, n_acc, max_markers=0):
    """Materialise (outside the timed region) the panel rows the sample touches, as the in-RAM int8 matrix the
    reference would read from HDF5."""
    from snpmatch_b200 import synth
    rows = sample["rows"][sample["rows"] >= 0]
    if max_markers and len(rows) > max_markers:
        rows = rows[:max_markers]
    codes = synth.panel_codes(synth.SEED_PANEL, rows, n_acc)
    return rows, codes


def cpu_run_sample(positions, regions, sample, rows, codes):
    """Timed region of the CPU arm: Genotyper.genotyper of the reference (snpmatch.py:207-233) as restated by
    the oracle — the (chrom,pos) join over the database's per-row chromosome labels, then 1000-row chunks of
    matchGTsAccs — plus the likelihood epilogue.  Returns (comparisons, seconds, score, ninfo)."""
    from oracle import snpmatch_oracle as orc
    from snpmatch_b200 import synth
    n_acc = codes.shape[1]
    names = np.array(synth.TAIR10_CHRS)
    s_chrs = np.char.add("Chr", names[sample["chr_ix"]])
    s_pos = sample["pos"].astype(np.int64)
    lookup = np.full(len(positions), -1, dtype=np.int64)
    lookup[rows] = np.arange(len(rows))
    t0 = time.perf_counter()
    labels = orc.db_chromosome_labels(names, regions)                 # pygwas/genotype.py:156-161
    common = orc.get_common_positions(labels, positions, s_chrs, s_pos)
    keep = lookup[common[0]] >= 0                                     # bounded sample: only the materialised rows
    c0, c1 = common[0][keep], common[1][keep]
    score = np.zeros(n_acc)
    ninfo = np.zeros(n_acc, dtype=np.int64)
    for j in range(0, len(c0), 1000):
        t_s, t_n = orc.match_gts_accs(sample["wei"][c1[j:j + 1000]], codes[lookup[c0[j:j + 1000]]])
        score = score + t_s
        ninfo = ninfo + t_n
    with np.errstate(all="ignore"):
        orc.calculate_likelihoods(score.astype(np.int64), ninfo)
    dt = time.perf_counter() - t0
    return len(c0) * n_acc, dt, score, ninfo


def oracle_parity(cpu_score, cpu_ninfo, res, i, exact_score=None, bitwise=True):
    """The bar of tests/test_gpu_coded.py on one sample of a bench run: integers ==, grouped fp64 scores to 1e-12, and the
    order-exact kernel's scores (when given) == on one GPU / to 1e-12 on a sharded panel (per-rank sums added by the reduce:
    the last bits of an fp64 sum depend on that split; the integers do not)."""
    ok = bool(np.array_equal(cpu_score.astype(np.int64), res["matches"][i]) and np.array_equal(cpu_ninfo, res["ninfo"][i]) and
              np.allclose(cpu_score, res["score"][i], rtol=1e-12, atol=0.0))
    if exact_score is not None:
        ok = ok and bool(np.array_equal(cpu_score, exact_score) if bitwise else np.allclose(cpu_score, exact_score, rtol=1e-12, atol=0.0))
    return ok


_W = {}


def _worker(i):
    s = _W["samples"][i]
    comps, dt, _, _ = cpu_run_sample(_W["positions"], _W["regions"], s, *_W["prepared"][i])
    return comps, dt


def _prepare(i):
    return cpu_prepare_sample(_W["samples"][i], _W["n_acc"], _W["cap"])


def run_reference_arm(args):
    """--impl reference: one process per sample on all host cores (README.md:9 deployment model)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    from snpmatch_b200 import synth
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    procs = max(1, min(cores, 32))
    positions, regions = synth.panel_positions(args.rows)
    samples = make_samples(positions, regions, args.accessions, procs, args.markers)
    cap = args.cpu_markers or 0
    ctx = mp.get_context("fork")
    _W.update(positions=positions, regions=regions, samples=samples, n_acc=args.accessions, cap=cap)
    with ctx.Pool(procs) as pool:                       # untimed: materialise the panel rows every sample touches
        prepared = pool.map(_prepare, range(procs))
    _W.update(prepared=prepared)                        # the timed pool below is forked after this, so workers inherit it
    times = []
    comps = 0
    with ctx.Pool(procs) as pool:
        for step in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            res = pool.map(_worker, range(procs))
            dt = time.perf_counter() - t0
            if step >= args.warmup:
                times.append(dt)
                comps = sum(r[0] for r in res)
    total = sum(times)
    value = comps * len(times) / total if total > 0 else 0.0
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / max(len(times), 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, args.gpus, args.samples * args.gpus),      # the b200 arm's workload; a step here is a bounded sample of it
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "port",
                         "sample": "%d samples of that batch per step, one process each (join over the %d database labels + %d-marker "
                                   "chunked matchGTsAccs + likelihoods); NumPy oracle port of snpmatch.py:207-233, database "
                                   "rows held in RAM as int8" % (procs, args.rows, cap or args.markers)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
class ClockSampler(object):
    FIELDS = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(smax)) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class Ctx(object):
    """Process-wide handles of the GPU arm."""
    pass


def pinned(ctx, a):
    t = ctx.torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    ctx.keep.append(t)
    return t.numpy()


def rank_inputs(ctx, samples, positions, regions, r0, r1, hard=False):
    """What this rank uploads: of every sample the slice of its markers that can fall into rows [r0, r1) (position order),
    as pinned arrays — coded (chrom_pos words, PL codes, table) and plain (chromosome ids, positions, f64 weights)."""
    from snpmatch_b200 import lib, sharding, synth
    parts, slices = [], []
    for s in samples:
        i0, i1 = (0, len(s["pos"])) if ctx.world == 1 else sharding.shard_marker_range(s["chr_ix"], s["pos"], regions, positions, r0, r1)
        slices.append((i0, i1))
        parts.append({k: s[k][i0:i1] for k in ("chr_ix", "pos", "wei", "pl", "code")})
    offs = np.concatenate([[0], np.cumsum([len(p["pos"]) for p in parts])]).astype(np.int64)
    chrom = np.concatenate([p["chr_ix"] for p in parts]).astype(np.int32)
    pos = np.concatenate([p["pos"] for p in parts]).astype(np.int32)
    if hard:                                                     # called genotypes: one-hot weights, codes into {0.0, 1.0}
        wei = np.concatenate([synth.hard_weights(p["code"]) for p in parts])
        codes, table = wei.astype(np.uint16), np.array([0.0, 1.0])
    else:                                                        # the parser's integer PLs ARE the codes: no per-marker host work
        wei = np.concatenate([p["wei"] for p in parts]).astype(np.float64)
        pl = np.concatenate([p["pl"] for p in parts])
        codes, table = pl.astype(np.uint16), synth.pl_table(int(pl.max()) if len(pl) else 0)
        assert np.array_equal(table[pl], wei), "exp(-PL/10) table does not reproduce the weights bit for bit"
    cs = lib.code_markers(offs, chrom, pos, codes=codes, wtable=table)
    assert cs is not None
    cs = lib.CodedSamples(pinned(ctx, cs.offsets), pinned(ctx, cs.chrom_pos), pinned(ctx, cs.codes), pinned(ctx, cs.wtable),
                          codes32=pinned(ctx, cs.codes32) if cs.codes32 is not None else None)
    return cs, (pinned(ctx, offs), pinned(ctx, chrom), pinned(ctx, pos), pinned(ctx, wei)), slices


def out_buffers(ctx, S_loc, n_acc, guard_len):
    torch = ctx.torch
    t = {k: torch.empty((S_loc, n_acc), dtype=torch.float64 if k in ("score", "prob", "L", "LR") else torch.int64).pin_memory()
         for k in ("score", "matches", "ninfo", "prob", "L", "LR")}
    t["m"] = torch.empty(S_loc, dtype=torch.int64).pin_memory()
    t["guard"] = torch.zeros(guard_len, dtype=torch.int32).pin_memory()
    ctx.keep.append(t)
    return {k: v.numpy() for k, v in t.items()}


def reduce_totals(ctx, b):
    """Reduce-scatter of the per-sample totals: every rank is left with the totals of its S/world samples and finishes
    (epilogue) and reads back only those.  p2p: one kernel that is barrier + pull over peer memory (k_reduce_peers)."""
    from snpmatch_b200 import sharding
    if ctx.world == 1 or ctx.args.reduce == "none":
        return
    if ctx.args.reduce == "p2p":
        sharding.p2p_reduce_scatter(b)
    else:
        sharding.reduce_scatter_batch(b, ctx.dist, ctx.dev, ctx.rank, ctx.world)


def reduce_begin(ctx, b):
    """First half of reduce_totals: with NCCL the exchange is queued and nothing waits for it yet (sharding.reduce_scatter_begin);
    the peer kernel (one kernel on the compute stream) and the single-GPU case complete here."""
    from snpmatch_b200 import sharding
    if ctx.world > 1 and ctx.args.reduce == "nccl":
        return sharding.reduce_scatter_begin(b, ctx.dist, ctx.dev, ctx.rank, ctx.world)
    reduce_totals(ctx, b)
    return None


def reduce_end(ctx, handle):
    from snpmatch_b200 import sharding
    if handle is not None:
        sharding.reduce_scatter_end(handle)


def run_batch(ctx, b, **kw):
    from snpmatch_b200 import sharding
    if ctx.world > 1 and ctx.args.reduce == "p2p":
        sharding.p2p_before_run(b, ctx.dist, ctx.rank, ctx.world, ctx.host_pg)      # maps the peers' buffers on first use (host collective)
    b.run(**kw)


def barrier(ctx):
    if ctx.world > 1:
        ctx.dist.barrier()
    ctx.torch.cuda.synchronize()


def timed_steps(ctx, step, wait, warmup, steps, flush=None):
    """W untimed + K timed steps on the compute stream: barrier + synchronize on both sides, CUDA events, max over ranks.
    flush: queues whatever a pipelined step leaves for the next one (inside the timed region)."""
    torch = ctx.torch
    for _ in range(warmup):
        step()
    if flush:
        flush()
    wait()
    barrier(ctx)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ctx.stream)
    for _ in range(steps):
        step()
    if flush:
        flush()
    e1.record(ctx.stream)
    wait()
    barrier(ctx)
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=ctx.dev)
    if ctx.world > 1:
        ctx.dist.all_reduce(ms, op=ctx.dist.ReduceOp.MAX)
    return float(ms[0])


def all_max(ctx, vals):
    t = ctx.torch.tensor([float(v) for v in vals], dtype=ctx.torch.float64, device=ctx.dev)
    if ctx.world > 1:
        ctx.dist.all_reduce(t, op=ctx.dist.ReduceOp.MAX)
    return [float(x) for x in t]


def all_sum(ctx, vals):
    t = ctx.torch.tensor([float(v) for v in vals], dtype=ctx.torch.float64, device=ctx.dev)
    if ctx.world > 1:
        ctx.dist.all_reduce(t)
    return [float(x) for x in t]


def last_step_outputs(b):
    """What a caller of the resident path receives from batch `b` after its step: Batch.fetch() and the guard counts."""
    out = b.fetch()
    out["guard"] = b.guard_counts()
    return out


def measure_inbred(ctx, g, samples, positions, regions, r0, r1, n_acc, steps, warmup, chunk, e2e=True, exact=True, hard=False,
                   keep_last=False):
    """Resident and end-to-end arms of inbred scoring of `samples` against this rank's shard.  Returns a dict of numbers plus
    `res`: the last step's results of this rank's share (for the parity checks), and with keep_last `last_step`: the results
    of the last timed step of the resident arm, read from the batch that ran it."""
    from snpmatch_b200 import lib
    torch = ctx.torch
    db = g.db
    world, rank = ctx.world, ctx.rank
    S = len(samples)
    S_loc = S // world
    cs, plain, slices = rank_inputs(ctx, samples, positions, regions, r0, r1, hard=hard)
    h_off, h_chr, h_pos, h_wei = plain
    out = out_buffers(ctx, S_loc, n_acc, S_loc)

    def own_share(b):
        if world > 1:
            b.set_result_range(rank * S_loc, S_loc)
        return b

    gb = lib.Batch(db, h_off, h_chr, h_pos, h_wei)               # position order: also the order-exact kernel's batch
    own_share(gb)
    r = {}
    with torch.cuda.stream(ctx.stream):
        # ---- the order-exact fp64 kernel on the same samples (position order), for comparison and as the bit-exact reference
        if exact:
            def exact_step():
                run_batch(ctx, gb, kernel_mode=lib.KERNEL_POPCOUNT if hard else lib.KERNEL_FP64)
                reduce_totals(ctx, gb)
                gb.epilogue()
            x_steps = max(2, min(steps, 5))
            x_ms = timed_steps(ctx, exact_step, gb.wait, max(1, min(warmup, 2)), x_steps)
            x_kernel = []
            for _ in range(x_steps):
                exact_step()
                x_kernel.append(gb.timings()["score_ms"])
            r["exact_res"] = {k: v.copy() for k, v in gb.fetch().items()}
            r["exact_ms_per_step"] = x_ms / x_steps
            r["exact_kernel_ms"] = float(np.mean(x_kernel))
        # ---- resident arm: the coded samples are on the device; every step does all the per-marker work again
        gb.set_group_chunk(chunk)
        gb.set_track_pairs(False)                                # scores only: the marker indices of the pairs are not read back
        gb.upload_coded(cs)

        def device_step():
            run_batch(ctx, gb, kernel_mode=lib.KERNEL_GROUPED)
            reduce_totals(ctx, gb)
            gb.epilogue()
        if world > 1 and ctx.args.reduce == "nccl":
            # two resident batches alternate: the exchange of step k runs next to the join and grouping kernels of step k + 1,
            # its epilogue follows them.  Every step's work, the last epilogue included, is inside the timed region.
            gb2 = lib.Batch(db, h_off[:2] * 0, h_chr[:0], h_pos[:0], h_wei[:0])
            own_share(gb2)
            gb2.set_group_chunk(chunk)
            gb2.set_track_pairs(False)
            gb2.upload_coded(cs)
            pair, pend, count = [gb, gb2], [None], [0]

            def flush_step():
                if pend[0] is not None:
                    pb, ph = pend[0]
                    reduce_end(ctx, ph)
                    pb.epilogue()
                    pend[0] = None

            def piped_step():
                b_ = pair[count[0] % 2]
                count[0] += 1
                run_batch(ctx, b_, kernel_mode=lib.KERNEL_GROUPED)
                h_ = reduce_begin(ctx, b_)
                flush_step()
                pend[0] = (b_, h_)

            def wait_both():
                gb.wait()
                gb2.wait()
            dev_ms = timed_steps(ctx, piped_step, wait_both, warmup, steps, flush=flush_step)
            if keep_last:
                r["last_step"] = last_step_outputs(pair[(count[0] - 1) % 2])
            gb2.close()
            r["resident_loop"] = "two batches alternate; the NCCL reduce-scatter of a step overlaps the join and grouping kernels of the next"
        else:
            dev_ms = timed_steps(ctx, device_step, gb.wait, warmup, steps)
            if keep_last:
                r["last_step"] = last_step_outputs(gb)
        stage = {}
        for _ in range(steps):                                   # one more pass that reads the library's own events each step
            device_step()
            for k, v in gb.coded_timings().items():
                stage.setdefault(k, []).append(v)
            t = gb.timings()
            stage.setdefault("epilogue_ms", []).append(t["epilogue_ms"])
            launches = t["launches"]
        r.update(dev_ms_per_step=dev_ms / steps, stages_ms={k: float(np.mean(v)) for k, v in stage.items()}, launches=int(launches))
        guard_resident = gb.guard_counts()
        gb.fetch(out={k: out[k] for k in ("score", "matches", "ninfo", "prob", "L", "LR", "m")})
        r["res"] = {k: v.copy() for k, v in out.items()}
        r["res"]["guard"] = guard_resident.copy()
        r["guard_flagged_local"] = int((guard_resident > 0).sum())
        barrier(ctx)
        # ---- end-to-end arm: pinned host buffers in, pinned host buffers out, every step
        if e2e:
            batches = [gb]
            for _ in range(E2E_DEPTH - 1):
                bx = lib.Batch(db, h_off[:2] * 0, h_chr[:0], h_pos[:0], h_wei[:0])
                bx.set_group_chunk(chunk)
                bx.set_track_pairs(False)
                batches.append(bx)
            outs = [out] + [out_buffers(ctx, S_loc, n_acc, S_loc) for _ in range(E2E_DEPTH - 1)]
            host_s = {"upload": 0.0, "launch": 0.0, "wait": 0.0}
            rescored = [0]

            def timed_call(key, fn, *a):
                t_ = time.perf_counter()
                v_ = fn(*a)
                host_s[key] += time.perf_counter() - t_
                return v_

            def up(bt):
                bt.upload_coded(cs)                              # 8 bytes per marker from pinned memory, on the batch's copy stream
                own_share(bt)

            pending = [None]

            def complete_pending():
                if pending[0] is not None:
                    k_, b_, h_ = pending[0]
                    reduce_end(ctx, h_)
                    b_.epilogue()
                    b_.fetch_async(outs[k_ % E2E_DEPTH])         # D2H of step k, queued behind its kernels
                    pending[0] = None

            def launch(k):
                b_ = batches[k % E2E_DEPTH]
                run_batch(ctx, b_, kernel_mode=lib.KERNEL_GROUPED)
                h_ = reduce_begin(ctx, b_)                       # NCCL: runs next to the join / grouping kernels of the step launched next
                complete_pending()                               # the step before this one: its exchange is over by now
                pending[0] = (k, b_, h_)
                if h_ is None:
                    complete_pending()                           # nothing to overlap (one GPU, peer kernel): finish at once

            flagged_all = []

            def finish(k):
                if pending[0] is not None and pending[0][0] == k:
                    complete_pending()
                res = batches[k % E2E_DEPTH].fetch_wait()        # results of step k (this rank's share) are on the host
                fl = np.flatnonzero(res["guard"])                # int(score) needs the reference's summation order (~1e-4 per sample)
                if world == 1:
                    for sidx in fl:
                        lo, hi = int(h_off[sidx]), int(h_off[sidx + 1])
                        one = db.scratch_batch([0, hi - lo], h_chr[lo:hi], h_pos[lo:hi], h_wei[lo:hi])
                        one.run()
                        one.epilogue()
                        r1_ = one.fetch()
                        for key in r1_:
                            res[key][sidx] = r1_[key][0]
                        rescored[0] += 1
                else:
                    flagged_all.extend(int(x) for x in fl)       # re-scoring is a collective job: counted, and reported below
                return res

            def run_pipeline(n):
                """n complete steps, each from the upload of its samples to its results on the host."""
                for key in host_s:
                    host_s[key] = 0.0
                for j in range(min(E2E_DEPTH, n)):
                    timed_call("upload", up, batches[j])
                for j in range(min(E2E_DEPTH - 1, n)):
                    timed_call("launch", launch, j)
                res = None
                for k in range(n):
                    if k + E2E_DEPTH - 1 < n:
                        timed_call("launch", launch, k + E2E_DEPTH - 1)
                    res = timed_call("wait", finish, k)
                    if k + E2E_DEPTH < n:
                        timed_call("upload", up, batches[k % E2E_DEPTH])
                return res

            run_pipeline(max(warmup, E2E_DEPTH))                   # every rotating batch has run once (peer mappings, allocations)
            barrier(ctx)
            rescored[0] = 0
            del flagged_all[:]
            t0 = time.perf_counter()
            run_pipeline(steps)                                  # includes filling the pipeline: the first upload overlaps nothing
            barrier(ctx)
            e2e_s = time.perf_counter() - t0
            e2e_ms = torch.tensor([e2e_s * 1e3], dtype=torch.float64, device=ctx.dev)
            if world > 1:
                ctx.dist.all_reduce(e2e_ms, op=ctx.dist.ReduceOp.MAX)
            try:                                                 # device stage times of the last step, as it ran inside the pipeline
                r["e2e_stages_ms"] = batches[(steps - 1) % E2E_DEPTH].coded_timings()
            except Exception:
                r["e2e_stages_ms"] = None
            r.update(e2e_ms_per_step=float(e2e_ms[0]) / steps, host_ms_per_step={k: 1e3 * v / steps for k, v in host_s.items()},
                     h2d_bytes=int(cs.h2d_bytes), d2h_bytes=int(sum(v.nbytes for v in out.values())),
                     rescored=int(rescored[0]), flagged_e2e=len(flagged_all))
            for bx in batches[1:]:
                bx.close()
    m_tot, flagged = all_sum(ctx, [float(r["res"]["m"].astype(np.int64).sum()), float(r["guard_flagged_local"])])
    r["m_total"] = int(m_tot)
    r["guard_flagged_samples"] = int(flagged)
    r["local_rows"] = int(sum(int(((s["rows"] >= r0) & (s["rows"] < r1)).sum()) for s in samples))
    r["n_weights"] = int(len(cs.wtable))
    r["batch"] = gb
    r["slices"] = slices
    return r


DUMP_BYTES = 64 << 20


def dump_outputs(ctx, res, n_samples, out_dir):
    """--dump-outputs: `res` (this rank's share of the samples, rows rank * S_loc ...) as out_dir/<name>.npy in float64 (the
    counts are exact in it).  All samples, or a fixed seeded subset of them when they would take more than DUMP_BYTES;
    sample_index.npy names the samples either way.  Every rank sends its rows; rank 0 writes."""
    per_sample = 8 * (1 + sum(int(np.prod(v.shape[1:])) for v in res.values()))
    keep = np.arange(n_samples)
    if n_samples * per_sample > DUMP_BYTES:
        if per_sample > DUMP_BYTES:
            raise SystemExit("--dump-outputs: the results of one sample exceed %d bytes" % DUMP_BYTES)
        keep = np.sort(np.random.default_rng(0).choice(n_samples, size=DUMP_BYTES // per_sample, replace=False))
    s_loc = n_samples // ctx.world
    mine = keep[(keep >= ctx.rank * s_loc) & (keep < (ctx.rank + 1) * s_loc)] - ctx.rank * s_loc
    part = {k: v[mine] for k, v in res.items()}
    if ctx.world > 1:
        box = [None] * ctx.world
        ctx.dist.all_gather_object(box, part, group=ctx.host_pg)
        part = {k: np.concatenate([p[k] for p in box]) for k in part}
    if ctx.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        part["sample_index"] = keep
        for k, v in part.items():
            np.save(os.path.join(out_dir, k + ".npy"), v.astype(np.float64))


def gather_last_rank_sample(ctx, res, i_local):
    """Rank 0 receives (matches, ninfo, score) of local sample i_local of the LAST rank (host collective over gloo)."""
    payload = None
    if ctx.rank == ctx.world - 1:
        payload = {k: res[k][i_local].copy() for k in ("matches", "ninfo", "score")}
    box = [None] * ctx.world
    ctx.dist.all_gather_object(box, payload, group=ctx.host_pg)
    return box[ctx.world - 1]


def roofline(peak, algo_bytes, kernel_ms, kernel, extra=None):
    ach = algo_bytes / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else 0.0
    d = {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak if peak else None,
         "algorithmic_bytes_per_launch": int(algo_bytes), "kernel_ms": kernel_ms}
    if extra:
        d.update(extra)
    return d


def measured_traffic(args, world, n_samples):
    """dram bytes of one launch of the dominant kernel from the committed ncu capture; null for any other workload."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as fh:
            t = json.load(fh)
    except Exception:
        return {"traffic": None, "traffic_source": "no capture under profiles/"}
    here = {"n_gpus": world, "panel_rows": args.rows, "accessions": args.accessions, "samples_per_step": n_samples,
            "markers": args.markers, "group_chunk": args.group_chunk}
    if here != t["workload"]:
        return {"traffic": None, "traffic_source": "%s was captured on another workload (%s)" % (t["source"], json.dumps(t["workload"]))}
    return {"traffic": int(t["dram_bytes_read"] + t["dram_bytes_write"]), "traffic_unit": "bytes per launch",
            "traffic_source": t["source"], "traffic_note": t["note"]}


def bind_to_gpu_numa_node(local_rank):
    """Run this rank on the host cores next to its GPU (one process per GPU): pinned buffers allocated afterwards land in that
    NUMA node's memory, so that eight ranks uploading at once do not pull half of their bytes across the socket link.  Returns
    a description for the JSON line; does nothing when the topology cannot be read."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        index = int(vis.split(",")[local_rank]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else local_rank
        hdl = pynvml.nvmlDeviceGetHandleByIndex(index)
        bus = pynvml.nvmlDeviceGetPciInfo(hdl).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(":", 1)
        path = "/sys/bus/pci/devices/%s:%s" % (dom[-4:].lower(), rest.lower())
        with open(path + "/local_cpulist") as fh:
            spec = fh.read().strip()
        with open(path + "/numa_node") as fh:
            node = int(fh.read().strip())
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"bound": False, "why": "no local cores in this process's affinity mask"}
        os.sched_setaffinity(0, cpus)
        return {"bound": True, "numa_node": node, "cores": len(cpus)}
    except Exception as e:  # noqa: BLE001 - the binding is an optimisation
        return {"bound": False, "why": "%s: %s" % (type(e).__name__, e)}


def run_b200_arm(args):
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    numa = bind_to_gpu_numa_node(local_rank) if not args.no_numa_bind else {"bound": False, "why": "--no-numa-bind"}
    import torch
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib, sharding, synth
    from snpmatch_b200.core import snp_genotype

    ctx = Ctx()
    ctx.args, ctx.torch, ctx.keep = args, torch, []
    ctx.rank = rank = int(os.environ.get("RANK", "0"))
    ctx.world = world = int(os.environ.get("WORLD_SIZE", "1"))
    assert lib.device_count() > 0, "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    ctx.dist = ctx.host_pg = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        ctx.dist = dist
        ctx.host_pg = dist.new_group(backend="gloo")     # host-side exchanges must not queue behind kernels
    ctx.dev = torch.device("cuda", local_rank)
    ctx.stream = torch.cuda.Stream(device=ctx.dev)

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peaks = json.load(fh)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_source = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)"

    n_rows, n_acc = args.rows, args.accessions
    S = args.samples * world
    positions, regions = synth.panel_positions(n_rows)
    r0, r1 = sharding.shard_rows(n_rows, world, rank)
    g = snp_genotype.Genotype.synthetic(n_rows, n_acc, row_range=(r0, r1), device=local_rank)
    g.db.set_stream(ctx.stream.cuda_stream)
    samples = make_samples(positions, regions, n_acc, S, args.markers)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    h = measure_inbred(ctx, g, samples, positions, regions, r0, r1, n_acc, args.steps, args.warmup, args.group_chunk,
                       keep_last=bool(args.dump_outputs))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(ctx, h["last_step"], S, args.dump_outputs)
    comps = h["m_total"] * n_acc
    line = None
    if rank == 0:
        value = comps / (h["dev_ms_per_step"] * 1e-3)
        algo_bytes = h["local_rows"] * ((n_acc + 3) // 4 + 24) + 16 * n_acc * S
        k_ms = h["stages_ms"]["score_ms"]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": h["dev_ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, world, S),
            "e2e": {"value": comps / (h["e2e_ms_per_step"] * 1e-3), "unit": UNIT, "ms_per_step": h["e2e_ms_per_step"],
                    "host_ms_per_step": h["host_ms_per_step"],
                    "device_stages_ms_last_step_in_pipeline": h.get("e2e_stages_ms"),
                    "pipeline_fill": "inside the timed region: the first upload and the first step overlap nothing, so the per-step figure "
                                     "falls as --steps grows",
                    "h2d_bytes_per_step": int(world * h["h2d_bytes"]), "d2h_bytes_per_step": int(world * h["d2h_bytes"]),
                    "untimed_per_sample_host_work": "none: the timed region starts from the parser's arrays" if world == 1 else
                                                    "two binary searches per sample and rank (which slice of the sample's position-ordered markers can "
                                                    "fall into the rank's row range), done once when the samples are handed to the ranks; the timed "
                                                    "region starts from those slices",
                    "inputs": "pinned host arrays as a parser hands them over, markers in position order: chromosome id and position in one "
                              "uint32, the three integer PLs of a marker as weight codes in a second uint32 (10 bits each; 8 bytes per marker), + the table exp(-PL/10) "
                              "(%d f64); join, grouping by weight triple and scoring all happen on the device inside the step; three batches rotate "
                              "in a software pipeline (H2D of step k+3 and D2H of step k overlap the kernels of steps k+1 and k+2; filling the "
                              "pipeline is inside the timed region); the D2H holds scores, counts, likelihoods and the per-sample guard "
                              "counts" % h["n_weights"],
                    "samples_rescored_in_reference_order": h["rescored"], "flagged_not_rescored_multi_gpu": h["flagged_e2e"]},
            "gpu_launches": int(h["launches"] * args.steps),
            "roofline": roofline(peak, algo_bytes, k_ms, "k_score_grouped2", {
                **measured_traffic(args, world, S),
                "peak_source": peak_source, "rows_gathered_per_launch": h["local_rows"]}),
            "stages_ms": h["stages_ms"], "distinct_weight_values": h["n_weights"], "group_chunk_rows": int(args.group_chunk),
            "headline_kernel": "k_score_grouped2 (counting kernel, device-grouped pairs)",
            "guard_flagged_samples": h["guard_flagged_samples"], "clocks": clocks, "matched_markers_per_step": h["m_total"],
            "host_numa_binding_rank0": numa,
            "resident_loop": h.get("resident_loop", "one batch; the steps run one after the other"),
        }
        x_ach_bytes = algo_bytes
        line["order_exact_fp64"] = {
            "workload": "same batch in position order, fp64 kernel k_score_segments (sums in the reference's order: fp64 scores bit-identical)",
            "value": comps / (h["exact_ms_per_step"] * 1e-3), "unit": UNIT, "ms_per_step": h["exact_ms_per_step"],
            "roofline": roofline(peak, x_ach_bytes, h["exact_kernel_ms"], "k_score_segments")}
    # ---- grouped vs order-exact on this rank's share, and the CPU oracle ------------------------------------------------
    ok = h["res"]["guard"] == 0
    gve = [float(np.array_equal(h["res"]["matches"][ok], h["exact_res"]["matches"][ok])), float(np.array_equal(h["res"]["ninfo"], h["exact_res"]["ninfo"]))]
    agree = all_sum(ctx, gve)
    rel = float(np.max(np.abs(h["res"]["score"] - h["exact_res"]["score"]) / np.maximum(h["exact_res"]["score"], 1.0))) if len(h["res"]["m"]) else 0.0
    if rank == 0:
        line["order_exact_fp64"]["grouped_vs_exact"] = {"matches_equal_on_all_ranks": agree[0] == world, "ninfo_equal_on_all_ranks": agree[1] == world,
                                                         "score_max_rel_diff_rank0": rel}
    if not args.no_cpu_baseline:
        last = gather_last_rank_sample(ctx, h["res"], len(h["res"]["m"]) - 1) if world > 1 else None
        last_exact = gather_last_rank_sample(ctx, h["exact_res"], len(h["res"]["m"]) - 1) if world > 1 else None
        if rank == 0:
            s0 = samples[0]
            rows, codes = cpu_prepare_sample(s0, n_acc, args.cpu_markers)
            c, dt, cpu_score, cpu_ninfo = cpu_run_sample(positions, regions, s0, rows, codes)
            line["cpu_baseline"] = {"value": c / dt, "unit": UNIT, "cores": 1, "kind": "port", "seconds": dt,
                                    "sample": "sample 0 of the batch (%d matched markers x %d accessions): join over the %d "
                                              "database labels + chunked matchGTsAccs + likelihoods, NumPy oracle port of "
                                              "snpmatch.py:207-233, database rows held in RAM as int8" % (len(rows), n_acc, n_rows)}
            if not args.cpu_markers:
                par = {"sample_0_finished_by_rank_0": oracle_parity(cpu_score, cpu_ninfo, h["res"], 0, h["exact_res"]["score"][0], bitwise=world == 1)}
                if world > 1:
                    sl = samples[S - 1]
                    rows_l, codes_l = cpu_prepare_sample(sl, n_acc, 0)
                    _, _, ls, ln = cpu_run_sample(positions, regions, sl, rows_l, codes_l)
                    par["sample_%d_finished_by_rank_%d" % (S - 1, world - 1)] = oracle_parity(
                        ls, ln, {k: last[k][None] for k in last}, 0, last_exact["score"], bitwise=False)
                line["cpu_baseline"]["parity"] = bool(all(par.values()))
                line["cpu_baseline"]["parity_detail"] = par
                line["cpu_baseline"]["parity_bar"] = "integers (matches = int(score), informative sites) ==; counting-kernel fp64 scores rtol 1e-12; order-exact kernel scores %s" % (
                    "==" if world == 1 else "rtol 1e-12 (sums of per-rank partial sums)")
    h["batch"].close()
    extras = {}
    if not args.headline_only:
        extras["called_genotypes"] = sub_called(ctx, g, samples, positions, regions, r0, r1, n_acc, peak)
        extras["cross"] = sub_cross(ctx, g, positions, regions, r0, r1, n_acc)
        if world == 1:
            extras["e2e_api"] = sub_api(ctx, g, samples, n_acc)
            extras["batched_shared_panel"] = sub_a9(ctx, g, n_rows, n_acc, peaks)
    g.close()
    if not args.headline_only:
        extras["panel_20k"] = sub_wide(ctx, peak, peak_source)
    if rank == 0:
        line.update(extras)
        print(json.dumps(line))
    if world > 1:
        ctx.dist.destroy_process_group()


def sub_called(ctx, g, samples, positions, regions, r0, r1, n_acc, peak):
    """The same samples as called genotypes (0/1 weights, as BED / GT-only VCF inputs give)."""
    args = ctx.args
    steps = max(2, min(args.steps, 5))
    h = measure_inbred(ctx, g, samples, positions, regions, r0, r1, n_acc, steps, max(1, min(args.warmup, 2)), args.group_chunk, e2e=False, hard=True)
    same = all(np.array_equal(h["res"][k], h["exact_res"][k], equal_nan=True) for k in ("score", "matches", "ninfo", "m", "L", "LR"))
    same_all = all_sum(ctx, [float(same)])[0] == ctx.world
    h["batch"].close()
    if ctx.rank != 0:
        return None
    comps = h["m_total"] * n_acc
    h_bytes = h["local_rows"] * ((n_acc + 3) // 4 + 5) + 16 * n_acc * len(samples)
    return {"workload": "same batch with one-hot weights (BED / GT-only VCF inputs): coded path (two weight values), device grouping + counting kernel",
            "value": comps / (h["dev_ms_per_step"] * 1e-3), "unit": UNIT, "ms_per_step": h["dev_ms_per_step"], "stages_ms": h["stages_ms"],
            "roofline": roofline(peak, h_bytes, h["stages_ms"]["score_ms"], "k_score_grouped2"),
            "popcount_kernel": {"kernel": "k_score_hard (position order)", "value": comps / (h["exact_ms_per_step"] * 1e-3),
                                "ms_per_step": h["exact_ms_per_step"], "kernel_ms": h["exact_kernel_ms"],
                                "frac": h_bytes / (h["exact_kernel_ms"] * 1e-3) / 1e9 / peak, "identical_results_on_all_ranks": bool(same_all)}}


def sub_api(ctx, g, samples, n_acc):
    """`core.batch.genotype_many` on ParseInputs objects: the public call, host work included."""
    from snpmatch_b200 import synth
    from snpmatch_b200.core import batch, parsers
    names = np.array(["Chr" + c for c in synth.TAIR10_CHRS])
    inputs = []
    for s in samples:
        inp = parsers.ParseInputs("")
        inp.load_snp_info(names[s["chr_ix"]], s["pos"], synth._gt_strings(s["code"]), s["wei"], s["dp"])
        table = synth.pl_table(int(s["pl"].max()))
        inp._coded = (s["pl"].astype(np.uint16), table, inp.wei)           # what read_vcf keeps for a VCF with integer PLs
        inputs.append(inp)
    ts = []
    res = None
    for _ in range(3):
        t0 = time.perf_counter()
        res = batch.genotype_many(g, inputs)
        ts.append(time.perf_counter() - t0)
    m = sum(r.num_snps for r in res)
    for r in res[:4]:
        r.get_likelihoods()
    ok = all(int(np.nanargmin(r.likelis)) == (7 + 13 * i) % n_acc for i, r in enumerate(res[:4]))
    t = float(np.median(ts))
    return {"call": "core.batch.genotype_many(g, %d ParseInputs)" % len(inputs), "value": m * n_acc / t, "unit": UNIT, "ms_per_call": 1e3 * t,
            "includes": "chromosome-name mapping and marker ordering per sample (host), merging the samples' PL tables, pageable H2D, device join + grouping + "
                        "scoring + epilogue, D2H, re-scoring of flagged samples, GenotyperOutput objects", "true_accessions_recovered": bool(ok)}


def sub_cross(ctx, g, positions, regions, r0, r1, n_acc):
    """configs[2]: `snpmatch cross` device work for one PL sample: 399 windows of 300 kb + the 45 simulated F1s.  On a sharded
    panel every rank scores the windows' rows it holds and ONE all-reduce sums the per-window partials (sharding.py).  Parity:
    every window's informative sites and scores, totals and a sample of the per-window calls against the CPU oracle."""
    from oracle import snpmatch_oracle as orc
    from snpmatch_b200 import lib, sharding, synth
    from snpmatch_b200.core import genomes, snpmatch
    world, rank = ctx.world, ctx.rank
    s = synth.make_sample_fast(positions, regions, n_acc, 7, seed=777)
    gen = genomes.Genome("athaliana_tair10")
    cnt, off, n_w, _ = gen.window_layout(np.array(synth.TAIR10_CHRS), 300000)
    kmax = snpmatch.identity_kmax_table(4000, 0.02)
    i0, i1 = (0, len(s["pos"])) if world == 1 else sharding.shard_marker_range(s["chr_ix"], s["pos"], regions, positions, r0, r1)
    b = lib.Batch(g.db, [0, i1 - i0], s["chr_ix"][i0:i1], s["pos"][i0:i1], s["wei"][i0:i1])
    res = {}

    def run():
        sharding.run_windows_sharded(b, ctx.dist, ctx.dev, False, 300000, cnt, off, n_w, kmax)
        b.epilogue()
        tot = b.fetch()
        res["w"] = b.fetch_window_rows()             # the surviving rows, compacted on the device
        top = np.argsort(-tot["prob"][0])[:10]
        res["f1"] = sharding.f1_pairs_sharded(b, ctx.dist, ctx.dev, top)
        res["tot"] = tot
    with ctx.torch.cuda.stream(ctx.stream):
        for _ in range(2):
            run()
        barrier(ctx)
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            run()
            ts.append(time.perf_counter() - t0)
        tm = b.timings()
        full = b.fetch_windows() if rank == 0 else None
    t = float(np.median(ts))
    t = max(all_max(ctx, [t]))
    m = int(res["w"]["nrows"].sum())
    out = None
    if rank == 0:
        # oracle on the compact panel of the rows the sample touches (same windows, same arithmetic: snpmatch.py / csmatch.py)
        rows = s["rows"][s["rows"] >= 0]
        codes = synth.panel_codes(synth.SEED_PANEL, rows, n_acc)
        row_chr = np.searchsorted(regions[:, 1], rows, side="right")
        creg = np.array([[int((row_chr < c).sum()), int((row_chr <= c).sum())] for c in range(len(regions))], dtype=np.int64)
        names = np.array(synth.TAIR10_CHRS)
        t0 = time.perf_counter()
        o = orc.window_genotyper(codes, names, creg, positions[rows], np.char.add("Chr", names[s["chr_ix"]]), s["pos"].astype(np.int64), s["wei"],
                                 gen.chrs, gen.chrlen, 300000)
        cpu_s = time.perf_counter() - t0
        ok = o.num_snps == m and len(o.windows) == int((full["nrows"] > 0).sum())
        calls_ok = True
        for k, (widx, sc, ni) in enumerate(o.windows):
            ok = ok and np.array_equal(full["ninfo"][widx - 1], ni)
            ok = ok and (np.array_equal(full["score"][widx - 1], sc) if world == 1 else np.allclose(full["score"][widx - 1], sc, rtol=1e-12, atol=0))
            if k % 20 == 0:                          # per-window epilogue on a sample of the windows
                lik, lr, ident, num_amb, keep = orc.window_epilogue(sc, ni)
                calls_ok = calls_ok and np.array_equal(full["identical"][widx - 1], ident.astype(np.uint8)) and int(full["num_amb"][widx - 1]) == num_amb
        ok = ok and np.array_equal(res["tot"]["ninfo"][0], o.tot_ninfo) and np.array_equal(res["tot"]["matches"][0], o.tot_score.astype(np.int64))
        out = {"workload": "configs[2]: cross, %d windows of 300 kb + 45 simulated F1s, one PL sample (%d markers, %d matched) vs %d x %d, %s" % (
                   n_w, len(s["pos"]), m, n_acc, len(positions), "one GPU" if world == 1 else "panel sharded over %d GPUs, one all-reduce of the per-window partials" % world),
               "value": m * n_acc / t, "unit": UNIT, "host_call_ms": 1e3 * t, "device_ms_rank0": tm["total_ms"], "score_kernel_ms_rank0": tm["score_ms"],
               "join_ms_rank0": tm["join_ms"], "windows_with_markers": int((res["w"]["nrows"] > 0).sum()), "surviving_rows": int(len(res["w"]["acc"])),
               "top_accession_is_true": bool(int(np.nanargmin(res["tot"]["L"][0])) == 7),
               "parity": bool(ok and calls_ok), "parity_bar": "every window: informative sites ==, float scores %s; totals ==; identity calls and num_amb of every 20th window ==" % (
                   "==" if world == 1 else "rtol 1e-12 (boundary windows are sums of two ranks)"),
               "cpu_oracle_s": cpu_s}
    b.close()
    return out


def sub_a9(ctx, g, n_rows, n_acc, peaks):
    """configs[3]: batched shared-panel mode, 4096 called-genotype samples on 20 000 shared markers as a one-hot int8 GEMM on
    tcgen05.  The panel operand is expanded once per panel (snpm_panel_create); a call uploads the samples' 2-bit codes from
    pinned memory, expands the sample operand, runs the GEMM and copies the int32 matches / informative sites back."""
    from oracle import snpmatch_oracle as orc
    from snpmatch_b200 import lib, synth
    rng = np.random.default_rng(9)
    S9, K9 = 4096, 20000
    rows9 = np.sort(rng.choice(n_rows, size=K9, replace=False))
    codes9 = rng.choice(np.array([0, 1, 2, 3], dtype=np.uint8), size=(S9, K9), p=[0.6, 0.28, 0.02, 0.1])
    t0 = time.perf_counter()
    sp = g.db.shared_panel(rows9)
    create_ms = 1e3 * (time.perf_counter() - t0)
    packed = pinned(ctx, lib.pack_codes2(codes9))
    out = {"matches": pinned(ctx, np.empty((S9, n_acc), np.int32)), "ninfo": pinned(ctx, np.empty((S9, n_acc), np.int32))}
    g9, dev, exp, call = [], [], [], []
    for i in range(5):
        t0 = time.perf_counter()
        r9 = sp.score(packed, packed=True, out=out)
        if i >= 1:                                   # the first call allocates the panel's scratch
            call.append(time.perf_counter() - t0)
            g9.append(r9["gemm_ms"])
            dev.append(r9["device_ms"])
            exp.append(r9["expand_ms"])
    g9, call, dev, exp = min(g9), float(np.median(call)), float(np.median(dev)), float(np.median(exp))
    # oracle parity on the first and the last sample (matchGTsAccs with one-hot weights, snpmatch.py:74-89)
    panel = synth.panel_codes(synth.SEED_PANEL, rows9, n_acc)
    ok = True
    for smp in (0, S9 - 1):
        have = np.flatnonzero(codes9[smp] < 3)
        sc, ni = orc.match_gts_accs(synth.hard_weights(codes9[smp][have].astype(np.int8)), panel[have], False)
        ok = ok and np.array_equal(r9["matches"][smp], sc.astype(np.int64)) and np.array_equal(r9["ninfo"][smp], ni)
    sp.close()
    ops9 = 2.0 * (2 * S9) * n_acc * (3 * K9)          # SURVEY 8(d): algorithmic int8 ops (the kernel pads A to 1280 and K-slots to 4 per row)
    peak9 = 2.0 * float(peaks.get("bf16_tflops", 1590.0))
    return {"workload": "configs[3]: %d called-genotype samples x %d shared markers vs %d accessions, one-hot int8 GEMM on tcgen05" % (S9, K9, n_acc),
            "value": S9 * K9 * n_acc / (g9 * 1e-3), "unit": UNIT, "gemm_ms": g9, "parity": bool(ok),
            "parity_bar": "samples 0 and %d against the CPU oracle: matches and informative sites ==" % (S9 - 1),
            "e2e": {"value": S9 * K9 * n_acc / call, "unit": UNIT, "host_call_ms": 1e3 * call, "device_ms": dev, "h2d_and_sample_operand_ms": exp,
                    "h2d_bytes": int(packed.nbytes), "d2h_bytes": int(out["matches"].nbytes + out["ninfo"].nbytes),
                    "panel_operand_once_ms": create_ms,
                    "includes": "per call: H2D of the 2-bit packed codes from pinned memory, sample-operand expansion, GEMM, D2H of matches and "
                                "informative sites (int32) into pinned memory; once per panel (panel_operand_once_ms, not in the call): gather + "
                                "one-hot expansion of the %d panel rows" % K9},
            "roofline": {"bound": "tensor", "kernel": "k_onehot_gemm", "achieved": ops9 / (g9 * 1e-3) / 1e12, "peak": peak9, "unit": "TOP/s (int8)",
                         "frac": ops9 / (g9 * 1e-3) / 1e12 / peak9, "scope": "GEMM kernel only (k_onehot_expand_* and the copies are in e2e)",
                         "peak_source": "2 x measured dense bf16 burst TFLOP/s of MEASURED_PEAKS.json (int8 dense is nominally 2x bf16: 4500 vs 2250)"}}


def sub_wide(ctx, peak, peak_source):
    """configs[4]: the 20 000-accession panel (53.6 GB packed), SNP-row sharded over the ranks, a FIXED batch of PL samples
    (strong scaling).  Parity: a bounded sample (3000 matched markers) against the CPU oracle, through the same sharded path."""
    from snpmatch_b200 import lib, sharding, synth
    from snpmatch_b200.core import snp_genotype
    args = ctx.args
    world, rank = ctx.world, ctx.rank
    n_rows, n_acc = args.rows, N_ACC_WIDE
    S = max(world, (args.wide_samples // world) * world)
    positions, regions = synth.panel_positions(n_rows)
    r0, r1 = sharding.shard_rows(n_rows, world, rank)
    g = snp_genotype.Genotype.synthetic(n_rows, n_acc, row_range=(r0, r1), device=ctx.dev.index)
    g.db.set_stream(ctx.stream.cuda_stream)
    samples = make_samples(positions, regions, n_acc, S, args.markers, first_seed=9000)
    steps = max(2, min(args.steps, 5))
    h = measure_inbred(ctx, g, samples, positions, regions, r0, r1, n_acc, steps, max(1, min(args.warmup, 2)), args.wide_group_chunk, e2e=True, exact=False)
    recovered = all(int(np.nanargmin(h["res"]["L"][i])) == (7 + 13 * (rank * (S // world) + i)) % n_acc for i in range(len(h["res"]["m"])))
    recovered = all_sum(ctx, [float(recovered)])[0] == world
    h["batch"].close()
    # bounded parity sample: the first 3000 panel markers of sample 0 (+ its non-panel markers in between), all ranks together
    s0 = samples[0]
    cut = int(np.flatnonzero(s0["rows"] >= 0)[2999]) + 1
    sp = {k: s0[k][:cut] for k in ("chr_ix", "pos", "wei", "pl", "code", "rows")}
    cs, plain, _ = rank_inputs(ctx, [sp] * world, positions, regions, r0, r1)       # `world` copies: the reduce-scatter wants S % world == 0
    pb = lib.Batch(g.db, *plain)
    if world > 1:
        pb.set_result_range(rank, 1)
    pb.set_group_chunk(args.wide_group_chunk)
    pb.upload_coded(cs)
    with ctx.torch.cuda.stream(ctx.stream):
        run_batch(ctx, pb, kernel_mode=lib.KERNEL_GROUPED)
        reduce_totals(ctx, pb)
        pb.epilogue()
        pres = pb.fetch()
    parity = None
    if rank == 0:
        rows, codes = cpu_prepare_sample(sp, n_acc, 0)
        _, _, cs_, cn_ = cpu_run_sample(positions, regions, sp, rows, codes)
        parity = oracle_parity(cs_, cn_, pres, 0)
    pb.close()
    g.close()
    if rank != 0:
        return None
    comps = h["m_total"] * n_acc
    algo_bytes = h["local_rows"] * ((n_acc + 3) // 4 + 24) + 16 * n_acc * S
    return {"workload": "configs[4]: %d PL samples (fixed batch: strong scaling) vs the 20 000-accession x %d panel (%.1f GB packed), SNP-row sharded over %d GPU(s)" % (
                S, n_rows, n_rows * 5008 / 1e9, world),
            "scaling": "strong", "value": comps / (h["dev_ms_per_step"] * 1e-3), "unit": UNIT, "ms_per_step": h["dev_ms_per_step"],
            "e2e": {"value": comps / (h["e2e_ms_per_step"] * 1e-3), "unit": UNIT, "ms_per_step": h["e2e_ms_per_step"],
                    "h2d_bytes_per_step": int(world * h["h2d_bytes"]), "d2h_bytes_per_step": int(world * h["d2h_bytes"])},
            "stages_ms": h["stages_ms"], "roofline": roofline(peak, algo_bytes, h["stages_ms"]["score_ms"], "k_score_grouped2",
                                                               {"peak_source": peak_source, "rows_gathered_per_launch": h["local_rows"]}),
            "true_accessions_recovered_on_all_ranks": bool(recovered), "guard_flagged_samples": h["guard_flagged_samples"],
            "group_chunk_rows": int(args.wide_group_chunk), "parity": parity, "parity_sample": "the first 3000 panel markers of sample 0 (x 20 000 accessions) through the same sharded coded path vs the CPU oracle: "
                                               "integers ==, scores rtol 1e-12"}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
