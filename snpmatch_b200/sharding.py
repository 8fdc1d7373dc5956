"""
SNP-row sharding of the panel over the GPUs of one box (SURVEY.md section 8e).

The database is cut into contiguous row ranges, one per rank (boundaries ignore chromosomes:
low-coverage markers are spread evenly over the genome, so matched rows balance).  Samples are
replicated.  Every rank joins and scores against its own rows; the per-sample partial totals
(score f64, ninfo, matched pairs) travel in ONE buffer and are summed with one all-reduce, after
which every rank runs the likelihood epilogue on identical totals.

This module is the host logic of that scheme and is independent of CUDA, so that it can be tested
with the gloo backend on CPU; `bench.py` and `allreduce_batch` below use it with NCCL on the
device buffer of a `lib.Batch`.
"""
import numpy as np


def shard_rows(n_rows, world, rank):
    """Contiguous row range [r0, r1) of `rank`."""
    return rank * n_rows // world, (rank + 1) * n_rows // world


def local_regions(chr_regions, r0, r1):
    """Chromosome row ranges clipped to a shard and shifted to shard-local row numbers; chromosomes
    outside the shard become empty ranges (the join then finds nothing there)."""
    reg = np.asarray(chr_regions, dtype=np.int64).reshape(-1, 2)
    return np.clip(reg, r0, r1) - r0


def shard_marker_range(chr_ix, pos, chr_regions, positions, r0, r1):
    """Slice [i0, i1) of a sample's markers (sorted by (database chromosome index, position)) that can match
    rows [r0, r1) of the panel: only that slice has to be uploaded to the rank holding the shard, which keeps
    per-GPU join work and H2D traffic constant as ranks are added.  Markers of unknown chromosomes (index < 0)
    never match and are left out."""
    chr_ix = np.asarray(chr_ix)
    pos = np.asarray(pos)
    if r1 <= r0 or len(pos) == 0:
        return 0, 0
    reg = np.asarray(chr_regions, dtype=np.int64).reshape(-1, 2)
    c_lo = int(np.searchsorted(reg[:, 1], r0, side="right"))
    c_hi = int(np.searchsorted(reg[:, 1], r1 - 1, side="right"))
    key = chr_ix.astype(np.int64) * (1 << 32) + pos.astype(np.int64)
    known = chr_ix >= 0
    assert np.all(np.diff(key[known]) > 0), "markers must be sorted by (chromosome index, position)"
    lo = c_lo * (1 << 32) + int(positions[r0])
    hi = c_hi * (1 << 32) + int(positions[r1 - 1])
    first_unknown = int(np.argmax(~known)) if (~known).any() else len(key)
    assert known[:first_unknown].all() and not known[first_unknown:].any(), "unknown chromosomes must come last"
    k = key[:first_unknown]
    return int(np.searchsorted(k, lo, side="left")), int(np.searchsorted(k, hi, side="right"))


def reduce_row_len(n_acc):
    """f64 per sample in the reduce buffer: score[n_acc] | ninfo[n_acc] | matched pairs | y>n count."""
    return 2 * n_acc + 2


def pack_reduce_rows(score, ninfo, m):
    """Host-side picture of the device reduce buffer (csrc/score.cuh k_combine): integers are stored as
    f64, exact below 2**53, so that one sum collective carries everything."""
    score = np.atleast_2d(np.asarray(score, dtype=np.float64))
    ninfo = np.atleast_2d(np.asarray(ninfo))
    S, A = score.shape
    out = np.zeros((S, reduce_row_len(A)), dtype=np.float64)
    out[:, :A] = score
    out[:, A:2 * A] = ninfo
    out[:, 2 * A] = np.asarray(m).reshape(S)
    return out


def unpack_reduce_rows(buf, n_acc):
    buf = np.asarray(buf, dtype=np.float64).reshape(-1, reduce_row_len(n_acc))
    return buf[:, :n_acc], buf[:, n_acc:2 * n_acc].astype(np.int64), buf[:, 2 * n_acc].astype(np.int64)


def truncation_guard(score, rel_eps=1e-12):
    """Accessions whose int(score) could depend on the summation order: a sharded run adds the chunk
    partials in another order than the single-GPU reference, which moves the fp64 sum by a few ulp;
    only sums within that distance of an integer can truncate differently (SURVEY section 7, hard part 1).
    Returns a boolean mask (True = ambiguous, must be re-scored in reference order)."""
    s = np.asarray(score, dtype=np.float64)
    frac = s - np.floor(s)
    tol = np.maximum(np.abs(s), 1.0) * rel_eps
    near_int = (frac < tol) | (1.0 - frac < tol)
    exact_int = s == np.floor(s)
    # sums of 0/1 weights are exact integers in every order: not ambiguous
    return near_int & ~exact_int


def allreduce_batch(batch, dist, device):
    """Sum the per-sample partial totals of a lib.Batch over all ranks, in place on the device buffer
    (NCCL; the buffer is wrapped zero-copy through __cuda_array_interface__)."""
    import torch

    class _Dev(object):
        pass

    ptr, n = batch.reduce_buffer()
    holder = _Dev()
    holder.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}
    t = torch.as_tensor(holder, device=device)
    dist.all_reduce(t)
    return t


# ---- grouped counting kernel (csrc/grouped.cuh): the score travels as an exact integer part I and a fractional part F ----
def grouped_row_len(n_acc):
    """f64 per sample in the reduce buffer of a grouped batch: F[n_acc] | ninfo[n_acc] | matched pairs | overflow flag (the y>n
    count after the epilogue) | I[n_acc]."""
    return 3 * n_acc + 2


def grouped_partials(wei, codes, skip_db_hets=False):
    """Host picture of what k_score_grouped + k_combine_grouped leave for one sample on one shard.
    wei f64 [k,3] in the reference's column order (ref, het, alt; parsers.py:89-94), codes int8 [k,A] (-1/0/1/2).
    Returns (F f64[A], I int64[A], ninfo int64[A]): matches of weights that are exactly 1.0 are counted in I, every other
    weight is summed in F (any order: the device sums group by group)."""
    wei = np.asarray(wei, dtype=np.float64).reshape(-1, 3)
    codes = np.asarray(codes)
    if skip_db_hets:
        codes = np.where(codes == 2, -1, codes)
    A = codes.shape[1] if codes.ndim == 2 else 0
    F = np.zeros(A)
    I = np.zeros(A, dtype=np.int64)
    for col, code in ((0, 0), (1, 2), (2, 1)):            # weight column -> database code (snpmatch.py:81-87)
        hit = codes == code
        w = wei[:, col]
        one = w == 1.0
        I += hit[one].sum(axis=0)
        F += (hit[~one] * w[~one, None]).sum(axis=0)
    return F, I, (codes >= 0).sum(axis=0).astype(np.int64)


def pack_grouped_rows(F, ninfo, m, I, overflow=0):
    """overflow: per sample, 1 when this shard's device grouping ran out of dense ids (csrc/group_sort.cuh), else 0."""
    F = np.atleast_2d(np.asarray(F, dtype=np.float64))
    S, A = F.shape
    out = np.zeros((S, grouped_row_len(A)), dtype=np.float64)
    out[:, :A] = F
    out[:, A:2 * A] = np.atleast_2d(ninfo)
    out[:, 2 * A] = np.asarray(m).reshape(S)
    out[:, 2 * A + 1] = np.broadcast_to(np.asarray(overflow, dtype=np.float64), (S,))
    out[:, 2 * A + 2:] = np.atleast_2d(I)
    return out


def finalize_grouped(buf, n_acc):
    """NumPy restatement of k_grouped_finalize on (all-reduced) totals: returns (score f64[S,A], matches int64[S,A],
    ninfo int64[S,A], m int64[S], guard bool[S,A]).  matches = I + floor(F): the reference's fp64 sum is >= I (monotone
    rounding of non-negative terms) and < I + F + eps, so its truncation can only differ where F lies within the summation
    error bound of an integer k >= 1 — those cells are flagged for re-scoring in reference order.  A sample whose summed overflow
    slot is > 0 (some shard folded its weight triples together) is unreliable as a whole: all its cells are flagged."""
    buf = np.asarray(buf, dtype=np.float64).reshape(-1, grouped_row_len(n_acc))
    F, ninfo, m, I = buf[:, :n_acc], buf[:, n_acc:2 * n_acc], buf[:, 2 * n_acc], buf[:, 2 * n_acc + 2:]
    depth = 1010.0 + m[:, None] / 500.0
    g = 4.0 * depth * 1.1102230246251565e-16 * (I + F + 1.0)
    k = np.rint(F)
    guard = ((k >= 1.0) & (np.abs(F - k) <= g)) | (buf[:, 2 * n_acc + 1] > 0.0)[:, None]
    want = I + np.floor(F)
    v = I + F
    bump = np.floor(v) != want
    v = np.where(bump, np.nextafter(want + 1.0, 0.0), v)
    return v, want.astype(np.int64), ninfo.astype(np.int64), m.astype(np.int64), guard


def reduce_scatter_batch(batch, dist, device, rank, world):
    """Sum the per-sample partial totals of a lib.Batch over all ranks and leave every rank with ITS share of the samples
    (rows [rank*S/world, (rank+1)*S/world) of the device buffer): half the bytes of an all-reduce on the wire, and the
    epilogue / read-back of a rank shrink to S/world samples (lib.Batch.set_result_range).  S must be a multiple of world."""
    import torch

    class _Dev(object):
        pass

    ptr, n = batch.reduce_buffer()
    assert n % world == 0 and batch.n_samples % world == 0, "samples must divide evenly over the ranks"
    holder = _Dev()
    holder.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}
    t = torch.as_tensor(holder, device=device)
    out = getattr(batch, "_rs_out", None)
    if out is None or out.numel() != n // world:
        out = torch.empty(n // world, dtype=torch.float64, device=device)
        batch._rs_out = out
    dist.reduce_scatter_tensor(out, t)
    t.view(world, -1)[rank].copy_(out)
    return out


def reduce_scatter_begin(batch, dist, device, rank, world):
    """reduce_scatter_batch in two halves, so that the exchange of step k runs next to the join and grouping kernels of step
    k + 1 (they are latency bound and leave most SMs idle): this queues the NCCL reduce-scatter behind the kernels already on
    the current stream and returns at once; nothing later on the current stream waits for it until reduce_scatter_end.  The
    batch's reduce buffer must not be written (no run of the same batch) in between."""
    import torch

    class _Dev(object):
        pass

    ptr, n = batch.reduce_buffer()
    assert n % world == 0 and batch.n_samples % world == 0, "samples must divide evenly over the ranks"
    holder = _Dev()
    holder.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}
    t = torch.as_tensor(holder, device=device)
    out = getattr(batch, "_rs_out", None)
    if out is None or out.numel() != n // world:
        out = torch.empty(n // world, dtype=torch.float64, device=device)
        batch._rs_out = out
    work = dist.reduce_scatter_tensor(out, t, async_op=True)
    return work, out, t.view(world, -1)[rank]


def reduce_scatter_end(handle):
    """The current stream waits for the exchange begun by reduce_scatter_begin and copies this rank's share of the sums into
    the batch's buffer (the epilogue may follow)."""
    work, out, mine = handle
    work.wait()
    mine.copy_(out)


# ---- one-shot reduce over peer memory (csrc/grouped.cuh: k_reduce_peers) ------------------------------------------------
# The same reduce-scatter as reduce_scatter_batch with no collective library on the path: every rank maps the reduce buffers of
# all ranks (CUDA IPC over NVLink / NVSwitch) and ONE kernel per step does the cross-rank barrier (step-counter flags in peer
# memory) and pulls + sums the rows of this rank's samples.  torch.distributed is used once, to exchange the 64-byte handles.
def p2p_before_run(batch, dist, rank, world, host_group=None):
    """Call before batch.run() on every rank at the same point: (re)maps the peers' reduce buffers when this batch has not been
    set up yet or its buffer changed (another sample count or row layout).  The set-up is a host collective."""
    import torch

    st = getattr(batch, "_p2p", None)
    if st is None:
        st = batch._p2p = {"key": None}
    key = batch.reduce_buffer()                    # (device pointer, doubles): allocates for the current samples and row layout
    if st["key"] != key:
        torch.cuda.current_stream().synchronize()
        seen = [None] * world
        dist.all_gather_object(seen, key[1], group=host_group)      # nobody is still using the old mapping; sizes agree
        assert len(set(seen)) == 1, "every rank must hold the same samples (reduce buffers of %s doubles)" % seen
        handle = batch.ipc_export()                # may move the buffer (IPC wants its own mapping): export before the run
        handles = [None] * world
        dist.all_gather_object(handles, handle, group=host_group)
        batch.ipc_open(handles, rank)
        st["key"] = batch.reduce_buffer()


def p2p_reduce_scatter(batch):
    """After batch.run() on every rank: rows [rank*S/world, (rank+1)*S/world) of this rank's reduce buffer become the sums
    over all ranks (lib.Batch.set_result_range must select that share).  One kernel, stream-ordered; the host does not wait."""
    batch.reduce_peers()


# ---- `cross` on a sharded panel (SURVEY 8e; csmatch.py:64-129) --------------------------------------------------------------
def device_view(ptr, n, device):
    """Zero-copy torch view of n f64 at a device pointer of the library."""
    import torch

    class _Dev(object):
        pass

    holder = _Dev()
    holder.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}
    return torch.as_tensor(holder, device=device)


def run_windows_sharded(batch, dist, device, skip_db_hets, bin_len, win_count, win_off, n_windows, kmax, lr_thres=3.841):
    """CrossIdentifier.window_genotyper (csmatch.py:64-104) over a panel sharded by SNP-row ranges: every rank scores the
    windows' rows it holds, ONE all-reduce sums the per-window partials (score, informative sites, rows: a window lies in one
    shard except at the shard boundaries), then every rank runs totals, per-window likelihoods, identity calls and the
    compaction on identical sums.  `batch` holds this rank's slice of the sample's markers (position order)."""
    ptr, n = batch.run_windows_begin(skip_db_hets, bin_len, win_count, win_off, n_windows, kmax, lr_thres)
    if dist is not None and dist.get_world_size() > 1:
        dist.all_reduce(device_view(ptr, n, device))
    batch.run_windows_finish()


def f1_pairs_sharded(batch, dist, device, acc_idx):
    """match_insilico_f1s (csmatch.py:106-129) over a sharded panel: partial (score, numinfo) of the 45 pairs per rank, summed."""
    import torch
    score, ninfo = batch.f1_pairs(acc_idx)
    if dist is not None and dist.get_world_size() > 1:
        t = torch.tensor(np.concatenate([score, ninfo.astype(np.float64)]), dtype=torch.float64, device=device)
        dist.all_reduce(t)
        v = t.cpu().numpy()
        score, ninfo = v[:len(score)], v[len(score):].astype(np.int64)
    return score, ninfo


def window_partials_host(win_score, win_ninfo, win_nrows):
    """Host picture of the packed buffer of snpm_batch_run_windows_begin (csrc/windows.cuh k_window_pack) for a_pad == n_acc:
    score [W*A] | ninfo as f64 [W*A] | rows as f64 [W] — used by the gloo test of the layout."""
    s = np.asarray(win_score, dtype=np.float64)
    return np.concatenate([s.ravel(), np.asarray(win_ninfo, dtype=np.float64).ravel(), np.asarray(win_nrows, dtype=np.float64).ravel()])


def unpack_window_partials(buf, n_windows, n_acc):
    buf = np.asarray(buf, dtype=np.float64)
    cells = n_windows * n_acc
    return (buf[:cells].reshape(n_windows, n_acc), buf[cells:2 * cells].astype(np.int64).reshape(n_windows, n_acc),
            buf[2 * cells:2 * cells + n_windows].astype(np.int64))
