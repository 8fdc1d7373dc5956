"""Host-side resources of the library: a destroyed batch gives back all of its device memory, the window buffers of a sharded
`cross` run included, and the asynchronous fetch reports the same device-counted errors as the synchronous one."""
import ctypes
import os

import numpy as np
import pytest

from snpmatch_b200 import synth

N_ACC = 1135          # 36-word rows: the packed window partials of 200 windows take (2 * 200 * 36 * 32 + 200) doubles, 3.7 MB
BIN_LEN = 600000      # 200 windows on the TAIR10 chromosomes
CYCLES = 20


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from snpmatch_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


@pytest.fixture(scope="module")
def wide(lib):
    """A 1135-accession panel on cuda:0, one sample on it, and the window layout of the TAIR10 chromosomes."""
    from snpmatch_b200.core import genomes
    p = synth.small_panel(n_rows=20000, n_acc=N_ACC)
    s = synth.make_sample(p["positions"], p["chr_regions"], p["chrs"], N_ACC, true_acc=7, n_db=3000, n_extra=300, seed=611)
    db = lib.Database(p["positions"], p["chr_regions"], N_ACC, device=0)
    db.load_int8(p["snps"])
    cnt, off, n_w, _ = genomes.Genome("athaliana_tair10").window_layout(p["chrs"], BIN_LEN)
    yield db, s, (cnt, off, n_w)
    db.close()


class _ProcInfo(ctypes.Structure):                 # nvmlProcessInfo_t
    _fields_ = [("pid", ctypes.c_uint), ("usedGpuMemory", ctypes.c_ulonglong), ("gpuInstanceId", ctypes.c_uint),
                ("computeInstanceId", ctypes.c_uint)]


def _own_device_bytes():
    """Device memory NVML charges to this process, summed over the GPUs; None when NVML does not list the process (a PID
    namespace, no driver library) or does not report its memory."""
    try:
        nvml = ctypes.CDLL("libnvidia-ml.so.1")
    except OSError:
        return None
    if nvml.nvmlInit_v2() != 0:
        return None
    try:
        n_dev = ctypes.c_uint(0)
        if nvml.nvmlDeviceGetCount_v2(ctypes.byref(n_dev)) != 0:
            return None
        total, listed = 0, False
        for i in range(n_dev.value):
            h = ctypes.c_void_p()
            if nvml.nvmlDeviceGetHandleByIndex_v2(i, ctypes.byref(h)) != 0:
                continue
            cap = 1024
            while True:
                n = ctypes.c_uint(cap)
                procs = (_ProcInfo * cap)()
                rc = nvml.nvmlDeviceGetComputeRunningProcesses_v3(h, ctypes.byref(n), procs)
                if rc != 7:                        # NVML_ERROR_INSUFFICIENT_SIZE: n holds the count now
                    break
                cap = n.value + 64
            if rc != 0:
                continue
            for p in procs[:n.value]:
                if p.pid == os.getpid():
                    if p.usedGpuMemory == ctypes.c_ulonglong(-1).value:     # NVML_VALUE_NOT_AVAILABLE
                        return None
                    total += p.usedGpuMemory
                    listed = True
        return total if listed else None
    finally:
        nvml.nvmlShutdown()


def _window_cycle(lib, db, s, layout):
    """One batch's life as a shard of `cross` sees it: create, windows in two halves, epilogue, fetch, close."""
    from snpmatch_b200.core import snpmatch
    cnt, off, n_w = layout
    b = lib.Batch(db, [0, len(s["pos"])], s["chr_ix"], s["pos"], s["wei"])
    _, n_doubles = b.run_windows_begin(False, BIN_LEN, cnt, off, n_w, snpmatch.identity_kmax_table(500, 0.02))
    b.run_windows_finish()
    b.epilogue()
    r = b.fetch()
    b.close()
    return r, n_doubles


@pytest.mark.gpu
def test_destroyed_batches_free_their_window_buffers(lib, wide):
    db, s, layout = wide
    r, n_doubles = _window_cycle(lib, db, s, layout)          # warm-up: module load, the driver's first pools
    assert layout[2] == 200 and n_doubles * 8 >= 2 << 20
    assert int(r["m"][0]) > 0
    before = _own_device_bytes()
    if before is None:
        pytest.skip("NVML does not list this process's device memory")
    for _ in range(CYCLES):
        _window_cycle(lib, db, s, layout)
    grown = _own_device_bytes() - before
    assert grown <= 2 << 20, "%d batch lifetimes kept %.1f MB of device memory" % (CYCLES, grown / 2.0 ** 20)


@pytest.mark.gpu
def test_fetch_wait_reports_what_fetch_reports(lib, wide):
    """A one-entry identity table is too short for every window with a matched marker: the windows' epilogue counts that on the
    device, and both read-backs of the totals report it."""
    db, s, layout = wide
    cnt, off, n_w = layout
    b = lib.Batch(db, [0, len(s["pos"])], s["chr_ix"], s["pos"], s["wei"])
    b.run_windows(False, BIN_LEN, cnt, off, n_w, np.zeros(1, np.int32))
    b.epilogue()
    with pytest.raises(lib.SnpmError, match="identity table too short"):
        b.fetch()
    A = db.n_acc
    out = {"score": np.empty((1, A)), "matches": np.empty((1, A), np.int64), "ninfo": np.empty((1, A), np.int64),
           "m": np.empty(1, np.int64), "prob": np.empty((1, A)), "L": np.empty((1, A)), "LR": np.empty((1, A))}
    b.fetch_async(out)
    with pytest.raises(lib.SnpmError, match="identity table too short"):
        b.fetch_wait()
    b.close()
