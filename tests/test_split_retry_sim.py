"""The device-side retry of zpb_unpack_device_async (split_retry_kernel, zpack_b200/csrc/split_entries.cuh) on the CPU
emulation (tests/sim/sim_rt.h): every split parent marked for a retry lands exactly once in the list of its method, with
the descriptor the caller gave; nothing else in the batch changes."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from zpack_b200.lib import Entry

HERE = os.path.dirname(os.path.abspath(__file__))
SIM = os.path.join(HERE, "sim")
LIB = os.path.join(SIM, "libsplit_retry_sim.so")
CSRC = os.path.join(os.path.dirname(HERE), "zpack_b200", "csrc")

M_LZ4_BLOCK, M_ZSTD_FRAME, M_SPLIT = 0x102, 0x103, 0x104
ST_SPLIT_RETRY = 0x5350
CNT_RETRY_LZ4, CNT_RETRY_ZSTD = 19, 21
SplitJob = np.dtype([("kib0", "<u8"), ("desc_base", "<u8"), ("parent", "<u4"), ("row0", "<u4"), ("nrows", "<u4"),
                     ("slot_base", "<u4"), ("method", "<u4"), ("pad", "<u4")])
SENTINEL = 0xA5A5A5A5


def _build():
    deps = [os.path.join(SIM, f) for f in ("split_retry_sim.cpp", "sim_rt.h", "sim_cuda.h")]
    deps += [os.path.join(CSRC, f) for f in ("split_entries.cuh", "lz4_fast.cuh", "ptx.cuh", "common.cuh")]
    if os.path.exists(LIB) and all(os.path.getmtime(d) <= os.path.getmtime(LIB) for d in deps):
        return
    subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-DZPB_SIM", "-shared", "-fPIC", "-w",
                    os.path.join(SIM, "split_retry_sim.cpp"), "-o", LIB], check=True)


@pytest.fixture(scope="module")
def sim():
    _build()
    lib = C.CDLL(LIB)
    vp = C.c_void_p
    lib.sim_split_job_size.restype = C.c_uint32
    lib.sim_split_retry.argtypes = [vp, C.c_uint32, vp, vp, vp, vp, vp, C.c_uint64]
    assert lib.sim_split_job_size() == SplitJob.itemsize
    return lib


def _batch(rng, n_caller, kinds):
    """A batch as the pre-pass and the chain kernel leave it.  kinds[k] of job k: (method, verdict) with verdict
    'retry' (split, a piece failed), 'ok' (split, decoded) or 'declined' (the pre-pass kept it whole).  Returns the
    caller's rows, the rows after the kernels, statuses and jobs."""
    parents = rng.choice(n_caller, size=len(kinds), replace=False)
    parents.sort()
    n = n_caller + 3 * len(kinds)
    given = np.zeros(n, Entry)
    raw = rng.integers(0, 2**63, size=(n, 8), dtype=np.int64).view(np.uint8).reshape(n, 64)
    given.view(np.uint8).reshape(n, 64)[:] = raw
    given["method"] = rng.choice([0, 1, 2], size=n)
    status = rng.choice([0, 12, 13, 15, 16], size=n).astype(np.int32)
    jobs = np.zeros(len(kinds), SplitJob)
    rows = given.copy()
    for k, ((method, verdict), p) in enumerate(zip(kinds, parents)):
        given["method"][p] = method
        rows["method"][p] = method
        jobs[k]["parent"], jobs[k]["row0"], jobs[k]["nrows"], jobs[k]["method"] = p, n_caller + 3 * k, 3, method
        jobs[k]["kib0"], jobs[k]["desc_base"], jobs[k]["slot_base"] = 192 * k, 7 * k, 5 * k
        for r in range(3):
            rows["method"][n_caller + 3 * k + r] = M_ZSTD_FRAME if method == 1 else M_LZ4_BLOCK
        if verdict != "declined":
            rows["method"][p] = M_SPLIT
            status[p] = ST_SPLIT_RETRY if verdict == "retry" else rng.choice([0, 15])
    return given, rows, status, jobs


def _run(sim, rows, status, jobs, seed):
    rows = rows.copy()
    cap = max(len(jobs), 1) + 4
    lz4 = np.full(cap, SENTINEL, np.uint32)
    zstd = np.full(cap, SENTINEL, np.uint32)
    counters = np.zeros(64, np.uint32)
    counters[:19] = np.arange(1, 20)                  # slots of the kernels before: left as they are
    before = counters.copy()
    sim.sim_split_retry(jobs.ctypes.data, len(jobs), rows.ctypes.data, status.ctypes.data, lz4.ctypes.data,
                        zstd.ctypes.data, counters.ctypes.data, seed)
    return rows, lz4, zstd, counters, before


KINDS = [
    [(2, "retry")],
    [(1, "retry")],
    [(2, "retry"), (1, "retry"), (2, "ok"), (1, "ok"), (2, "declined"), (1, "declined")],
    [(2, "ok"), (1, "declined")],
    [(m, v) for m in (1, 2) for v in ("retry", "ok", "declined")] * 50,   # more jobs than one CTA
]


@pytest.mark.parametrize("case", range(len(KINDS)))
@pytest.mark.parametrize("seed", [1, 2])
def test_retry_parents_land_once_in_their_list(sim, case, seed):
    rng = np.random.default_rng(100 * case + seed)
    kinds = KINDS[case]
    given, rows, status, jobs = _batch(rng, 40 + 2 * len(kinds), kinds)
    status_before = status.copy()
    got, lz4, zstd, counters, before = _run(sim, rows, status, jobs, seed)
    want_lz4 = sorted(int(j["parent"]) for j, (m, v) in zip(jobs, kinds) if v == "retry" and m == 2)
    want_zstd = sorted(int(j["parent"]) for j, (m, v) in zip(jobs, kinds) if v == "retry" and m == 1)
    n_lz4, n_zstd = int(counters[CNT_RETRY_LZ4]), int(counters[CNT_RETRY_ZSTD])
    assert sorted(lz4[:n_lz4].tolist()) == want_lz4 and sorted(zstd[:n_zstd].tolist()) == want_zstd
    assert (lz4[n_lz4:] == SENTINEL).all() and (zstd[n_zstd:] == SENTINEL).all()
    keep = np.ones(64, bool)
    keep[[CNT_RETRY_LZ4, CNT_RETRY_ZSTD]] = False
    assert (counters[keep] == before[keep]).all()
    retried = want_lz4 + want_zstd
    assert got[retried].tobytes() == given[retried].tobytes()            # the caller's descriptor, method included
    others = np.setdiff1d(np.arange(len(rows)), retried)
    assert got[others].tobytes() == rows[others].tobytes()               # split, declined, pseudo and plain rows
    assert (status == status_before).all()


def test_batch_without_jobs_is_untouched(sim):
    rng = np.random.default_rng(7)
    _, rows, status, _ = _batch(rng, 64, [])
    status[:8] = ST_SPLIT_RETRY                                          # no job names these rows
    got, lz4, zstd, counters, before = _run(sim, rows, status, np.zeros(0, SplitJob), 3)
    assert got.tobytes() == rows.tobytes()
    assert (lz4 == SENTINEL).all() and (zstd == SENTINEL).all() and (counters == before).all()
