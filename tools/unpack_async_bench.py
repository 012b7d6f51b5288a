#!/usr/bin/env python
"""zpb_unpack_device_async against zpb_unpack_device on one GPU, device-resident, on the C2 archive (65 536 x 128 KiB,
reference-format LZ4, built by bench.build_archive).

Reports, one JSON line each (stdout and appended to --out), with the GPU's name and power limit read in the same run:
  host_call    host time of one call until it returns (perf_counter), async against sync, median of --reps;
  queued       decoded GB/s of --queue async calls on one stream with one final synchronise, against --queue sync calls;
               the two runs' outputs, statuses and digests are compared, and checked against the archive's hashes;
  overlap      wall time of --queue async calls on one stream next to a fixed bf16 matmul loop on another, against the
               two run alone (each ends in a device synchronise)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=int, default=65536)
    ap.add_argument("--size", type=int, default=131072)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--queue", type=int, default=10)
    ap.add_argument("--mm", type=int, default=8192, help="side of the bf16 matmuls of the overlap run")
    ap.add_argument("--mm-iters", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_unpack_async.jsonl"))
    a = ap.parse_args()
    import torch
    import bench
    import zpack_b200
    from zpack_b200 import container

    assert torch.cuda.is_available(), "needs a GPU"
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    gpu = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"

    def emit(rec):
        rec = dict(rec, gpu=gpu, entries=a.entries, entry_bytes=a.size)
        print(json.dumps(rec), flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(json.dumps(rec) + "\n")

    arch = bench.build_archive(a.entries, a.size)
    d = container.parse(arch)
    e = d.entries()
    out_size = int(e["dst_off"][-1] + e["dst_cap"][-1])
    total = int(d.uncomp_size.sum())
    n = len(e)
    ctx = zpack_b200.Context(0)
    d_arch = torch.from_numpy(arch).cuda()
    d_out = torch.empty(out_size, dtype=torch.uint8, device="cuda")
    d_out2 = torch.empty(out_size, dtype=torch.uint8, device="cuda")
    d_status = torch.empty(n, dtype=torch.int32, device="cuda")
    d_digest = torch.empty(n, dtype=torch.int64, device="cuda")
    s = torch.cuda.Stream()
    want = np.asarray(d.hash, np.uint64)

    def sync_call(out):
        return ctx.unpack_device(d_arch, len(arch), out, out_size, e, s.cuda_stream)

    def async_call(out):
        ctx.unpack_device_async(d_arch, len(arch), out, out_size, e, d_status, d_digest, s.cuda_stream)

    for _ in range(3):
        st, dg = sync_call(d_out)
        async_call(d_out2)
        s.synchronize()
    assert (st == 0).all() and np.array_equal(dg, want)

    # ---- host time of one call
    t_sync, t_async = [], []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        sync_call(d_out)
        t_sync.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        async_call(d_out2)
        t_async.append(time.perf_counter() - t0)
        s.synchronize()
    emit({"what": "host_call", "sync_ms": 1e3 * statistics.median(t_sync), "async_ms": 1e3 * statistics.median(t_async),
          "sync_kernel_ms": ctx.last_kernel_ms()["unpack_ms"]})

    # ---- queued calls against back-to-back synchronous calls
    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    rates = {"sync": [], "async": []}
    for _ in range(3):
        rates["sync"].append(a.queue * total / timed(lambda: [sync_call(d_out) for _ in range(a.queue)]) / 1e9)
        rates["async"].append(a.queue * total / timed(lambda: [async_call(d_out2) for _ in range(a.queue)]) / 1e9)
    st, dg = sync_call(d_out)
    s.synchronize()
    same = (bool(torch.equal(d_out, d_out2)) and np.array_equal(d_status.cpu().numpy(), st)
            and np.array_equal(d_digest.cpu().numpy().view(np.uint64), dg) and np.array_equal(dg, want))
    assert same, "async and sync results differ"
    emit({"what": "queued", "calls": a.queue, "sync_gbps": max(rates["sync"]), "async_gbps": max(rates["async"]),
          "sync_gbps_runs": rates["sync"], "async_gbps_runs": rates["async"], "outputs_equal": same})

    # ---- the decode next to a matmul loop on another stream
    x = torch.randn(a.mm, a.mm, dtype=torch.bfloat16, device="cuda")
    y = torch.randn(a.mm, a.mm, dtype=torch.bfloat16, device="cuda")
    z = torch.empty_like(x)
    s2 = torch.cuda.Stream()

    def mm_loop():
        with torch.cuda.stream(s2):
            for _ in range(a.mm_iters):
                torch.matmul(x, y, out=z)

    def decode():
        for _ in range(a.queue):
            async_call(d_out2)

    def both():
        mm_loop()
        decode()

    mm_loop()
    torch.cuda.synchronize()
    runs = {"decode_alone": [], "matmul_alone": [], "both": []}
    for _ in range(3):
        runs["decode_alone"].append(timed(decode))
        runs["matmul_alone"].append(timed(mm_loop))
        runs["both"].append(timed(both))
    emit({"what": "overlap", "calls": a.queue, "matmul": f"{a.mm}^3 bf16 x {a.mm_iters}",
          **{k + "_ms": 1e3 * min(v) for k, v in runs.items()}})
    ctx.close()


if __name__ == "__main__":
    main()
