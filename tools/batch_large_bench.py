#!/usr/bin/env python
"""Large entries inside a device-resident batch (zpb_unpack_device) on one GPU.

Times, with CUDA events around each call (the call ends in a device synchronise): --small entries of 128 KiB
(corpus.entry_bytes, packed by the GPU as LZ4) alone; the same batch plus one --big-mib GPU-written LZ4 entry (independent
64 KB blocks); plus one GPU-written zstd entry of 64 KB frames; plus both.  Each large entry is also timed alone through
zpb_unpack_blocks_device + zpb_blocks_digest (one shard).  With --profile, one more pass per batch under torch.profiler
gives the device time of each kernel by name.  Every call's statuses and digests are checked.

Only C-ABI functions of the previous release are called, so `--lib` can point at an older build of libzpack_b200.so and
the two builds can be compared in the same session.  One JSON line per measurement on stdout and appended to --out, with
the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=None, help="libzpack_b200.so to load (default: the tree's)")
    ap.add_argument("--tag", default="this")
    ap.add_argument("--small", type=int, default=8192)
    ap.add_argument("--big-mib", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--big-reps", type=int, default=3, help="repetitions of the batches with a large entry")
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_batch_large.jsonl"))
    a = ap.parse_args()
    import torch
    from zpack_b200 import lib as zlib
    if a.lib:
        zlib.load_library(os.path.abspath(a.lib))
    import zpack_b200
    from test_gpu_lz4hc import _pack_device
    from oracle import oracle as O
    from zpack_b200 import container, corpus

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    gpu = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"
    ctx = zpack_b200.Context(0)

    def emit(rec):
        rec = dict(rec, tag=a.tag, gpu=gpu)
        print(json.dumps(rec), flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(json.dumps(rec) + "\n")

    small = [corpus.entry_bytes(i, 131072) for i in range(a.small)]
    frames = []
    for k in range(0, a.small, 1024):
        f, _, _, st = _pack_device(ctx, small[k:k + 1024], [2] * len(small[k:k + 1024]), [1] * len(small[k:k + 1024]))
        assert (st == 0).all()
        frames += f
    big = corpus.big_entry(a.big_mib << 20, piece=(1 << 20) + 333, first=7)
    big_lz4 = _pack_device(ctx, [big], [2], [1])[0][0]
    big_zst = _pack_device(ctx, [big], [1], [3])[0][0]
    h_small = [O.xxh3_port(b) for b in small]
    h_big = O.xxh3_port(big)

    def batch(extra):
        fr = frames + [f for f, _ in extra]
        sz = [131072] * a.small + [len(big)] * len(extra)
        arch = container.assemble([f"e{i}" for i in range(len(fr))], fr, sz, h_small + [h_big] * len(extra),
                                  [2] * a.small + [m for _, m in extra])
        return arch, container.parse(arch).entries()

    def timed(arch, e, reps):
        d_arch = torch.from_numpy(arch).cuda()
        out_size = int((e["dst_off"] + e["dst_cap"]).max())
        d_out = torch.empty(out_size + 64, dtype=torch.uint8, device="cuda")
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ts = []
        for r in range(reps + 1):
            ev0.record()
            st, dg = ctx.unpack_device(d_arch, len(arch), d_out, out_size, e)
            ev1.record()
            torch.cuda.synchronize()
            assert (st == 0).all() and (dg == e["hash"]).all(), np.flatnonzero(st)
            if r:
                ts.append(ev0.elapsed_time(ev1))
        kern = {}
        if a.profile:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                ctx.unpack_device(d_arch, len(arch), d_out, out_size, e)
                torch.cuda.synchronize()
            for ev in prof.key_averages():
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                if t and ("kernel" in ev.key or "Kernel" in ev.key):
                    kern[ev.key.split("(")[0]] = round(t / 1e3, 3)
        del d_arch, d_out
        torch.cuda.empty_cache()
        return ts, kern

    for name, extra in (("small", []), ("small+lz4", [(big_lz4, 2)]), ("small+zstd", [(big_zst, 1)]),
                        ("small+lz4+zstd", [(big_lz4, 2), (big_zst, 1)])):
        arch, e = batch(extra)
        ts, kern = timed(arch, e, a.reps if not extra else a.big_reps)
        dec = 131072 * a.small + len(big) * len(extra)
        emit({"what": "batch", "batch": name, "entries": len(e), "big_mib": a.big_mib, "ms": ts,
              "ms_median": float(np.median(ts)), "decoded_gbs": dec / (np.median(ts) * 1e6), "kernels_ms": kern})

    # each large entry alone on the dedicated path: the whole entry as one shard
    for name, fr in (("lz4", big_lz4), ("zstd", big_zst)):
        blocks = (zlib.lz4_frame_index(fr)[0] if name == "lz4" else zlib.zstd_frame_index(fr)[0])
        d_fr = torch.from_numpy(fr).cuda()
        d_out = torch.empty(len(big) + 64, dtype=torch.uint8, device="cuda")
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ts = []
        for r in range(a.reps + 1):
            ev0.record()
            assert ctx.unpack_blocks_device(d_fr, len(fr), d_out, len(big), blocks, 65536, len(big)) == 0
            _, dg = ctx.blocks_digest(None, 0, len(big), d_out)
            ev1.record()
            torch.cuda.synchronize()
            assert dg == h_big
            if r:
                ts.append(ev0.elapsed_time(ev1))
        emit({"what": "dedicated", "entry": name, "big_mib": a.big_mib, "comp": len(fr), "ms": ts,
              "ms_median": float(np.median(ts))})
        del d_fr, d_out
    ctx.close()


if __name__ == "__main__":
    main()
