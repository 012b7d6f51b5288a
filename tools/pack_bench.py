#!/usr/bin/env python
"""Developer benchmark for BASELINE config C3: LZ4 pack of the zpk-synth-v1 corpus, device-resident.
Prints one JSON line per class: uncompressed GB/s, ratio vs the reference algorithm at level 0, kernel ms; with
--level N (LZ4 HC from 3 on) also the block / framing stage ms and the GPU's level-0 ratio on the same data."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _gen(args):
    lo, hi, size, cls = args
    from zpack_b200 import corpus
    from oracle import oracle as O
    out = np.empty((hi - lo, size), np.uint8)
    ref = 0
    for k, i in enumerate(range(lo, hi)):
        out[k] = corpus.entry_bytes(4 * i + cls if cls >= 0 else i, size)
        if k % 16 == 0:
            ref += len(O.lz4f_encode_port(out[k], 0, True)) * 16
    return out, ref


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=int, default=16384)
    ap.add_argument("--size", type=int, default=131072)
    ap.add_argument("--classes", default="-1")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--method", type=int, default=2, help="2 = LZ4 (default), 1 = zstd")
    ap.add_argument("--level", type=int, default=0, help="LZ4 level; >= 3 turns the context's HC switch on (zpb_set_lz4hc)")
    a = ap.parse_args()
    import multiprocessing as mp
    import torch
    import zpack_b200
    from zpack_b200 import lib as zlib
    ctx = zpack_b200.Context(0)
    if a.level >= 3:
        ctx.set_lz4hc(True)
    gpu = torch.cuda.get_device_name(0)
    try:
        import subprocess
        gpu += ", power limit " + subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                                 capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pass
    names = {0: "random", 1: "text", 2: "runs", 3: "records", -1: "mixed"}
    for cls in [int(c) for c in a.classes.split(",")]:
        w = min(os.cpu_count() or 1, 64)
        step = max(1, a.entries // (4 * w))
        with mp.get_context("fork").Pool(w) as pool:
            res = pool.map(_gen, [(s, min(s + step, a.entries), a.size, cls) for s in range(0, a.entries, step)])
        data = np.concatenate([r[0] for r in res])
        ref_comp = sum(r[1] for r in res)
        n = a.entries
        f = np.zeros(n, zlib.File)
        cap = ctx.pack_bound(a.method, a.size)
        slot = (cap + 15) & ~15
        f["src_off"] = np.arange(n, dtype=np.uint64) * a.size
        f["size"] = a.size
        f["dst_off"] = np.arange(n, dtype=np.uint64) * slot
        f["dst_cap"] = cap
        f["method"] = a.method
        f["level"] = a.level
        d_in = torch.from_numpy(data.reshape(-1)).cuda()
        d_out = torch.empty(n * slot, dtype=torch.uint8, device="cuda")
        ms, stages = [], []
        for r in range(a.reps + 1):
            comp, dg, st = ctx.pack_device(d_in, d_in.numel(), d_out, d_out.numel(), f)
            if r:
                k = ctx.last_kernel_ms()
                ms.append(k["pack_ms"])
                stages.append((k["pack_blocks_ms"], k["pack_frames_ms"]))
        assert (st == 0).all()
        t = float(np.median(ms))
        unc = n * a.size
        line = {"method": a.method, "level": a.level, "class": names[cls], "entries": n, "pack_kernel_ms": round(t, 3),
                "uncomp_GBps": round(unc / t / 1e6, 1), "traffic_GBps": round((unc + int(comp.sum())) / t / 1e6, 1),
                "ratio_gpu": round(unc / float(comp.sum()), 3), "ratio_reference_level0_sampled": round(unc / ref_comp, 3)}
        if a.level:                   # the stages, and the GPU's level 0 on the same data
            line["blocks_ms"] = round(float(np.median([x[0] for x in stages])), 3)
            line["frames_ms"] = round(float(np.median([x[1] for x in stages])), 3)
            f["level"] = 0
            comp0, _, st0 = ctx.pack_device(d_in, d_in.numel(), d_out, d_out.numel(), f)
            assert (st0 == 0).all()
            line["ratio_gpu_level0"] = round(unc / float(comp0.sum()), 3)
        line["gpu"] = gpu
        print(json.dumps(line), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
