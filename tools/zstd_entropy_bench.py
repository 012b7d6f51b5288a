#!/usr/bin/env python
"""Developer benchmark for the zstd writer's entropy switch (zpb_set_zstd_entropy): device-resident zstd pack of the
zpk-synth-v1 corpus (mixed and its four classes) and of the classes of tests/entropy_data.py (bf16, fp16, fp32, int8
Laplace, int8 Laplace with inserted repeats), with the switch off and on.  Prints one JSON line per class and switch
state: uncompressed GB/s, ratio, the block and framing stage ms (zpb_last_pack_stage_ms), and the ratio against the
order-0 Huffman bound per 64 KB block (on the first 4 MiB).  --dump DIR writes the XXH3-64 of every frame, one .npy per
class and state, so that two builds can be compared frame for frame."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CORPUS = {"mixed": -1, "random": 0, "text": 1, "runs": 2, "records": 3}


def _gen(args):
    lo, hi, size, cls = args
    import entropy_data as ED
    from zpack_b200 import corpus
    out = np.empty((hi - lo, size), np.uint8)
    for k, i in enumerate(range(lo, hi)):
        if cls in CORPUS:
            c = CORPUS[cls]
            out[k] = corpus.entry_bytes(4 * i + c if c >= 0 else i, size)
        else:
            out[k] = ED.class_bytes(cls, size, seed=i)
    return out


def main():
    import entropy_data as ED
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=int, default=2048)
    ap.add_argument("--size", type=int, default=131072)
    ap.add_argument("--classes", default=",".join(list(CORPUS) + list(ED.CLASSES)))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--level", type=int, default=3)
    ap.add_argument("--states", default="0,1", help="switch states to run: 0 off, 1 on")
    ap.add_argument("--dump", default=None, help="directory for per-frame XXH3-64 digests (<class>_<state>.npy)")
    a = ap.parse_args()
    import multiprocessing as mp
    import torch
    import zpack_b200
    from zpack_b200 import lib as zlib
    ctx = zpack_b200.Context(0)
    has_switch = hasattr(ctx, "set_zstd_entropy")
    gpu = torch.cuda.get_device_name(0)
    try:
        import subprocess
        gpu += ", power limit " + subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                                 capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pass
    if a.dump:
        os.makedirs(a.dump, exist_ok=True)
    n = a.entries
    f = np.zeros(n, zlib.File)
    cap = ctx.pack_bound(1, a.size)
    slot = (cap + 15) & ~15
    f["src_off"] = np.arange(n, dtype=np.uint64) * a.size
    f["size"] = a.size
    f["dst_off"] = np.arange(n, dtype=np.uint64) * slot
    f["dst_cap"] = cap
    f["method"] = 1
    f["level"] = a.level
    d_out = torch.empty(n * slot, dtype=torch.uint8, device="cuda")
    for cls in a.classes.split(","):
        w = min(os.cpu_count() or 1, 64)
        step = max(1, n // (4 * w))
        with mp.get_context("fork").Pool(w) as pool:
            data = np.concatenate(pool.map(_gen, [(s, min(s + step, n), a.size, cls) for s in range(0, n, step)]))
        bound = ED.huffman_bound(data.reshape(-1)[:4 << 20])
        d_in = torch.from_numpy(data.reshape(-1)).cuda()
        for state in [int(s) for s in a.states.split(",")]:
            if has_switch:
                ctx.set_zstd_entropy(bool(state))
            elif state:
                continue                       # a build without the switch runs with it off only
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
            ratio = unc / float(comp.sum())
            line = {"class": cls, "zstd_entropy": state, "level": a.level, "entries": n, "entry_size": a.size,
                    "pack_kernel_ms": round(t, 3), "uncomp_GBps": round(unc / t / 1e6, 2), "ratio": round(ratio, 4),
                    "blocks_ms": round(float(np.median([x[0] for x in stages])), 3),
                    "frames_ms": round(float(np.median([x[1] for x in stages])), 3),
                    "huffman_bound_4MiB": round(bound, 4), "ratio_over_bound": round(ratio / bound, 4), "gpu": gpu}
            if a.dump:
                digests = ctx.xxh3_device(d_out, f["dst_off"], comp)
                np.save(os.path.join(a.dump, f"{cls}_{state}.npy"), np.stack([comp, digests]))
            print(json.dumps(line), flush=True)
        del d_in
    ctx.close()


if __name__ == "__main__":
    main()
