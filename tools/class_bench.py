#!/usr/bin/env python
"""Developer microbenchmark: unpack+verify throughput per corpus class (random / text / runs /
records) and per tuning, device-resident.  Not the contract bench (that is bench.py) — this is
what tells which class bounds the kernel.  Prints one JSON line per (class, tuning)."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _pack(args):
    cls, lo, hi, size, indep, method = args
    from zpack_b200 import corpus
    from oracle import oracle as O
    fr, hs = [], np.empty(hi - lo, np.uint64)
    for k, i in enumerate(range(lo, hi)):
        b = corpus.entry_bytes(4 * i + cls if cls >= 0 else i, size)
        fr.append(O.zstd_compress_ref(b, 3) if method == 1 else O.lz4f_encode_port(b, 0, indep))
        hs[k] = O.xxh3_port(b)
    return fr, hs


def build(cls, n, size, indep, method=2):
    import multiprocessing as mp
    from zpack_b200 import container
    w = min(os.cpu_count() or 1, 64)
    step = max(1, n // (4 * w))
    jobs = [(cls, a, min(a + step, n), size, indep, method) for a in range(0, n, step)]
    with mp.get_context("fork").Pool(w) as pool:
        res = pool.map(_pack, jobs, chunksize=1)
    frames = [f for fr, _ in res for f in fr]
    hashes = np.concatenate([h for _, h in res])
    return container.assemble([f"{i}" for i in range(n)], frames, [size] * n, hashes, [method] * n)


def _counters(ctx):
    import ctypes as C
    if not hasattr(ctx.lib, "zpb_debug_counters"):
        return None
    a = (C.c_uint32 * 16)()
    ctx.lib.zpb_debug_counters(C.c_void_p(ctx.h), a)
    return {"heavy": a[8], "medium": a[9], "light": a[10], "split_second_tries": a[15], "split_retries": a[14], "general": a[1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=int, default=4096)
    ap.add_argument("--size", type=int, default=131072)
    ap.add_argument("--groups", default="4,8,16,32")
    ap.add_argument("--classes", default="0,1,2,3,-1")
    ap.add_argument("--independent", action="store_true")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--fast", type=int, default=1)
    ap.add_argument("--exec-ctas", default="", help="comma list of ZPB_EXEC_CTAS values to sweep (LZ4 execute kernel: 3 or 4)")
    ap.add_argument("--overlap", default="", help="comma list of 0/1: parse / execute overlap off / on")
    ap.add_argument("--method", default="lz4", choices=["lz4", "zstd"],
                    help="zstd: frames written by the unmodified reference (oracle/_ref), level 3")
    args = ap.parse_args()
    import torch
    import zpack_b200
    from zpack_b200 import container
    names = {0: "random", 1: "text", 2: "runs", 3: "records", -1: "mixed"}
    for cls in [int(c) for c in args.classes.split(",")]:
        arch = build(cls, args.entries, args.size, args.independent, 1 if args.method == 'zstd' else 2)
        d = container.parse(arch)
        e = d.entries()
        out_size = int(e["dst_off"][-1] + e["dst_cap"][-1])
        d_arch = torch.from_numpy(arch).cuda()
        d_out = torch.empty(out_size, dtype=torch.uint8, device="cuda")
        comp, unc = int(d.comp_size.sum()), int(d.uncomp_size.sum())
        sweep = [(g, c, ov) for g in [int(x) for x in args.groups.split(",")]
                 for c in ([int(x) for x in args.exec_ctas.split(",")] if args.exec_ctas else [0])
                 for ov in ([int(x) for x in args.overlap.split(",")] if args.overlap else [-1])]
        for g, xc, ov in sweep:
            if xc:
                os.environ["ZPB_EXEC_CTAS"] = str(xc)   # read when a context is created: one context per sweep point
            ctx = zpack_b200.Context(0)
            ctx.set_fast_path(bool(args.fast))
            ctx.set_tuning(group_lanes=g)
            if ov >= 0:
                ctx.set_overlap(bool(ov))
            ms = []
            for r in range(args.reps + 2):
                st, dg = ctx.unpack_device(d_arch, len(arch), d_out, out_size, e)
                if r >= 2:
                    ms.append(ctx.last_kernel_ms()["unpack_ms"])
            assert os.environ.get('ZPB_NOCHECK') or ((st == 0).all() and np.array_equal(dg, d.hash))
            t = float(np.median(ms))
            print(json.dumps({"method": args.method, "class": names[cls], "group": g, "exec_ctas": xc, "overlap": ov, "kernel_ms": round(t, 4),
                              "uncomp_GBps": round(unc / t / 1e6, 1), "traffic_GBps": round((comp + unc) / t / 1e6, 1),
                              "ratio": round(unc / comp, 3), "entries": args.entries,
                              "stages": {k: round(v, 4) for k, v in ctx.last_stage_ms().items()},
                              "counters": _counters(ctx)}), flush=True)
            if hasattr(ctx.lib, "zpb_debug_zstd_profile"):  # developer build (-DZPB_ZS_PROFILE)
                import ctypes as C
                a = (C.c_uint64 * 8)()
                ctx.lib.zpb_debug_zstd_profile(a)
                tot = float(sum(a)) or 1.0
                ph = ["literals", "seq_tables", "seq_decode", "exec_lit", "exec_par", "exec_order", "hash", "other"]
                print(json.dumps({"zstd_phase_share": {p: round(a[i] / tot, 3) for i, p in enumerate(ph)},
                                  "Mcycles_per_entry": round(tot / (args.reps + 2) / args.entries / 1e6, 3)}), flush=True)
            ctx.close()


if __name__ == "__main__":
    main()
