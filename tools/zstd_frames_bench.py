#!/usr/bin/env python
"""Large zstd entries written as one frame per 64 KB (ZPB_ZSTD_FRAMED_MIN and up) on one GPU: one entry each of the given
sizes, of the zpk-synth-v1 big-entry class mix (corpus.big_entry) and of bf16 (tests/entropy_data.py, entropy switch on).

Write side: zpb_pack_device time split by zpb_last_pack_stage_ms, the ratio against the same bytes packed as 128 KiB files,
and against the reference's zstd level 3 when oracle/_ref is built.  Read side, device-resident: the frame-parallel path
(zpb_unpack_blocks_device + zpb_blocks_digest, the entry as one shard), the single-warp path (the entry as one
zpb_unpack_device entry; only up to --single-max MiB, it is slow), zpb_unpack_entry_blocks_host end to end from pinned
host memory, and the reference's one-shot zpack_read_file on one host thread.  Every read is checked against the input's
XXH3-64.  Times are medians of --reps after one warm-up, host clock around calls that end in a device synchronise;
decoded GB/s is uncomp / t, and hbm_frac is (comp + uncomp) / t over MEASURED_PEAKS.json hbm_gbs (DESIGN §5).  One JSON
line per measurement, also appended to --out, with the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _median_time(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="64,256,1024", help="entry sizes in MiB")
    ap.add_argument("--kinds", default="mix,bf16")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--single-max", type=int, default=64, help="largest entry (MiB) timed on the single-warp path")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_zstd_frames.jsonl"))
    a = ap.parse_args()
    import torch
    import entropy_data as ED
    import zpack_b200
    from bench import peaks
    from oracle import oracle as O
    from zpack_b200 import container, corpus
    from zpack_b200 import lib as zlib

    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    gpu = torch.cuda.get_device_name(0)
    try:
        gpu += ", power limit " + subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                                 capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        gpu += ", power limit not read"
    hbm, hbm_src = peaks()
    O.port()
    have_ref = O.have_ref()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    sink = open(a.out, "a")

    def emit(**kv):
        kv.update(gpu=gpu)
        line = json.dumps(kv)
        print(line, flush=True)
        sink.write(line + "\n")
        sink.flush()

    ctx = zpack_b200.Context(0)
    K64, SMALL = 65536, 131072
    for kind in a.kinds.split(","):
        ctx.set_zstd_entropy(kind == "bf16")
        for mib in [int(s) for s in a.sizes.split(",")]:
            total = mib << 20
            data = corpus.big_entry(total, piece=1 << 20) if kind == "mix" else ED.class_bytes("bf16", total)
            want = O.xxh3_port(data)
            base = {"kind": kind, "zstd_entropy": int(kind == "bf16"), "uncomp_bytes": total}
            # ---- write: one file
            f = np.zeros(1, zlib.File)
            cap = ctx.pack_bound(1, total)
            f["size"], f["dst_cap"], f["method"], f["level"] = total, cap, 1, 3
            d_in = torch.from_numpy(data).cuda()
            d_pack = torch.empty(cap + 16, dtype=torch.uint8, device="cuda")
            res = {}

            def pack():
                res["r"] = ctx.pack_device(d_in, total, d_pack, cap + 16, f)
                res["k"] = ctx.last_kernel_ms()
            t = _median_time(pack, a.reps)
            comp, dg, st = res["r"]
            assert st[0] == 0 and int(dg[0]) == want
            comp = int(comp[0])
            entry = d_pack[:comp].cpu().numpy()
            # the same bytes as 128 KiB files
            n = total // SMALL
            fs = np.zeros(n, zlib.File)
            scap = ctx.pack_bound(1, SMALL)
            slot = (scap + 15) & ~15
            fs["src_off"] = np.arange(n, dtype=np.uint64) * SMALL
            fs["size"], fs["dst_cap"], fs["method"], fs["level"] = SMALL, scap, 1, 3
            fs["dst_off"] = np.arange(n, dtype=np.uint64) * slot
            d_small = torch.empty(n * slot, dtype=torch.uint8, device="cuda")
            c_small, _, s_small = ctx.pack_device(d_in, total, d_small, n * slot, fs)
            assert (s_small == 0).all()
            del d_small
            ratio = total / comp
            line = dict(base, side="write", comp_bytes=comp, wall_ms=round(t * 1e3, 2),
                        pack_kernel_ms=round(res["k"]["pack_ms"], 2), blocks_ms=round(res["k"]["pack_blocks_ms"], 2),
                        frames_ms=round(res["k"]["pack_frames_ms"], 2), uncomp_GBps=round(total / t / 1e9, 2),
                        ratio=round(ratio, 4), ratio_128KiB_files=round(total / float(c_small.sum()), 4))
            if have_ref:
                line["ratio_reference_zstd3"] = round(total / len(O.zstd_compress_ref(data, 3)), 4)
            emit(**line)
            del d_pack
            # ---- read, device-resident
            frames, content = zlib.zstd_frame_index(entry)
            assert content == total
            d_arch = torch.from_numpy(entry).cuda()
            d_out = torch.empty(total + 16, dtype=torch.uint8, device="cuda")
            got = {}

            def frame_parallel():
                assert ctx.unpack_blocks_device(d_arch, comp, d_out, total, frames, K64, total) == 0
                got["z"] = ctx.last_stage_ms()["zstd_ms"]
                _, got["d"] = ctx.blocks_digest(None, 0, total, d_out)
                got["c"] = ctx.last_chain_ms()
            t = _median_time(frame_parallel, a.reps)
            assert got["d"] == want
            emit(**dict(base, side="read", path="frame_parallel_device", comp_bytes=comp, frames=len(frames),
                        wall_ms=round(t * 1e3, 2), zstd_kernel_ms=round(got["z"], 2), chain_ms=round(got["c"], 2),
                        decoded_GBps=round(total / t / 1e9, 2),
                        hbm_frac=round((comp + total) / t / 1e9 / hbm, 4), hbm_gbs=hbm, hbm_source=hbm_src))
            if mib <= a.single_max:
                e = np.zeros(1, zlib.Entry)
                e["comp_size"], e["dst_cap"], e["uncomp_size"], e["hash"], e["method"] = comp, total, total, want, 1

                def single_warp():
                    got["s"] = ctx.unpack_device(d_arch, comp, d_out, total + 16, e)
                    got["z"] = ctx.last_stage_ms()["zstd_ms"]
                t = _median_time(single_warp, 1)
                assert got["s"][0][0] == 0
                emit(**dict(base, side="read", path="single_warp_device", comp_bytes=comp, wall_ms=round(t * 1e3, 2),
                            zstd_kernel_ms=round(got["z"], 2), decoded_GBps=round(total / t / 1e9, 3),
                            hbm_frac=round((comp + total) / t / 1e9 / hbm, 5), hbm_gbs=hbm, hbm_source=hbm_src))
            del d_arch, d_out
            # ---- read, host buffers (pinned)
            h_entry = torch.from_numpy(entry).pin_memory()
            h_out = torch.empty(total, dtype=torch.uint8).pin_memory()

            def entry_host():
                got["h"] = ctx.unpack_entry_blocks_host(h_entry.data_ptr(), comp, h_out.data_ptr(), total, total, want)
            t = _median_time(entry_host, a.reps)
            assert got["h"] == (0, want) and np.array_equal(h_out.numpy()[:1 << 20], data[:1 << 20])
            emit(**dict(base, side="read", path="entry_blocks_host", comp_bytes=comp, wall_ms=round(t * 1e3, 2),
                        decoded_GBps=round(total / t / 1e9, 2)))
            del h_entry, h_out
            if have_ref:
                arch = container.assemble(["e"], [entry], [total], [want], [1])
                rd = O.RefReader(arch)

                def ref_read():
                    got["r"] = rd.read(0)[0]
                t = _median_time(ref_read, 1)
                rd.close()
                assert got["r"] == 0
                emit(**dict(base, side="read", path="reference_one_thread", comp_bytes=comp, wall_ms=round(t * 1e3, 2),
                            decoded_GBps=round(total / t / 1e9, 3)))
            else:
                emit(**dict(base, side="read", path="reference_one_thread", note="not measured: oracle/_ref is not built"))
            del d_in
            torch.cuda.empty_cache()
    ctx.close()
    sink.close()


if __name__ == "__main__":
    main()
