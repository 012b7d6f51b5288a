#!/usr/bin/env python
"""bench.py — LZ4 unpack + XXH3-64 verify throughput (BASELINE.json metric) on N B200s.

A "step" is one pass of the hot path (zpb_unpack_device: descriptor upload, scan / parse / exec kernels, status /
digest download) over one synthetic archive.  See DESIGN.md §Measurement for the definitions of
value / e2e / roofline / cpu_baseline.  `--workload` selects the other BASELINE.json configurations in the same
contract format: c3 (LZ4 pack of the corpus), c4 (zstd level-3 unpack), c5 (one huge entry sharded by blocks);
`--impl reference` times the unmodified reference (oracle/_ref) on the host cores for the same workload.
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
sys.path.insert(0, ROOT)

METRIC = "lz4_unpack_xxh3_verify_uncompressed_GBps"
ENTRY_SIZE = 131072
# BASELINE.json configs that run on one GPU: C2 (the config the metric is quoted on; default) and C4
WORKLOADS = {
    "c2": {"method": 2, "metric": METRIC, "entries": 65536, "kernel": "lz4_fast_exec_kernel", "stage": "exec_ms",
           "what": "C2: LZ4 unpack + XXH3-64 verify"},
    "c4": {"method": 1, "metric": "zstd_unpack_xxh3_verify_uncompressed_GBps", "entries": 32768,
           "kernel": "zstd_unpack_kernel", "stage": "zstd_ms",
           "what": "C4: zstd level-3 unpack + XXH3-64 verify (frames written by the reference's ZSTD_compress)"},
    # LZ4 pack of the C2 corpus (run_c3 below); `entries` = files per GPU
    "c3": {"method": 2, "metric": "lz4_pack_xxh3_uncompressed_GBps", "entries": 65536, "kernel": "lz4_pack_blocks_kernel",
           "stage": "pack_ms", "what": "C3: LZ4 pack (independent 64 KB blocks) + XXH3-64 of the input"},
    # the same through the zstd writer (LZ4 block compressor's matches as zstd blocks: Huffman literals + predefined FSE sequences)
    "c3z": {"method": 1, "metric": "zstd_pack_xxh3_uncompressed_GBps", "entries": 16384, "kernel": "lz4_pack_blocks_kernel",
            "stage": "pack_ms", "what": "C3 with the zstd writer: zstd pack (64 KB blocks, one sub-block per 4 KB window) + XXH3-64 of the input"},
    # one entry of gpus x 2 GiB, independent 64 KB blocks, sharded by blocks (run_c5 below); `entries` = blocks per GPU
    "c5": {"method": 2, "metric": "lz4_single_entry_unpack_xxh3_verify_uncompressed_GBps", "entries": 32768,
           "kernel": "lz4_fast_exec_kernel", "stage": "exec_ms",
           "what": "C5: ONE LZ4 entry of independent 64 KB blocks, unpack sharded by blocks + XXH3-64 chain relayed across GPUs"},
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_SAMPLE = 1 << 22   # decoded bytes sampled for --dump-outputs (16 MB as float32)
DUMP_SEED = 20261020


def dump_sample_positions(out_size):
    """The fixed, seeded byte positions of the decoded output that --dump-outputs keeps (all of it when it is small)."""
    if out_size <= DUMP_SAMPLE:
        return np.arange(out_size, dtype=np.int64)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(out_size, DUMP_SAMPLE, replace=False))


def dump_outputs(out_dir, rank, world, status, digest, sample):
    """--dump-outputs: what the caller of the timed path received in its last timed step, as .npy files that two
    builds can compare array for array.  float64 holds the int32 statuses and each 32-bit half of the uint64 digests
    exactly; the decoded bytes are a seeded sample (dump_sample_positions), as float32."""
    os.makedirs(out_dir, exist_ok=True)
    digest = np.asarray(digest, np.uint64)
    arrays = {"status": np.asarray(status).astype(np.float64),
              "digest_hi32": (digest >> np.uint64(32)).astype(np.float64),
              "digest_lo32": (digest & np.uint64(0xFFFFFFFF)).astype(np.float64),
              "output_sample": np.asarray(sample).astype(np.float32)}
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


def _emit(args, line):
    """The contract line: printed, unless this run is a nested measurement for the `configs` block of another line."""
    if getattr(args, "nested", False):
        args.result = line
    else:
        print(json.dumps(line))


# ------------------------------------------------------------------ archive preparation (untimed)
def _pack_shard(args):
    """Worker: generate entries [lo,hi) and pack them with the CPU checker's LZ4 frame writer.
    (Archive preparation only — the reference-format writer, never part of a timed region.)"""
    lo, hi, size, independent, method = args
    from zpack_b200 import corpus
    from oracle import oracle as O
    frames, hashes = [], np.empty(hi - lo, np.uint64)
    for k, i in enumerate(range(lo, hi)):
        b = corpus.entry_bytes(i, size)
        # zstd: the unmodified reference's one-shot compressor, level 3 (what zpack_write_files calls)
        frames.append(O.zstd_compress_ref(b, 3) if method == 1 else O.lz4f_encode_port(b, 0, independent))
        hashes[k] = O.xxh3_port(b)
    return lo, frames, hashes


def build_archive(n_entries, size, first=0, independent=False, workers=None, method=2):
    """zpk-synth-v1 corpus -> ZPack archive with reference-format LZ4 frames (linked 64 KB blocks =
    what zpack_write_files emits; byte-identical to the reference's frames, tests/test_oracle.py)."""
    import multiprocessing as mp
    from zpack_b200 import container, corpus
    workers = workers or min(os.cpu_count() or 1, 64)
    step = max(1, min(256, n_entries // (workers * 4) or 1))
    if method == 1:
        from oracle import oracle as O
        if not O.have_ref():
            raise RuntimeError("the C4 archive is packed by oracle/_ref (the reference's zstd compressor), which is absent")
    jobs = [(first + a, first + min(a + step, n_entries), size, independent, method) for a in range(0, n_entries, step)]
    frames, hashes = [None] * len(jobs), [None] * len(jobs)
    if workers > 1 and len(jobs) > 1:
        with mp.get_context("fork").Pool(workers) as pool:
            for j, (lo, fr, hs) in enumerate(pool.imap(_pack_shard, jobs, chunksize=1)):
                frames[j], hashes[j] = fr, hs
    else:
        for j, job in enumerate(jobs):
            _, frames[j], hashes[j] = _pack_shard(job)
    payload = [f for fr in frames for f in fr]
    names = [corpus.entry_name(first + i) for i in range(n_entries)]
    arch = container.assemble(names, payload, [size] * n_entries, np.concatenate(hashes), [method] * n_entries)
    return arch


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------ reference arm (CPU)
_REF_OUT = None


def cpu_unpack_throughput(arch, d, n_sample, threads, repeat=1, method=2):
    """The reference's own zpack_read_file (oracle/_ref) — or the port when _ref is absent — over
    `n_sample` entries split across `threads` host threads, one dctx each (lib/zpack.h:335-341).
    The per-entry loop runs in C (oracle/ref_driver.c); Python only starts the threads."""
    import ctypes as C
    from oracle import oracle as O
    n_sample = min(n_sample, len(d))
    threads = max(1, min(threads, n_sample))
    use_ref = O.have_ref() and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_driver.so"))
    if not use_ref and method == 1:
        threads = 1  # the port's zstd context is a single static object
    size = int(d.uncomp_size[:n_sample].max())
    bad = [0] * threads
    if use_ref:
        # BASELINE.md §4: "each calling zpack_read_file into a preallocated output slice" — ONE output of n_sample slots,
        # entry i decoded into slot i, so that the decoded bytes land in host DRAM as the GPU arm's do
        global _REF_OUT
        if _REF_OUT is None or len(_REF_OUT) < n_sample * size:
            _REF_OUT = np.empty(n_sample * size, np.uint8)
        rd = O.RefReader(arch)
        drv = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_driver.so"))
        drv.ref_unpack_slices.restype = C.c_long
        drv.ref_unpack_slices.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_void_p,
                                          C.c_size_t, C.c_int, C.c_void_p]
        ents = C.cast(rd.r.file_entries, C.c_void_p)

        def work(t):
            bad[t] = drv.ref_unpack_slices(C.byref(rd.r), ents, t, n_sample, threads, _REF_OUT.ctypes.data, size, method, None)
    else:
        outs = [np.empty(size, np.uint8) for _ in range(threads)]
        lib = O.port()
        lib.orc_unpack_range.restype = C.c_long
        lib.orc_unpack_range.argtypes = [C.c_void_p] * 6 + [C.c_size_t] * 3 + [C.c_void_p, C.c_size_t, C.c_void_p]
        cols = [np.ascontiguousarray(x) for x in (d.offset, d.comp_size, d.uncomp_size, d.hash, d.method)]

        def work(t):
            bad[t] = lib.orc_unpack_range(arch.ctypes.data, *[c.ctypes.data for c in cols], t, n_sample, threads,
                                          outs[t].ctypes.data, size, None)
    best = None
    for _ in range(repeat):
        ts = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        t0 = time.perf_counter()
        [t.start() for t in ts]
        [t.join() for t in ts]
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    if use_ref:
        rd.close()
    assert sum(bad) == 0, f"CPU baseline: {sum(bad)} entries failed to verify"
    nbytes = float(d.uncomp_size[:n_sample].sum())
    return nbytes / best / 1e9, best, ("reference" if use_ref else "port")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from zpack_b200 import container
    cores = os.cpu_count() or 1
    wl = WORKLOADS[args.workload]
    n_sample = args.ref_entries or args.entries or wl["entries"]
    if args.workload in ("c3", "c3z"):
        pm, pl = (1, 3) if args.workload == "c3z" else (2, 0)
        data, _, _ = build_corpus(n_sample, ENTRY_SIZE, 0, cores)
        for _ in range(args.warmup):
            cpu_pack_throughput(data, ENTRY_SIZE, min(n_sample, 512), cores, pm, pl)
        vals = [cpu_pack_throughput(data, ENTRY_SIZE, n_sample, cores, pm, pl) for _ in range(args.steps)]
        value, kind = float(np.mean([v[0] for v in vals])), vals[0][2]
        line = {"metric": wl["metric"], "value": value, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * n_sample * ENTRY_SIZE / (value * 1e9),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "impl": "reference",
                "config": {"workload": f"{wl['what']}, sample of {n_sample} x 128 KiB files (zpk-synth-v1), reference "
                                       f"zpack_write_archive ({'zstd level 3' if pm == 1 else 'LZ4 level 0'}) on host cores", "ratio": vals[0][3]},
                "cpu_baseline": {"value": value, "unit": "GB/s", "cores": cores, "kind": kind,
                                 "sample": f"{n_sample} files x 128 KiB per step, {cores} independent writers"},
                "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return
    arch = build_archive(n_sample, ENTRY_SIZE, independent=False, method=wl["method"])
    d = container.parse(arch)
    for _ in range(args.warmup):
        cpu_unpack_throughput(arch, d, min(n_sample, 512), cores, method=wl["method"])
    t_best, vals = None, []
    for _ in range(args.steps):
        v, dt, kind = cpu_unpack_throughput(arch, d, n_sample, cores, method=wl["method"])
        vals.append(v)
        t_best = dt if t_best is None else min(t_best, dt)
    value = float(np.mean(vals))
    line = {"metric": wl["metric"], "value": value, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * float(d.uncomp_size.sum()) / (value * 1e9),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "impl": "reference",
            "config": {"workload": f"{wl['what']}, {n_sample} entries x 128 KiB "
                                   f"({float(d.uncomp_size.sum()) / 2**30:.2f} GiB uncompressed), zpk-synth-v1, reference zpack_read_file on host "
                                   "cores, every entry decoded into its own slice of one preallocated output",
                       "entries": n_sample, "entry_bytes": ENTRY_SIZE},
            "cpu_baseline": {"value": value, "unit": "GB/s", "cores": cores, "kind": kind,
                             "sample": f"the whole {n_sample}-entry archive per step, {cores} threads, one dctx each, "
                                       "entry i -> slot i of one output buffer"},
            "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------ C5: one large entry, sharded by blocks
PIECE = 1 << 20   # the four corpus classes cycle every 1 MiB inside the big entry (SURVEY §8(d))


def _pack_pieces(args):
    lo, hi, total, first = args
    from zpack_b200 import corpus
    from oracle import oracle as O
    bodies, raw = [], []
    for k in range(lo, hi):
        b = corpus.big_entry_piece(k, PIECE, total, first)
        f = O.lz4f_encode_port(b, 0, True)
        bodies.append(f[7:-4])                      # the piece's blocks without frame header / EndMark
        raw.append(b)
    return lo, bodies, raw, O.lz4f_encode_port(np.zeros(1, np.uint8), 0, True)[:7]


def build_big_entry_shard(shard_bytes, first_piece, workers):
    """This rank's run of blocks of the big entry, as a self-contained B.Indep frame (header + blocks + EndMark),
    plus the plaintext.  Blocks are independent, so a run of them is the concatenation of the pieces' blocks."""
    import multiprocessing as mp
    n = shard_bytes // PIECE
    step = max(1, n // (workers * 4))
    jobs = [(a, min(a + step, n), shard_bytes, first_piece) for a in range(0, n, step)]
    res = [None] * len(jobs)
    if workers > 1 and len(jobs) > 1:
        with mp.get_context("fork").Pool(workers) as pool:
            for j, r in enumerate(pool.imap(_pack_pieces, jobs, chunksize=1)):
                res[j] = r
    else:
        res = [_pack_pieces(j) for j in jobs]
    header = res[0][3]
    frame = np.concatenate([header] + [b for r in res for b in r[1]] + [np.zeros(4, np.uint8)])
    data = np.concatenate([b for r in res for b in r[2]])
    return frame, data


def run_c5(args):
    import torch
    import torch.distributed as dist
    import zpack_b200
    from zpack_b200 import shard
    from zpack_b200 import lib as zlib
    from oracle import oracle as O

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    wl = WORKLOADS["c5"]
    nblk = args.entries or wl["entries"]
    bs = 65536
    shard_bytes = nblk * bs
    assert shard_bytes % PIECE == 0
    total = world * shard_bytes
    pos = rank * shard_bytes
    t_prep = time.time()
    frame, data = build_big_entry_shard(shard_bytes, rank * (shard_bytes // PIECE), max(1, (os.cpu_count() or 1) // world))
    blocks, bsz, _ = zlib.lz4_frame_index(frame)
    assert bsz == bs and len(blocks) == nblk
    prep_s = time.time() - t_prep
    comp_bytes = int(blocks["comp_size"].sum())

    ctx = zpack_b200.Context(local)
    h_frame = torch.from_numpy(frame).pin_memory()
    d_arch = h_frame.cuda()
    d_out = torch.empty(shard_bytes, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    # The only data that moves between GPUs: the 64-byte XXH3 accumulator state, rank r -> rank r + 1, once per read.
    # It goes through a host-memory mailbox (a shared-memory file mapped by every rank; one 128-byte slot per receiver:
    # sequence number, "has a state" flag, 8 accumulators) — no NCCL, no collective on the data path (north_star).
    mbox, seq = None, [0]
    if world > 1:
        path = f"/dev/shm/zpb_relay_{os.environ.get('MASTER_PORT', '0')}"
        if rank == 0:
            np.zeros(world * 16, np.uint64).tofile(path)
        dist.barrier()
        mbox = np.memmap(path, dtype=np.uint64, mode="r+", shape=(world, 16))

    def send(dst, acc):
        mbox[dst, 2:10] = 0 if acc is None else np.asarray(acc, np.uint64)
        mbox[dst, 1] = 0 if acc is None else 1
        mbox[dst, 0] = seq[0]          # published last: x86 stores become visible in program order

    def recv(src):
        while int(mbox[rank, 0]) != seq[0]:
            pass
        return np.array(mbox[rank, 2:10], np.uint64) if int(mbox[rank, 1]) else None

    times = {"decode": [], "chain": [], "stages": []}

    def step(arch_t=d_arch):
        st = ctx.unpack_blocks_device(arch_t, len(frame), d_out, shard_bytes, blocks, bs, shard_bytes, stream)
        assert st == 0, f"shard declined: {st}"
        times["decode"].append(ctx.last_kernel_ms()["unpack_ms"])
        times["stages"].append(ctx.last_stage_ms())
        seq[0] += 1
        dg = shard.relay_digest(rank, world, lambda a: ctx.blocks_digest(a, pos, total, d_out, stream), send, recv)
        times["chain"].append(ctx.last_chain_ms())
        return dg

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        digest = step()
    # ---- parity gate: this rank's bytes are the plaintext; the relayed digest is the oracle's XXH3 of the WHOLE entry
    assert torch.equal(d_out, torch.from_numpy(data).cuda()), "decoded shard differs from the plaintext"
    if world > 1:
        parts = [torch.empty(shard_bytes, dtype=torch.uint8, device="cuda") for _ in range(world)] if rank == 0 else None
        dist.gather(d_out, parts, dst=0)
        want = O.xxh3_port(torch.cat(parts).cpu().numpy()) if rank == 0 else None
        del parts
        t = torch.from_numpy(np.array([want if rank == 0 else 0], np.uint64).view(np.int64)).cuda()
        dist.broadcast(t, 0)
        want = int(t.cpu().numpy().view(np.uint64)[0])
    else:
        want = O.xxh3_port(data)
    if rank == world - 1:
        assert digest == want, f"relayed digest {digest:#x} != oracle {want:#x}"

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count
    for k in times:
        times[k].clear()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        digest = step()
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - launches0
    if rank == world - 1:
        assert digest == want
    decode_timed, chain_timed = float(np.mean(times["decode"])), float(np.mean(times["chain"]))
    # per-kernel durations: two extra, untimed steps with scan / parse / execute back to back on one stream
    # (in the timed steps the execute kernel overlaps the tail of the parse kernel)
    ctx.set_overlap(False)
    times["stages"].clear()
    for _ in range(2):
        step()
    stages = {k: float(np.mean([s[k] for s in times["stages"]])) for k in times["stages"][0]}
    ctx.set_overlap(True)

    # ---- e2e: pinned host frame -> H2D -> decode -> relay -> D2H of every decoded byte, per step
    e2e_s = 0.0
    if args.e2e:
        h_out = torch.empty(shard_bytes, dtype=torch.uint8).pin_memory()
        if world == 1:
            h_frame_np, h_out_np = h_frame.numpy(), h_out.numpy()
            ctx.unpack_entry_blocks_host(h_frame_np, len(frame), h_out_np, shard_bytes, total, want)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                r = ctx.unpack_entry_blocks_host(h_frame_np, len(frame), h_out_np, shard_bytes, total, want)
            e2e_s = (time.perf_counter() - t0) / args.e2e_steps
            assert r == (0, want)
            assert np.array_equal(h_out_np[:1 << 20], data[:1 << 20]) and np.array_equal(h_out_np[-(1 << 20):], data[-(1 << 20):])
        else:
            d_in = torch.empty_like(d_arch)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                d_in.copy_(h_frame, non_blocking=True)
                dg = step(d_in)
                h_out.copy_(d_out, non_blocking=True)
                torch.cuda.synchronize()
            barrier()
            e2e_s = (time.perf_counter() - t0) / args.e2e_steps
            if rank == world - 1:
                assert dg == want
            assert np.array_equal(h_out.numpy()[:1 << 20], data[:1 << 20])
    clocks = sampler.stop() if rank == 0 else None

    t = torch.tensor([ms_total, decode_timed, e2e_s, stages["exec_ms"]], dtype=torch.float64, device="cuda")
    tc = torch.tensor([chain_timed], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tc, op=dist.ReduceOp.SUM)      # the chain is serial across ranks: its cost is the sum
    ms_total, decode_ms, e2e_s, kern_ms = [float(x) for x in t.cpu()]
    chain_ms = float(tc.cpu()[0])
    if rank == 0:
        peak, peak_src = peaks()
        ms_step = ms_total / args.steps
        value = total / (ms_step * 1e-3) / 1e9
        algo_bytes = comp_bytes + shard_bytes
        achieved = algo_bytes / (kern_ms * 1e-3) / 1e9
        cores = os.cpu_count() or 1
        line = {"metric": wl["metric"], "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": f"{wl['what']}: entry of {total / 2**30:.0f} GiB = {world} x {nblk} blocks "
                                       f"({shard_bytes / 2**30:.2f} GiB per GPU, ratio {shard_bytes / comp_bytes:.3f}), zpk-synth-v1 classes cycling every 1 MiB",
                           "blocks_per_gpu": nblk, "block_bytes": bs,
                           "sharding": f"contiguous block runs x{world}; the only cross-GPU data is the 64-byte XXH3 state, relayed in shard order",
                           "l2": "inputs+outputs per step exceed the 126 MB L2 (no flush needed)",
                           "pipeline": "scan -> parse || exec (warp per block, per-KiB stripe sums) -> xxh3_chain_kernel, 7 launches per step",
                           "archive_prep_s": round(prep_s, 1)},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": None, "peak_source": peak_src, "kernel": wl["kernel"], "kernel_ms": kern_ms,
                             "algorithmic_bytes_per_launch": algo_bytes, "decode_ms_max_over_ranks": decode_ms,
                             "xxh3_chain_ms_sum_over_ranks": chain_ms,
                             "decode_only_GBps": total / (decode_ms * 1e-3) / 1e9, "stages_ms": stages,
                             "note": "the XXH3 scramble chain (one dependent step per KiB of the ENTRY, xxhash.h:3527-3534) is serial "
                                     "across blocks and across GPUs: it, not the decode, bounds a single huge entry"},
                "gpu_launches": int(launches), "clocks": clocks}
        if args.e2e:
            line["e2e"] = {"value": total / e2e_s / 1e9, "unit": "GB/s", "h2d_bytes_per_step": world * len(frame),
                           "d2h_bytes_per_step": total,
                           "how": ("zpb_unpack_entry_blocks_host (what zpack_read_file calls for a large entry): pinned host buffers, "
                                   "chunked H2D / decode / chain / D2H over worker streams" if world == 1 else
                                   "per rank: H2D of its block run, zpb_unpack_blocks_device, relayed zpb_blocks_digest, D2H of its output")}
        if not args.no_cpu:
            # the reference reads one entry on ONE thread (zpack_read_file is per entry; blocks of one frame are not
            # exposed to its callers): time it on a bounded prefix of the same entry
            nb = min(nblk, 4096)
            sub = np.concatenate([frame[:int(blocks["src_off"][nb - 1] + blocks["comp_size"][nb - 1])], np.zeros(4, np.uint8)])
            plain = data[:nb * bs]
            h = O.xxh3_port(plain)
            if O.have_ref():
                from zpack_b200 import container
                arch = container.assemble(["big"], [sub], [len(plain)], [h], [2])
                rd = O.RefReader(arch)
                rd.read(0)
                t0 = time.perf_counter()
                rc, _ = rd.read(0)
                dt = time.perf_counter() - t0
                rd.close()
                kind = "reference"
            else:
                t0 = time.perf_counter()
                rc, _, _ = O.read_entry_port(2, sub, len(plain), len(plain), h)
                dt = time.perf_counter() - t0
                kind = "port"
            assert rc == 0
            line["cpu_baseline"] = {"value": len(plain) / dt / 1e9, "unit": "GB/s", "cores": 1, "kind": kind,
                                    "sample": f"first {nb} blocks ({len(plain) >> 20} MiB) of the same entry through zpack_read_file, "
                                              "1 thread (one entry = one LZ4F_decompress loop + one XXH3 pass)"}
        _emit(args, line)
    if world > 1 and not getattr(args, "nested", False):
        dist.destroy_process_group()
    ctx.close()


# ------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    import zpack_b200
    from zpack_b200 import container

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    wl = WORKLOADS[args.workload]
    # Strong scaling (the default; BASELINE config 2: ONE archive of `entries` entries at 1 / 2 / 4 / 8 GPUs): the archive's
    # entries are cut into `world` contiguous runs balanced by decoded bytes (zpack_b200/shard.py, the rule of
    # zpb_group_partition) and rank r unpacks run r — it builds and holds only that run's share of the archive.
    # --scaling weak: every rank unpacks its own archive of `entries` entries (the round-1 measurement).
    n_total = args.entries or wl["entries"]
    strong = args.scaling == "strong"
    if strong:
        from zpack_b200 import shard
        lo_e, hi_e = shard.partition(np.full(n_total, ENTRY_SIZE), world)[rank]
        n_per_gpu, first_entry = hi_e - lo_e, lo_e
    else:
        n_per_gpu, first_entry = n_total, rank * n_total
    t_prep = time.time()
    arch = build_archive(n_per_gpu, ENTRY_SIZE, first=first_entry, independent=args.independent,
                         workers=max(1, (os.cpu_count() or 1) // world), method=wl["method"])
    d = container.parse(arch)
    entries = d.entries()
    out_size = int(entries["dst_off"][-1] + entries["dst_cap"][-1])
    comp_bytes, uncomp_bytes = int(d.comp_size.sum()), int(d.uncomp_size.sum())
    prep_s = time.time() - t_prep

    ctx = zpack_b200.Context(local)
    if args.group:
        ctx.set_tuning(group_lanes=args.group)
    h_arch = torch.from_numpy(arch).pin_memory()
    d_arch = h_arch.cuda(non_blocking=False)
    d_out = torch.empty(out_size, dtype=torch.uint8, device="cuda")
    h_out = torch.empty(out_size, dtype=torch.uint8).pin_memory() if args.e2e else None
    stream = torch.cuda.current_stream().cuda_stream

    def step_device():
        status, digest = ctx.unpack_device(d_arch, len(arch), d_out, out_size, entries, stream)
        return status, digest

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        status, digest = step_device()
    assert (status == 0).all() and np.array_equal(digest, d.hash), "parity gate failed before timing"

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count
    kernel_ms, stage_ms = [], []
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        status, digest = step_device()
        kernel_ms.append(ctx.last_kernel_ms()["unpack_ms"])
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - launches0
    assert (status == 0).all() and np.array_equal(digest, d.hash)
    if getattr(args, "dump_outputs", None):
        # taken before anything below writes d_out again
        pos = torch.from_numpy(dump_sample_positions(out_size)).cuda()
        dump = (status.copy(), digest.copy(), d_out[pos].cpu().numpy())
        del pos
    # per-kernel durations for the roofline: in the timed steps the execute kernel overlaps the tail of the parse
    # kernel (separate streams), so its own duration is taken from two extra, untimed steps with the kernels back to back
    ctx.set_overlap(False)
    kernel_ms_serial, stage_ms = [], []
    for _ in range(2):
        status, digest = step_device()
        kernel_ms_serial.append(ctx.last_kernel_ms()["unpack_ms"])
        stage_ms.append(ctx.last_stage_ms())
    ctx.set_overlap(True)
    assert (status == 0).all() and np.array_equal(digest, d.hash)

    # end-to-end through the host-buffer C-ABI call (pinned host archive -> H2D -> kernel -> D2H output)
    e2e, e2e_verify = None, None
    if args.e2e:
        h_arch_np, h_out_np = h_arch.numpy(), h_out.numpy()
        h_out_np[:] = 0
        ctx.unpack_host(h_arch_np, len(arch), h_out_np, out_size, entries)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            st2, dg2 = ctx.unpack_host(h_arch_np, len(arch), h_out_np, out_size, entries)
        torch.cuda.synchronize()
        e2e_s = (time.perf_counter() - t0) / args.e2e_steps
        assert (st2 == 0).all() and np.array_equal(dg2, d.hash)
        # the host copy really holds the decoded bytes: spot-check entries against the device-resident result
        for i in (0, len(entries) // 2, len(entries) - 1):
            o, sz = int(entries["dst_off"][i]), int(entries["uncomp_size"][i])
            assert np.array_equal(h_out_np[o:o + sz], d_out[o:o + sz].cpu().numpy()), "e2e output mismatch"
        e2e = e2e_s
        # verdict-only variant (`zpack t`): same call, entries flagged ZPB_F_DISCARD -> no D2H of the bytes
        ev = entries.copy()
        ev["flags"] |= 2
        ctx.unpack_host(h_arch_np, len(arch), h_out_np, out_size, ev)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            st3, dg3 = ctx.unpack_host(h_arch_np, len(arch), h_out_np, out_size, ev)
        torch.cuda.synchronize()
        e2e_verify = (time.perf_counter() - t0) / args.e2e_steps
        assert (st3 == 0).all() and np.array_equal(dg3, d.hash)
        # what the link itself allows on this box, measured here: pinned D2H and H2D of up to 1 GiB (CUDA events)
        nb = min(out_size, len(arch), 1 << 30)
        pcie = {}
        for name, dst, src in (("d2h_GBps", h_out[:nb], d_out[:nb]), ("h2d_GBps", d_out[:nb], h_out[:nb])):
            dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(3):
                dst.copy_(src, non_blocking=True)
            b.record()
            torch.cuda.synchronize()
            pcie[name] = 3 * nb / (a.elapsed_time(b) * 1e-3) / 1e9
        # the same D2H while an H2D stream is busy in the other direction — the condition of the e2e pipeline, which
        # uploads the next chunk's compressed bytes while decoded bytes go down
        side = torch.cuda.Stream()
        h_src2 = h_arch[:min(len(arch), nb)]
        d_dst2 = torch.empty(len(h_src2), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(side):
            for _ in range(6):
                d_dst2.copy_(h_src2, non_blocking=True)
        a.record()
        for _ in range(3):
            h_out[:nb].copy_(d_out[:nb], non_blocking=True)
        b.record()
        torch.cuda.synchronize()
        pcie["d2h_GBps_while_h2d"] = 3 * nb / (a.elapsed_time(b) * 1e-3) / 1e9
        del d_dst2
    clocks = sampler.stop() if rank == 0 else None

    stages = {k: float(np.mean([s[k] for s in stage_ms])) for k in stage_ms[0]}
    t = torch.tensor([ms_total, float(np.mean(kernel_ms)), e2e or 0.0, stages[wl["stage"]], e2e_verify or 0.0],
                     dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(uncomp_bytes), float(comp_bytes), float(n_per_gpu), float(stages.get("parse_ms", 0.0)),
                        float(stages.get("exec_ms", 0.0))], dtype=torch.float64, device="cuda")
    per_rank = [tot.clone() for _ in range(world)]
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_gather(per_rank, tot)
    ms_total, all_kern_ms, e2e_s, kern_ms, e2e_verify_s = [float(x) for x in t.cpu()]
    per_rank = [[float(v) for v in x.cpu()] for x in per_rank]
    job_uncomp = sum(x[0] for x in per_rank)       # what ALL ranks decoded per step
    job_comp = sum(x[1] for x in per_rank)

    if rank == 0:
        peak, peak_src = peaks()
        ms_step = ms_total / args.steps
        value = job_uncomp / (ms_step * 1e-3) / 1e9
        algo_bytes = comp_bytes + uncomp_bytes     # this rank's launch (the roofline is per kernel launch)
        achieved = algo_bytes / (kern_ms * 1e-3) / 1e9
        cores = os.cpu_count() or 1
        line = {"metric": wl["metric"], "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": f"{wl['what']}, " + (f"ONE archive of {n_total} entries x 128 KiB cut into {world} contiguous runs "
                                                            f"({job_uncomp / 2**30:.2f} GiB uncompressed in all, ratio {job_uncomp / job_comp:.3f})" if strong else
                                                            f"{n_per_gpu} entries x 128 KiB per GPU ({uncomp_bytes / 2**30:.2f} GiB uncompressed each, "
                                                            f"ratio {uncomp_bytes / comp_bytes:.3f})") + ", zpk-synth-v1"
                                       + (f", {'independent' if args.independent else 'reference-format linked'} 64 KB blocks"
                                          if wl["method"] == 2 else ""),
                           "entries_per_gpu": n_per_gpu, "entries_per_rank": [int(x[2]) for x in per_rank], "entry_bytes": ENTRY_SIZE,
                           "sharding": f"entries x{world}, contiguous runs balanced by decoded bytes, no collective",
                           "per_rank_parse_exec_ms": [[round(x[3], 3), round(x[4], 3)] for x in per_rank],
                           "l2": "inputs+outputs per step exceed the 126 MB L2 (no flush needed)",
                           "pipeline": ("scan -> parse || exec (3 grids sharing one work queue; the first starts with the parse kernel) -> general fallback, 6 launches per step" if wl["method"] == 2
                                        else "scan -> zstd_unpack_kernel (warp per entry), 5 launches per step"),
                           "archive_prep_s": round(prep_s, 1)},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak,
                             "traffic": (algo_bytes * NCU_TRAFFIC_RATIO[args.workload][0] if args.workload in NCU_TRAFFIC_RATIO else None),
                             "traffic_source": (NCU_TRAFFIC_RATIO[args.workload][1] if args.workload in NCU_TRAFFIC_RATIO else None),
                             "peak_source": peak_src,
                             "kernel": wl["kernel"], "kernel_ms": kern_ms,
                             "algorithmic_bytes_per_launch": algo_bytes,
                             "all_kernels_ms": all_kern_ms, "all_kernels_frac": algo_bytes / (all_kern_ms * 1e-3) / 1e9 / peak,
                             "stages_ms": stages,
                             "timing_note": "all_kernels_ms: first launch to last, timed steps (execute overlaps the parse tail); "
                                            "kernel_ms / stages_ms: the same kernels back to back on one stream (2 extra steps), "
                                            f"whose sum is {float(np.mean(kernel_ms_serial)):.3f} ms"},
                "gpu_launches": int(launches), "clocks": clocks}
        if args.e2e:
            line["e2e"] = {"value": job_uncomp / e2e_s / 1e9, "unit": "GB/s",
                           "h2d_bytes_per_step": comp_bytes + entries.nbytes, "d2h_bytes_per_step": uncomp_bytes + 12 * len(entries),
                           "how": "zpb_unpack_host, pinned host buffers: chunked H2D / kernels / D2H of every decoded byte, "
                                  "overlapped on 6 streams; PCIe-bound (D2H of every decoded byte)",
                           # the link's own ceiling for this step on rank 0's GPU: every decoded byte has to cross it
                           "pcie_probe": {k: round(v, 2) for k, v in pcie.items()},
                           "pcie_ceiling_GBps_per_gpu": round(uncomp_bytes / ((uncomp_bytes + 12 * len(entries)) / (pcie["d2h_GBps"] * 1e9)) / 1e9, 2)}
            line["e2e_verify_only"] = {"value": job_uncomp / e2e_verify_s / 1e9, "unit": "GB/s",
                                       "h2d_bytes_per_step": comp_bytes + entries.nbytes, "d2h_bytes_per_step": 12 * len(entries),
                                       "how": "same call with ZPB_F_DISCARD (the `zpack t` integrity test): status + digest come back, "
                                              "decoded bytes stay on the device"}
        if not args.no_cpu:
            n_s = min(args.cpu_entries, len(d))
            # best of two passes: the first one also pays the first touch of the output buffer (the reference arm,
            # `--impl reference`, has a warm-up step for the same reason)
            v, dt, kind = cpu_unpack_throughput(arch, d, n_s, cores, repeat=2, method=wl["method"])
            v1, dt1, _ = cpu_unpack_throughput(arch, d, min(n_s, 2048), 1, method=wl["method"])
            line["cpu_baseline"] = {"value": v, "unit": "GB/s", "cores": cores, "kind": kind,
                                    "sample": f"first {n_s} entries of the same archive, {cores} threads, each entry into its own slot "
                                              f"of one output, best of 2 passes; single-thread: {v1:.3f} GB/s"}
        _emit(args, line)
    if getattr(args, "dump_outputs", None):
        dump_outputs(args.dump_outputs, rank, world, *dump)
    if world > 1 and not getattr(args, "nested", False):
        dist.destroy_process_group()
    ctx.close()


# ------------------------------------------------------------------ C3: pack
_C3_SHARED = None


def _gen_shard(args):
    """Worker (fork): fills its slice of the shared corpus buffer, returns the XXH3-64 of every entry and the size
    the CPU checker's reference-format writer gives for every 17th entry (ratio reference, untimed)."""
    lo, hi, first, size = args
    from zpack_b200 import corpus
    from oracle import oracle as O
    buf = np.frombuffer(_C3_SHARED, np.uint8)
    hashes, ref = np.empty(hi - lo, np.uint64), 0
    for k, i in enumerate(range(lo, hi)):
        b = corpus.entry_bytes(first + i, size)
        buf[i * size:(i + 1) * size] = b
        hashes[k] = O.xxh3_port(b)
        if i % 17 == 0:   # 17: coprime with the 4-class cycle of the corpus
            ref += len(O.lz4f_encode_port(b, 0, False))
    return lo, hashes, ref


def build_corpus(n, size, first, workers):
    """(n x size) bytes of zpk-synth-v1 in one anonymous shared mapping, filled by `workers` forked processes."""
    import mmap
    import multiprocessing as mp
    global _C3_SHARED
    _C3_SHARED = mmap.mmap(-1, n * size)
    step = max(1, min(256, n // (workers * 4) or 1))
    jobs = [(a, min(a + step, n), first, size) for a in range(0, n, step)]
    hashes, ref = np.empty(n, np.uint64), 0
    with mp.get_context("fork").Pool(workers) as pool:
        for lo, hs, r in pool.imap_unordered(_gen_shard, jobs, chunksize=1):
            hashes[lo:lo + len(hs)] = hs
            ref += r
    return np.frombuffer(_C3_SHARED, np.uint8), hashes, ref * 17


def cpu_pack_throughput(data, size, n_sample, threads, method=2, level=0):
    """The reference's own writer (zpack_write_archive into a heap writer, oracle/_ref) over `n_sample` files split
    across `threads` independent writers (the reference writer is single-threaded by contract, lib/zpack.h:476-485:
    this is the T-way sharded variant of SURVEY section 8(d)); the port's frame writer when _ref is absent."""
    from oracle import oracle as O
    n_sample = min(n_sample, len(data) // size)
    threads = max(1, min(threads, n_sample))
    use_ref = O.have_ref()
    comp = [0] * threads

    def work(t):
        idx = range(t, n_sample, threads)
        bufs = [data[i * size:(i + 1) * size] for i in idx]
        if use_ref:
            comp[t] = len(O.write_archive_ref([f"f{i}" for i in idx], bufs, method, level))
        else:
            comp[t] = sum(len(O.lz4f_encode_port(b, 0, False)) for b in bufs)
    ts = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    t0 = time.perf_counter()
    [t.start() for t in ts]
    [t.join() for t in ts]
    dt = time.perf_counter() - t0
    return n_sample * size / dt / 1e9, dt, ("reference" if use_ref else "port"), n_sample * size / max(1, sum(comp))


def run_c3(args):
    """BASELINE config C3: LZ4 pack of the C2 corpus, files sharded across ranks, no collective; the compressed-size
    offset table is assembled on the host from comp_size[].  Gates before timing: every status 0, every digest equal
    to the XXH3-64 of the input, every GPU-written frame decodes back to its digest (GPU reader, all files) and a
    sample opens bit-exactly in the CPU checker / the unmodified reference reader."""
    import torch
    import torch.distributed as dist
    import zpack_b200
    from zpack_b200 import lib as zlib
    from oracle import oracle as O

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    wl = WORKLOADS[args.workload if args.workload in ("c3", "c3z") else "c3"]
    method = wl["method"]
    n = args.entries or wl["entries"]
    size = ENTRY_SIZE
    t_prep = time.time()
    data, hashes, ref_comp = build_corpus(n, size, rank * n, max(1, (os.cpu_count() or 1) // world))
    prep_s = time.time() - t_prep
    ctx = zpack_b200.Context(local)
    cap = ctx.pack_bound(method, size)
    slot = (cap + 15) & ~15
    f = np.zeros(n, zlib.File)
    f["src_off"] = np.arange(n, dtype=np.uint64) * size
    f["size"] = size
    f["dst_off"] = np.arange(n, dtype=np.uint64) * slot
    f["dst_cap"] = cap
    f["method"] = method
    in_size, out_size = n * size, n * slot
    h_in = torch.from_numpy(data).pin_memory()
    d_in = h_in.cuda()
    d_out = torch.empty(out_size, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        comp, dg, st = ctx.pack_device(d_in, in_size, d_out, out_size, f, stream)
    assert (st == 0).all() and np.array_equal(dg, hashes), "pack parity gate failed: status / XXH3-64 of the input"
    # validity gates: (1) every frame decodes back to its digest on the GPU reader, (2) a sample through the CPU checker
    e = np.zeros(n, zlib.Entry)
    e["src_off"], e["comp_size"], e["uncomp_size"] = f["dst_off"], comp, size
    e["dst_off"] = np.arange(n, dtype=np.uint64) * size
    e["dst_cap"], e["hash"], e["method"] = size, hashes, method
    d_back = torch.empty(in_size, dtype=torch.uint8, device="cuda")
    st2, dg2 = ctx.unpack_device(d_out, out_size, d_back, in_size, e, stream)
    assert (st2 == 0).all() and np.array_equal(dg2, hashes), "GPU-written frames do not read back"
    assert torch.equal(d_back[:64 * size], d_in[:64 * size])
    del d_back
    for i in range(0, n, max(1, n // 32)):
        fr = d_out[int(f["dst_off"][i]):int(f["dst_off"][i]) + int(comp[i])].cpu().numpy()
        rc, got, _ = O.read_entry_port(method, fr, size, size, int(hashes[i]))
        assert rc == 0 and np.array_equal(got, data[i * size:(i + 1) * size]), "CPU checker rejects a GPU-written frame"
    comp_bytes = int(comp.sum())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count
    kernel_ms, frames_ms = [], []
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        comp, dg, st = ctx.pack_device(d_in, in_size, d_out, out_size, f, stream)
        kms = ctx.last_kernel_ms()
        kernel_ms.append(kms["pack_blocks_ms"])
        frames_ms.append(kms["pack_frames_ms"])
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - launches0
    assert (st == 0).all() and np.array_equal(dg, hashes)

    e2e_s = 0.0
    if args.e2e:
        h_out = torch.empty(out_size, dtype=torch.uint8).pin_memory()
        h_in_np, h_out_np = h_in.numpy(), h_out.numpy()
        ctx.pack_host(h_in_np, in_size, h_out_np, out_size, f)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            comp3, dg3, st3 = ctx.pack_host(h_in_np, in_size, h_out_np, out_size, f)
        torch.cuda.synchronize()
        e2e_s = (time.perf_counter() - t0) / args.e2e_steps
        assert (st3 == 0).all() and np.array_equal(dg3, hashes) and np.array_equal(comp3, comp)
        for i in (0, n // 2, n - 1):   # the host copy really holds the frames
            o, c = int(f["dst_off"][i]), int(comp[i])
            assert np.array_equal(h_out_np[o:o + c], d_out[o:o + c].cpu().numpy()), "e2e output mismatch"
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms_total, float(np.mean(kernel_ms)), e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, kern_ms, e2e_s = [float(x) for x in t.cpu()]
    if rank == 0:
        peak, peak_src = peaks()
        ms_step = ms_total / args.steps
        value = world * in_size / (ms_step * 1e-3) / 1e9
        algo_bytes = in_size + comp_bytes        # the block compressor reads every input byte once and writes every payload byte once
        achieved = algo_bytes / (kern_ms * 1e-3) / 1e9
        line = {"metric": wl["metric"], "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": f"{wl['what']}, {n} files x 128 KiB per GPU ({in_size / 2**30:.2f} GiB), zpk-synth-v1",
                           "files_per_gpu": n, "file_bytes": size, "sharding": f"files x{world}, no collective; offsets assembled on the host",
                           "l2": "inputs+outputs per step exceed the 126 MB L2 (no flush needed)",
                           "pipeline": "per round of <= 1 GiB of blocks: lz4_pack_blocks_kernel (CTA per 64 KB block, block in shared memory) "
                                       "-> lz4_pack_kernel (warp per file: frame layout from the block slots + XXH3-64 of the input)",
                           "frames_kernel_ms": float(np.mean(frames_ms)),
                           "ratio_gpu": in_size / comp_bytes, "ratio_reference_level0_sampled": in_size / ref_comp,
                           "validity": "all frames read back on the GPU reader; 32 sampled frames decode bit-exactly in the CPU checker",
                           "corpus_prep_s": round(prep_s, 1)},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": None, "peak_source": peak_src, "kernel": wl["kernel"], "kernel_ms": kern_ms,
                             "algorithmic_bytes_per_launch": algo_bytes},
                "gpu_launches": int(launches), "clocks": clocks}
        if args.e2e:
            line["e2e"] = {"value": world * in_size / e2e_s / 1e9, "unit": "GB/s", "h2d_bytes_per_step": in_size + f.nbytes,
                           "d2h_bytes_per_step": comp_bytes + 20 * n,
                           "how": "zpb_pack_host, pinned host buffers: chunked H2D of every input byte / kernel / gather + D2H of every frame, "
                                  "overlapped on worker streams"}
        if world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            n_ref = min(n, args.ref_entries or 16384)       # ~0.4 s per step on 16 cores at the reference's ~5 GB/s
            v, dt, kind, ratio = cpu_pack_throughput(data, size, n_ref, cores, method, 3 if method == 1 else 0)
            v1, _, _, _ = cpu_pack_throughput(data, size, min(n, 1024), 1, method, 3 if method == 1 else 0)
            line["cpu_baseline"] = {"value": v, "unit": "GB/s", "cores": cores, "kind": kind, "ratio": ratio,
                                    "sample": f"first {n_ref} files, {cores} independent writers "
                                              f"(zpack_write_archive, {'zstd level 3' if method == 1 else 'LZ4 level 0'}); single writer: {v1:.3f} GB/s"}
        _emit(args, line)
    if world > 1 and not getattr(args, "nested", False):
        dist.destroy_process_group()
    ctx.close()


# dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from one `ncu --set full` capture, as a ratio
# to the algorithmic bytes of the captured launch (the capture runs fewer entries than the bench; the ratio carries over)
NCU_TRAFFIC_RATIO = {
    "c2": (7.0606 / (12297207239 * 28416 / 65536 / 1e9), "profiles/r2_ncu_full_exec_mixed28416.csv: 3.357 + 3.704 GB for 28 416 entries"),
}


def archive_block(n=16384):
    """The container level on the device (SURVEY §8(f) rows 1 and 4) for the `configs` block: archive build from pack-shaped
    slots (offset table + directory kernels, payload copy kernel), directory parse, archive-to-archive copy of every second
    entry.  Kernel times are the library's CUDA events around its own launches; the gate: the directory bytes equal the host
    mirror's, the parsed table equals the table that was built, sampled payloads equal their slots."""
    import torch
    import zpack_b200
    from zpack_b200 import container
    from zpack_b200.lib import ArcEntry
    hbm, _ = peaks()
    ctx = zpack_b200.Context(int(os.environ.get("LOCAL_RANK", "0")))
    rng = np.random.default_rng(3)
    comp = rng.integers(30000, 84000, n).astype(np.uint64)
    names = [f"dir{i % 64:02d}/entry_{i:07d}.bin" for i in range(n)]
    blob = np.frombuffer("".join(names).encode(), np.uint8)
    e = np.zeros(n, ArcEntry)
    e["comp_size"], e["uncomp_size"], e["hash"], e["method"] = comp, ENTRY_SIZE, rng.integers(0, 2**63, n).astype(np.uint64), 2
    e["name_len"] = [len(x) for x in names]
    e["name_off"] = np.concatenate([[0], np.cumsum(e["name_len"])[:-1]])
    cap = (comp + np.uint64(32768 + 15)) & ~np.uint64(15)
    e["src_off"] = np.concatenate([[0], np.cumsum(cap)[:-1]])
    src_size = int(cap.sum())
    d_src = torch.randint(0, 256, (src_size,), dtype=torch.uint8, device="cuda")
    total = 10 + int(comp.sum()) + 20 + 35 * n + len(blob) + 12
    d_arch = torch.empty(total + 64, dtype=torch.uint8, device="cuda")
    best = None
    for it in range(5):
        size = ctx.archive_build_device(d_src, src_size, e, blob, d_arch, total + 64)
        ms = ctx.last_archive_ms()
        if it >= 2 and (best is None or ms[1] < best[1]):
            best = ms
    assert size == total
    cdr_off = 10 + int(comp.sum())
    want_cdr = container.cdr_bytes(names, e["offset"], comp, e["uncomp_size"], e["hash"], e["method"])
    got_cdr = d_arch[cdr_off:cdr_off + len(want_cdr)].cpu().numpy()
    assert bytes(got_cdr) == want_cdr, "directory differs from the host mirror"
    for i in rng.integers(0, n, 48):
        a, b, k = int(e["offset"][i]), int(e["src_off"][i]), int(comp[i])
        assert torch.equal(d_arch[a:a + k], d_src[b:b + k]), "payload differs from its slot"
    for it in range(3):
        res, eo, nb = ctx.archive_open_device(d_arch, size)
    open_ms = ctx.last_archive_ms()[2]
    assert res == 0 and np.array_equal(eo["hash"], e["hash"]) and np.array_equal(eo["offset"], e["offset"])
    sub = np.ascontiguousarray(eo[::2])
    d_new = torch.empty(total + 64, dtype=torch.uint8, device="cuda")
    for it in range(3):
        ctx.archive_build_device(d_arch, size, sub, nb, d_new, total + 64)
    a2a = ctx.last_archive_ms()
    moved, moved2 = 2 * int(comp.sum()), 2 * int(sub["comp_size"].sum())
    launches = ctx.launch_count
    ctx.close()
    return {"workload": f"device-resident archive of {n} entries ({int(comp.sum()) / 1e9:.2f} GB of payload): build from pack slots, "
                        "directory parse, archive-to-archive copy of every second entry",
            "metric": "archive_copy_read_plus_write_GBps", "value": round(moved / best[1] / 1e6, 1), "unit": "GB/s",
            "kernel": "arc_copy_kernel", "roofline_frac": round(moved / best[1] / 1e6 / hbm, 3),
            "copy_ms": round(best[1], 4), "offset_table_and_directory_ms": round(best[0], 4), "directory_parse_ms": round(open_ms, 4),
            "archive_to_archive_GBps": round(moved2 / a2a[1] / 1e6, 1), "gpu_launches": int(launches)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS),
                    help="c2 (default): the config BASELINE.json's metric is quoted on; c3: LZ4 pack of the same corpus; c4: zstd level-3 unpack; "
                         "c5: one entry of gpus x 2 GiB sharded by independent blocks")
    ap.add_argument("--entries", type=int, default=0, help="entries per GPU (default: C2 65536 / C4 32768, x 128 KiB)")
    ap.add_argument("--independent", action="store_true", help="archive with B.Indep=1 frames (what the GPU packer writes)")
    ap.add_argument("--group", type=int, default=0)
    ap.add_argument("--no-e2e", dest="e2e", action="store_false")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-entries", type=int, default=32768)
    ap.add_argument("--ref-entries", type=int, default=0, help="entries of the reference arm's archive (default: the workload's own count)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): ONE archive cut over the ranks; weak: one archive of --entries per rank")
    ap.add_argument("--no-configs", dest="configs", action="store_false",
                    help="skip the C3 / C4 / C5 block that the default single-GPU C2 line carries")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (per-entry status, XXH3-64 digest, a seeded "
                         "sample of the decoded bytes) as DIR/<name>.npy; c2 and c4 only")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.workload not in ("c2", "c4")):
        ap.error("--dump-outputs is implemented for --impl ours with --workload c2 or c4")
    if args.impl == "reference":
        run_reference(args)
        return
    runner = {"c5": run_c5, "c3": run_c3, "c3z": run_c3}.get(args.workload, run_ours)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not (args.workload == "c2" and args.configs and world == 1 and not args.entries):
        runner(args)
        return
    # The default single-GPU line: C2 (the configuration the metric is quoted on), and — measured in this same process
    # after C2's timed region, at reduced sizes so that the whole run stays within minutes — the other BASELINE
    # configurations the GPU path covers, so that the driver's record holds them too.
    import copy
    args.nested = True
    runner(args)
    line = args.result
    block = {}
    for key, fn, n_small, what in (("c3", run_c3, 16384, "LZ4 pack, 16384 files x 128 KiB (2 GiB)"),
                                   ("c3z", run_c3, 8192, "zstd pack, 8192 files x 128 KiB (1 GiB): the LZ4 block compressor's matches as zstd blocks"),
                                   ("c4", run_ours, 8192, "zstd level-3 unpack + verify, 8192 entries x 128 KiB (1 GiB), frames written by the reference"),
                                   ("c5", run_c5, 16384, "one LZ4 entry of 16384 independent 64 KB blocks (1 GiB), block-sharded read")):
        sub = copy.copy(args)
        sub.workload, sub.entries, sub.warmup, sub.no_cpu, sub.e2e_steps, sub.result = key, n_small, 3, True, 2, None
        sub.dump_outputs = None
        try:
            fn(sub)
            r = sub.result
            block[key] = {"workload": what, "metric": r["metric"], "value": r["value"], "unit": r["unit"], "ms_per_step": r["ms_per_step"],
                          "roofline_frac": r.get("roofline", {}).get("frac"), "kernel": r.get("roofline", {}).get("kernel"),
                          "e2e": (r.get("e2e") or {}).get("value"), "gpu_launches": r.get("gpu_launches"),
                          **({"ratio": r["config"].get("ratio")} if isinstance(r.get("config"), dict) and "ratio" in r["config"] else {}),
                          **({"ratio_gpu": r["config"].get("ratio_gpu")} if isinstance(r.get("config"), dict) and "ratio_gpu" in r["config"] else {})}
        except Exception as ex:   # a configuration that cannot run here (e.g. no oracle/_ref for the zstd archive) says so
            block[key] = {"workload": what, "unavailable": f"{type(ex).__name__}: {ex}"[:300]}
    try:
        block["archive"] = archive_block()
    except Exception as ex:
        block["archive"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
    line["configs"] = block
    print(json.dumps(line))


if __name__ == "__main__":
    main()
