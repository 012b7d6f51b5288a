"""ctypes binding of include/zpack_b200.h — the C-ABI the reference's host loops are rerouted to.

Mirrors the argument meaning of the reference calls it stands in for
(/root/reference/lib/zpack_read.c:326 zpack_read_file, lib/zpack_write.c:280 zpack_write_files).
Fails loudly when the CUDA library has not been built or no GPU is present: there is no fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ZPB_LIB") or os.path.join(_HERE, "libzpack_b200.so")  # ZPB_LIB: developer builds (profiling)

METHOD_NONE, METHOD_ZSTD, METHOD_LZ4 = 0, 1, 2
F_NO_VERIFY = 1
F_DISCARD = 2

# enum zpack_result values the hot path can return (/root/reference/lib/zpack.h:189-218)
ST_OK = 0
ST_BUFFER_TOO_SMALL = 12
ST_DECOMPRESS_FAILED = 13
ST_COMPRESS_FAILED = 14
ST_HASH_MISMATCH = 15
ST_OFFSET_INVALID = 16
ST_FILE_INCOMPLETE = 17
ST_FILE_SIZE_INVALID = 18
ST_METHOD_INVALID = 19
ST_NOT_AVAILABLE = 24

#: numpy dtype of `struct zpb_entry` (64 bytes)
Entry = np.dtype(
    [("src_off", "<u8"), ("comp_size", "<u8"), ("dst_off", "<u8"), ("dst_cap", "<u8"),
     ("uncomp_size", "<u8"), ("hash", "<u8"), ("method", "<u4"), ("flags", "<u4"), ("reserved", "<u8")]
)
#: numpy dtype of `struct zpb_file` (64 bytes)
File = np.dtype(
    [("src_off", "<u8"), ("size", "<u8"), ("dst_off", "<u8"), ("dst_cap", "<u8"),
     ("method", "<u4"), ("level", "<i4"), ("reserved", "<u8", (3,))]
)
#: numpy dtype of `struct zpb_block` (16 bytes)
Block = np.dtype([("src_off", "<u8"), ("comp_size", "<u4"), ("flags", "<u4")])
BLK_STORED = 1
BLK_ZSTD = 2
INDEX_UNSUPPORTED = 1
#: ZPB_ZSTD_FRAMED_MIN: zstd files of at least this many bytes are written as one frame per 64 KB (zstd_frame_index)
ZSTD_FRAMED_MIN = 4 << 20
#: numpy dtype of `struct zpb_arc_entry` (64 bytes): one row of a device-resident archive's directory
ArcEntry = np.dtype(
    [("src_off", "<u8"), ("comp_size", "<u8"), ("uncomp_size", "<u8"), ("hash", "<u8"), ("name_off", "<u8"),
     ("name_len", "<u4"), ("method", "<u4"), ("offset", "<u8"), ("reserved", "<u8")]
)
assert Entry.itemsize == 64 and File.itemsize == 64 and Block.itemsize == 16 and ArcEntry.itemsize == 64

EXPORTS = [
    "zpb_abi_version", "zpb_create", "zpb_destroy", "zpb_last_error", "zpb_device_info",
    "zpb_launch_count", "zpb_unpack_device", "zpb_unpack_device_async", "zpb_unpack_host", "zpb_xxh3_device", "zpb_xxh3_host",
    "zpb_pack_bound", "zpb_pack_device", "zpb_pack_host", "zpb_last_kernel_ms", "zpb_last_pack_stage_ms", "zpb_set_tuning",
    "zpb_last_stage_ms", "zpb_set_fast_path", "zpb_set_overlap", "zpb_set_lz4hc", "zpb_set_zstd_entropy", "zpb_last_zstd_ms",
    "zpb_lz4_frame_index", "zpb_zstd_frame_index", "zpb_unpack_blocks_device", "zpb_blocks_digest", "zpb_last_chain_ms",
    "zpb_unpack_entry_blocks_host", "zpb_device_count",
    "zpb_archive_open_device", "zpb_archive_build_device", "zpb_copy_entries_device", "zpb_last_archive_ms",
    "zpb_file_read_device", "zpb_file_write_device",
]


class ZpbError(RuntimeError):
    pass


_lib = None


def load_library(path: str = LIB_PATH) -> C.CDLL:
    """dlopen the CUDA library; raises if it is missing (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise ZpbError(f"{path} not built — run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(path)
    vp, u64, i32p, u64p = C.c_void_p, C.c_uint64, C.POINTER(C.c_int32), C.POINTER(C.c_uint64)
    lib.zpb_abi_version.restype = C.c_int
    lib.zpb_create.restype = vp
    lib.zpb_create.argtypes = [C.c_int]
    lib.zpb_destroy.argtypes = [vp]
    lib.zpb_last_error.restype = C.c_char_p
    lib.zpb_last_error.argtypes = [vp]
    lib.zpb_device_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.zpb_launch_count.restype = u64
    lib.zpb_launch_count.argtypes = [vp]
    lib.zpb_set_tuning.argtypes = [vp, C.c_int, C.c_int]
    lib.zpb_unpack_device.argtypes = [vp, vp, u64, vp, u64, vp, u64, vp, vp, vp]
    lib.zpb_unpack_device_async.argtypes = [vp, vp, u64, vp, u64, vp, u64, vp, vp, vp]
    lib.zpb_unpack_host.argtypes = [vp, vp, u64, vp, u64, vp, u64, vp, vp]
    lib.zpb_xxh3_device.argtypes = [vp, vp, vp, vp, u64, vp, vp]
    lib.zpb_xxh3_host.argtypes = [vp, vp, u64, vp]
    lib.zpb_pack_bound.restype = u64
    lib.zpb_pack_bound.argtypes = [C.c_uint32, u64]
    lib.zpb_pack_device.argtypes = [vp, vp, u64, vp, u64, vp, u64, vp, vp, vp, vp]
    lib.zpb_pack_host.argtypes = [vp, vp, u64, vp, u64, vp, u64, vp, vp, vp]
    lib.zpb_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.zpb_last_pack_stage_ms.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.zpb_last_stage_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.zpb_set_fast_path.argtypes = [vp, C.c_int]
    lib.zpb_set_overlap.argtypes = [vp, C.c_int]
    lib.zpb_set_lz4hc.argtypes = [vp, C.c_int]
    lib.zpb_set_zstd_entropy.argtypes = [vp, C.c_int]
    lib.zpb_last_zstd_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.zpb_lz4_frame_index.argtypes = [vp, u64, u64, vp, u64, u64p, C.POINTER(C.c_uint32), u64p]
    lib.zpb_zstd_frame_index.argtypes = [vp, u64, u64, vp, u64, u64p, u64p]
    lib.zpb_unpack_blocks_device.argtypes = [vp, vp, u64, vp, u64, vp, u64, C.c_uint32, u64, i32p, vp]
    lib.zpb_blocks_digest.argtypes = [vp, vp, vp, u64, u64, vp, u64p, vp]
    lib.zpb_last_chain_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.zpb_unpack_entry_blocks_host.argtypes = [vp, vp, u64, vp, u64, u64, u64, C.c_uint32, i32p, u64p]
    lib.zpb_group_create.restype = vp
    lib.zpb_group_create.argtypes = [vp, C.c_int]
    lib.zpb_group_destroy.argtypes = [vp]
    lib.zpb_group_size.argtypes = [vp]
    lib.zpb_group_last_error.restype = C.c_char_p
    lib.zpb_group_last_error.argtypes = [vp]
    lib.zpb_group_partition.argtypes = [vp, u64, C.c_int, vp, vp]
    lib.zpb_group_unpack_host.argtypes = [vp, vp, u64, vp, u64, vp, u64, vp, vp]
    lib.zpb_group_pack_host.argtypes = [vp, vp, u64, vp, u64, vp, u64, vp, vp, vp]
    lib.zpb_group_last_ms.argtypes = [vp, C.POINTER(C.c_float), C.c_int]
    lib.zpb_archive_open_device.argtypes = [vp, vp, u64, vp, u64, u64p, vp, u64, u64p, i32p, vp]
    lib.zpb_archive_build_device.argtypes = [vp, vp, u64, vp, u64, vp, u64, vp, u64, u64p, vp]
    lib.zpb_copy_entries_device.argtypes = [vp, vp, u64, vp, u64, vp, u64, vp]
    lib.zpb_last_archive_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.zpb_file_read_device.argtypes = [vp, C.c_int, u64, u64, vp]
    lib.zpb_file_write_device.argtypes = [vp, C.c_int, u64, u64, vp]
    lib.zpb_host_alloc.restype = vp
    lib.zpb_host_alloc.argtypes = [u64]
    lib.zpb_host_free.argtypes = [vp]
    _lib = lib
    return lib


def group_partition(entries: np.ndarray, world: int):
    """zpb_group_partition: (order, cuts) — device k takes entries[order[cuts[k]:cuts[k+1]]] (host logic, no GPU needed)."""
    lib = load_library()
    assert entries.dtype == Entry and entries.flags.c_contiguous
    order = np.zeros(len(entries), np.uint64)
    cuts = np.zeros(world + 1, np.uint64)
    rc = lib.zpb_group_partition(entries.ctypes.data, len(entries), world, order.ctypes.data, cuts.ctypes.data)
    if rc != 0:
        raise ZpbError(f"zpb_group_partition: {rc}")
    return order, cuts


class Group:
    """Several GPUs of one box behind one call (`zpb_group`): entries cut into contiguous runs balanced by decoded bytes,
    one run per device, each on its own host thread; no collective."""

    def __init__(self, devices=None):
        self.lib = load_library()
        if devices is None:
            self.h = self.lib.zpb_group_create(None, 0)
        else:
            arr = (C.c_int * len(devices))(*devices)
            self.h = self.lib.zpb_group_create(arr, len(devices))
        if not self.h:
            raise ZpbError("zpb_group_create failed: " + self.lib.zpb_last_error(None).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.zpb_group_destroy(self.h)
            self.h = None

    __del__ = close

    @property
    def size(self) -> int:
        return self.lib.zpb_group_size(self.h)

    def _check(self, rc):
        if rc != 0:
            raise ZpbError(f"zpb error {rc}: {self.lib.zpb_group_last_error(self.h).decode()}")

    def unpack_host(self, h_archive, archive_size: int, h_out, out_size: int, entries: np.ndarray):
        assert entries.dtype == Entry and entries.flags.c_contiguous
        n = len(entries)
        status, digest = np.zeros(n, np.int32), np.zeros(n, np.uint64)
        self._check(self.lib.zpb_group_unpack_host(self.h, _ptr(h_archive), archive_size, _ptr(h_out), out_size,
                                                   entries.ctypes.data, n, status.ctypes.data, digest.ctypes.data))
        return status, digest

    def pack_host(self, h_in, in_size: int, h_out, out_size: int, files: np.ndarray):
        assert files.dtype == File and files.flags.c_contiguous
        n = len(files)
        comp, digest, status = np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.int32)
        self._check(self.lib.zpb_group_pack_host(self.h, _ptr(h_in), in_size, _ptr(h_out), out_size, files.ctypes.data, n,
                                                 comp.ctypes.data, digest.ctypes.data, status.ctypes.data))
        return comp, digest, status

    def last_ms(self):
        a = (C.c_float * 16)()
        self.lib.zpb_group_last_ms(self.h, a, 16)
        return [float(a[k]) for k in range(self.size)]


def _ptr(a) -> int:
    """address of a numpy array / torch tensor / raw int pointer"""
    if a is None:
        return 0
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    raise TypeError(type(a))


def lz4_frame_index(frame: np.ndarray, archive_off: int = 0):
    """Host-side framing walk of one block-independent LZ4 frame (no GPU needed, no codec work):
    returns (blocks: Block[n], block_size, content_size or None), or None when the frame is not a single
    checksum-free B.Indep frame of 64 KB blocks (zpb_lz4_frame_index -> ZPB_INDEX_UNSUPPORTED)."""
    lib = load_library()
    frame = np.ascontiguousarray(frame, np.uint8)
    n, bs, cs = C.c_uint64(), C.c_uint32(), C.c_uint64()
    cap = len(frame) // 5 + 2   # every block costs at least 4 header bytes + 1 payload byte
    blocks = np.zeros(cap, Block)
    rc = lib.zpb_lz4_frame_index(frame.ctypes.data, len(frame), archive_off, blocks.ctypes.data, cap,
                                 C.byref(n), C.byref(bs), C.byref(cs))
    if rc == INDEX_UNSUPPORTED:
        return None
    if rc != 0:
        raise ZpbError(f"zpb_lz4_frame_index: {rc}")
    return blocks[:n.value].copy(), bs.value, (None if cs.value == 2**64 - 1 else cs.value)


def zstd_frame_index(entry: np.ndarray, archive_off: int = 0):
    """Host-side framing walk of a zstd entry written as 64 KB frames (no GPU needed, no codec work): returns
    (frames: Block[n] with flags BLK_ZSTD, content_size), or None when the entry does not have that shape
    (zpb_zstd_frame_index -> ZPB_INDEX_UNSUPPORTED)."""
    lib = load_library()
    entry = np.ascontiguousarray(entry, np.uint8)
    n, cs = C.c_uint64(), C.c_uint64()
    cap = len(entry) // 9 + 1   # every frame costs at least a 6-byte header + a 3-byte block header
    frames = np.zeros(cap, Block)
    rc = lib.zpb_zstd_frame_index(entry.ctypes.data, len(entry), archive_off, frames.ctypes.data, cap,
                                  C.byref(n), C.byref(cs))
    if rc == INDEX_UNSUPPORTED:
        return None
    if rc != 0:
        raise ZpbError(f"zpb_zstd_frame_index: {rc}")
    return frames[:n.value].copy(), cs.value


class Context:
    """One GPU context (`zpb_ctx`): scratch arenas, a stream, CUDA-event timers."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        self.h = self.lib.zpb_create(device)
        if not self.h:
            raise ZpbError("zpb_create failed: " + self.lib.zpb_last_error(None).decode())
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.zpb_destroy(self.h)
            self.h = None

    __del__ = close

    def _check(self, rc: int):
        if rc != 0:
            raise ZpbError(f"zpb error {rc}: {self.lib.zpb_last_error(self.h).decode()}")

    def device_info(self):
        sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
        self._check(self.lib.zpb_device_info(self.h, C.byref(sm), C.byref(ma), C.byref(mi)))
        return {"sm_count": sm.value, "cc": (ma.value, mi.value)}

    def set_tuning(self, group_lanes: int = 0, ctas_per_sm: int = -1):
        self._check(self.lib.zpb_set_tuning(self.h, group_lanes, ctas_per_sm))

    def set_fast_path(self, enabled: bool):
        """False: every entry goes through the general decoder (A/B runs, tests of that kernel)."""
        self._check(self.lib.zpb_set_fast_path(self.h, int(enabled)))

    def set_overlap(self, enabled: bool):
        """False: scan, parse and execute run back to back on one stream (per-kernel timings are then meaningful)."""
        self._check(self.lib.zpb_set_overlap(self.h, int(enabled)))

    def set_lz4hc(self, enabled: bool):
        """True: LZ4 files of level >= 3 are compressed by the HC block compressor (levels above 12 act as 12);
        False (the default unless ZPB_LZ4HC=1 was set when the context was created): they get ST_NOT_AVAILABLE."""
        self._check(self.lib.zpb_set_lz4hc(self.h, int(enabled)))

    def set_zstd_entropy(self, enabled: bool):
        """True: zstd files also Huffman-code literals with byte values above 128 (FSE-compressed weights) where that
        pays, and blocks the LZ4 block compressor stores become Huffman-only Compressed_Blocks where that is smaller.
        False (the default unless ZPB_ZSTD_ENTROPY=1 was set when the context was created): today's frames."""
        self._check(self.lib.zpb_set_zstd_entropy(self.h, int(enabled)))

    def last_stage_ms(self):
        a = (C.c_float * 4)()
        self.lib.zpb_last_stage_ms(self.h, a)
        z = C.c_float()
        self.lib.zpb_last_zstd_ms(self.h, C.byref(z))
        return {"scan_ms": a[0], "parse_ms": a[1], "exec_ms": a[2], "general_ms": a[3], "zstd_ms": z.value}

    @property
    def launch_count(self) -> int:
        return int(self.lib.zpb_launch_count(self.h))

    def last_kernel_ms(self):
        a, b = C.c_float(), C.c_float()
        self.lib.zpb_last_kernel_ms(self.h, C.byref(a), C.byref(b))
        c, d = C.c_float(), C.c_float()
        self.lib.zpb_last_pack_stage_ms(self.h, C.byref(c), C.byref(d))
        return {"unpack_ms": a.value, "pack_ms": b.value, "pack_blocks_ms": c.value, "pack_frames_ms": d.value}

    # ---- unpack + verify -------------------------------------------------------------------
    def unpack_device(self, d_archive, archive_size: int, d_out, out_size: int, entries: np.ndarray,
                      stream: int = 0):
        """Archive and output resident in HBM (torch tensors or raw device pointers)."""
        assert entries.dtype == Entry and entries.flags.c_contiguous
        n = len(entries)
        status = np.empty(n, np.int32)
        digest = np.empty(n, np.uint64)
        self._check(self.lib.zpb_unpack_device(self.h, _ptr(d_archive), archive_size, _ptr(d_out), out_size,
                                               _ptr(entries), n, _ptr(status), _ptr(digest), stream))
        return status, digest

    def unpack_device_async(self, d_archive, archive_size: int, d_out, out_size: int, entries: np.ndarray, d_status,
                            d_digest, stream: int = 0) -> None:
        """Enqueue unpack_device's work on `stream` (a cudaStream_t, e.g. torch.cuda.current_stream().cuda_stream) and
        return without waiting for the GPU.  d_status (int32[n]) and d_digest (uint64[n], e.g. a torch.int64 tensor) are
        device buffers (torch tensors or raw pointers) that receive unpack_device's results in stream order; `entries`
        may be reused as soon as the call returns."""
        assert entries.dtype == Entry and entries.flags.c_contiguous
        self._check(self.lib.zpb_unpack_device_async(self.h, _ptr(d_archive), archive_size, _ptr(d_out), out_size,
                                                     _ptr(entries), len(entries), _ptr(d_status), _ptr(d_digest),
                                                     stream))

    def unpack_host(self, h_archive, archive_size: int, h_out, out_size: int, entries: np.ndarray):
        """Host buffers in, host buffers out (H2D + kernels + D2H inside the call)."""
        assert entries.dtype == Entry and entries.flags.c_contiguous
        n = len(entries)
        status = np.empty(n, np.int32)
        digest = np.empty(n, np.uint64)
        self._check(self.lib.zpb_unpack_host(self.h, _ptr(h_archive), archive_size, _ptr(h_out), out_size,
                                             _ptr(entries), n, _ptr(status), _ptr(digest)))
        return status, digest

    # ---- one large entry, sharded by blocks (C5) ------------------------------------------------
    def unpack_blocks_device(self, d_archive, archive_size: int, d_out, out_size: int, blocks: np.ndarray,
                             block_size: int, shard_uncomp_size: int, stream: int = 0) -> int:
        """Decode a contiguous run of one entry's independent blocks (LZ4) or frames (zstd, flags BLK_ZSTD; block_size
        65536); returns the shard status."""
        assert blocks.dtype == Block and blocks.flags.c_contiguous
        st = C.c_int32(-1)
        self._check(self.lib.zpb_unpack_blocks_device(self.h, _ptr(d_archive), archive_size, _ptr(d_out), out_size,
                                                      _ptr(blocks), len(blocks), block_size, shard_uncomp_size,
                                                      C.byref(st), stream))
        self._blk_uncomp = shard_uncomp_size if st.value == 0 else None
        return st.value

    def blocks_digest(self, acc_in: Optional[np.ndarray], shard_pos: int, total_size: int, d_out=None,
                      stream: int = 0):
        """XXH3 chain over the last decoded shard.  Returns (acc_out: uint64[8], digest or None)."""
        acc_out = np.empty(8, np.uint64)
        dg = C.c_uint64(0)
        if acc_in is not None:
            acc_in = np.ascontiguousarray(acc_in, np.uint64)
            assert acc_in.shape == (8,)
        self._check(self.lib.zpb_blocks_digest(self.h, _ptr(acc_in), _ptr(acc_out), shard_pos, total_size,
                                               _ptr(d_out), C.byref(dg), stream))
        final = shard_pos + (getattr(self, "_blk_uncomp", None) or 0) == total_size
        return acc_out, (dg.value if final else None)

    def unpack_entry_blocks_host(self, h_entry, comp_size: int, h_out, out_cap: int, uncomp_size: int,
                                 expect_hash: int, flags: int = 0):
        """One large block-independent LZ4 entry, or one zstd entry of 64 KB frames (what pack_* writes from
        ZSTD_FRAMED_MIN on), host buffers (pipelined chunks + XXH3 relay).  The index is chosen by the entry's magic
        number.  Returns (status, digest), or None when the entry is not eligible for the block path."""
        st, dg = C.c_int32(-1), C.c_uint64(0)
        rc = self.lib.zpb_unpack_entry_blocks_host(self.h, _ptr(h_entry), comp_size, _ptr(h_out), out_cap,
                                                   uncomp_size, expect_hash, flags, C.byref(st), C.byref(dg))
        if rc == INDEX_UNSUPPORTED:
            return None
        self._check(rc)
        return st.value, dg.value

    def last_chain_ms(self) -> float:
        a = C.c_float()
        self.lib.zpb_last_chain_ms(self.h, C.byref(a))
        return a.value

    # ---- digest ------------------------------------------------------------------------------
    def xxh3_host(self, data) -> int:
        buf = np.frombuffer(data, np.uint8) if not isinstance(data, np.ndarray) else data
        out = C.c_uint64()
        self._check(self.lib.zpb_xxh3_host(self.h, _ptr(buf) if len(buf) else 0, len(buf), C.byref(out)))
        return out.value

    def xxh3_device(self, d_data, offsets: Sequence[int], lengths: Sequence[int], stream: int = 0):
        off = np.ascontiguousarray(offsets, np.uint64)
        ln = np.ascontiguousarray(lengths, np.uint64)
        out = np.empty(len(off), np.uint64)
        self._check(self.lib.zpb_xxh3_device(self.h, _ptr(d_data), _ptr(off), _ptr(ln), len(off), _ptr(out), stream))
        return out

    # ---- the container level on the device ------------------------------------------------------
    def archive_open_device(self, d_archive, archive_size: int, want_names: bool = True, stream: int = 0):
        """(zpack_result, ArcEntry table, directory block that name_off points into) of the archive image in HBM."""
        n, nsz, res = C.c_uint64(), C.c_uint64(), C.c_int32(-1)
        rc = self.lib.zpb_archive_open_device(self.h, _ptr(d_archive), archive_size, None, 0, C.byref(n), None, 0, C.byref(nsz),
                                              C.byref(res), stream)
        if rc == 0:                      # refused by the fixed fields, or an empty archive
            return res.value, np.zeros(0, ArcEntry), np.zeros(0, np.uint8)
        if n.value == 0:
            self._check(rc)
        entries = np.zeros(n.value, ArcEntry)
        names = np.zeros(nsz.value if want_names else 0, np.uint8)
        self._check(self.lib.zpb_archive_open_device(self.h, _ptr(d_archive), archive_size, _ptr(entries), len(entries), C.byref(n),
                                                     _ptr(names) if want_names else None, len(names), C.byref(nsz), C.byref(res), stream))
        if res.value != 0:
            return res.value, np.zeros(0, ArcEntry), np.zeros(0, np.uint8)
        return 0, entries, names

    def archive_build_device(self, d_src, src_size: int, entries: np.ndarray, names: np.ndarray, d_archive, archive_cap: int,
                             stream: int = 0) -> int:
        """Header + payloads (from d_src + src_off, table order) + CDR + EOCDR into d_archive; fills entries['offset']."""
        assert entries.dtype == ArcEntry and entries.flags.c_contiguous
        names = np.ascontiguousarray(names, np.uint8)
        size = C.c_uint64()
        self._check(self.lib.zpb_archive_build_device(self.h, _ptr(d_src) if d_src is not None else None, src_size, _ptr(entries), len(entries),
                                                      _ptr(names) if len(names) else None, len(names), _ptr(d_archive), archive_cap,
                                                      C.byref(size), stream))
        return size.value

    def copy_entries_device(self, d_src, src_size: int, d_dst, dst_size: int, entries: np.ndarray, stream: int = 0):
        assert entries.dtype == ArcEntry and entries.flags.c_contiguous
        self._check(self.lib.zpb_copy_entries_device(self.h, _ptr(d_src), src_size, _ptr(d_dst), dst_size, _ptr(entries), len(entries), stream))

    def file_read_device(self, fd: int, file_off: int, size: int, d_dst):
        self._check(self.lib.zpb_file_read_device(self.h, fd, file_off, size, _ptr(d_dst)))

    def file_write_device(self, fd: int, file_off: int, size: int, d_src):
        self._check(self.lib.zpb_file_write_device(self.h, fd, file_off, size, _ptr(d_src)))

    def last_archive_ms(self):
        ms = (C.c_float * 3)()
        self._check(self.lib.zpb_last_archive_ms(self.h, ms))
        return tuple(float(x) for x in ms)

    # ---- pack --------------------------------------------------------------------------------
    def pack_bound(self, method: int, size: int) -> int:
        return int(self.lib.zpb_pack_bound(method, size))

    def pack_device(self, d_in, in_size: int, d_out, out_size: int, files: np.ndarray, stream: int = 0):
        assert files.dtype == File and files.flags.c_contiguous
        n = len(files)
        comp = np.empty(n, np.uint64)
        digest = np.empty(n, np.uint64)
        status = np.empty(n, np.int32)
        self._check(self.lib.zpb_pack_device(self.h, _ptr(d_in), in_size, _ptr(d_out), out_size, _ptr(files), n,
                                             _ptr(comp), _ptr(digest), _ptr(status), stream))
        return comp, digest, status

    def pack_host(self, h_in, in_size: int, h_out, out_size: int, files: np.ndarray):
        assert files.dtype == File and files.flags.c_contiguous
        n = len(files)
        comp = np.empty(n, np.uint64)
        digest = np.empty(n, np.uint64)
        status = np.empty(n, np.int32)
        self._check(self.lib.zpb_pack_host(self.h, _ptr(h_in), in_size, _ptr(h_out), out_size, _ptr(files), n,
                                           _ptr(comp), _ptr(digest), _ptr(status)))
        return comp, digest, status
