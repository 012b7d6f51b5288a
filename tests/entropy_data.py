"""Data with few repeats and a skewed byte distribution, the kind the zstd writer's entropy switch is for
(zpb_set_zstd_entropy): tensors in bf16 / fp16 / fp32, int8 quantised data, and int8 with inserted repeats so that the
LZ4 block compressor keeps the block and its literals take values on both sides of 128.  Also the order-0 Huffman bound
per 64 KB block that the tests and tools/zstd_entropy_bench.py hold the writer's ratio to."""
import heapq

import numpy as np

CLASSES = ("bf16", "fp16", "fp32", "int8", "int8rep")
HEADER_BYTES = 420          # per 64 KB block in the bound: block headers, literal section headers, jump tables, the tree


def class_bytes(name: str, size: int, seed: int = 0) -> np.ndarray:
    """`size` bytes of class `name`, deterministic in (name, seed)."""
    rng = np.random.default_rng([CLASSES.index(name), seed])
    if name == "bf16":
        x = rng.normal(0.0, 0.02, (size + 1) // 2).astype(np.float32)
        b = (x.view(np.uint32) >> 16).astype(np.uint16).view(np.uint8)
    elif name == "fp16":
        b = rng.normal(0.0, 1.0, (size + 1) // 2).astype(np.float16).view(np.uint8)
    elif name == "fp32":
        b = rng.normal(0.0, 0.02, (size + 3) // 4).astype(np.float32).view(np.uint8)
    else:
        b = np.clip(np.rint(rng.laplace(0.0, 6.0, size)), -128, 127).astype(np.int8).view(np.uint8)
        if name == "int8rep":       # every 160 bytes, a copy of 48 earlier bytes from up to 16 KB back
            for p in range(4096, size - 48, 160):
                d = int(rng.integers(64, min(p, 16384)))
                b[p:p + 48] = b[p - d:p - d + 48]
    return np.ascontiguousarray(b[:size])


def huffman_lengths(hist) -> dict:
    """Code lengths of an (unlimited) Huffman code for the symbols with a nonzero count."""
    heap = [(int(c), s, [s]) for s, c in enumerate(hist) if c]
    if len(heap) == 1:
        return {heap[0][1]: 1}
    heapq.heapify(heap)
    depth = {s: 0 for _, s, _ in heap}
    while len(heap) > 1:
        c1, k1, l1 = heapq.heappop(heap)
        c2, k2, l2 = heapq.heappop(heap)
        for s in l1 + l2:
            depth[s] += 1
        heapq.heappush(heap, (c1 + c2, min(k1, k2), l1 + l2))
    return depth


def huffman_bound(data: np.ndarray) -> float:
    """Ratio of an order-0 Huffman code per 64 KB block with HEADER_BYTES per block (a block that does not shrink stays raw)."""
    data = np.asarray(data, np.uint8)
    total = 0
    for o in range(0, len(data), 65536):
        blk = data[o:o + 65536]
        hist = np.bincount(blk, minlength=256)
        lens = huffman_lengths(hist)
        coded = sum(int(hist[s]) * l for s, l in lens.items()) / 8 + HEADER_BYTES
        total += min(coded, len(blk))
    return len(data) / total if total else 1.0
