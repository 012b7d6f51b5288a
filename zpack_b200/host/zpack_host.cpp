// zpack_host.cpp — libzpack.so: the lib/zpack.h API of the reference, backed by the GPU C-ABI.
//
// Host side of the drop-in (C++ because the reference's host side is compiled C and its toolchain's
// build system is not used here).  Container framing — header, data signature, central directory,
// EOCDR (docs/specs.md; lib/zpack_read.c:33-296, lib/zpack_write.c:36-123,687-829) — stays on the
// host, as the north-star asks; every per-entry (de)compression and digest goes through
// include/zpack_b200.h.  There is no CPU codec in this file: if the GPU library cannot create a
// context, the entry points that need it return ZPACK_ERROR_MALLOC_FAILED, as the reference does when a
// codec context cannot be allocated (lib/zpack_read.c:25-31).
#ifndef _FILE_OFFSET_BITS
#define _FILE_OFFSET_BITS 64
#endif
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <atomic>
#include <mutex>
#include <new>
#include <stdexcept>
#include <vector>

#include "../../include/zpack_b200.h"
#include "zpack_api.h"

namespace {

// ---- little-endian fields (docs/specs.md: all integers LE)
inline zpack_u16 get16(const zpack_u8 *p) { return (zpack_u16)(p[0] | p[1] << 8); }
inline zpack_u32 get32(const zpack_u8 *p) { return (zpack_u32)p[0] | (zpack_u32)p[1] << 8 | (zpack_u32)p[2] << 16 | (zpack_u32)p[3] << 24; }
inline zpack_u64 get64(const zpack_u8 *p) { return (zpack_u64)get32(p) | (zpack_u64)get32(p + 4) << 32; }
inline void put16(zpack_u8 *p, zpack_u16 v) { p[0] = (zpack_u8)v; p[1] = (zpack_u8)(v >> 8); }
inline void put32(zpack_u8 *p, zpack_u32 v) { for (int i = 0; i < 4; ++i) p[i] = (zpack_u8)(v >> (8 * i)); }
inline void put64(zpack_u8 *p, zpack_u64 v) { for (int i = 0; i < 8; ++i) p[i] = (zpack_u8)(v >> (8 * i)); }

// ---- GPU contexts.  Per-entry calls (zpack_read_file, the stream calls, zpack_write_files) use a context that belongs to
// the calling thread — the reference lets a buffer-mode reader be used from several threads with one decompression
// context each (lib/zpack.h:335-341), and nothing here serialises them; threads are dealt round-robin over the visible
// GPUs (ZPACK_GPU_DEVICE pins one).  The batched read uses every GPU at once through one process-wide group.
std::atomic<int> g_next_device{0};
struct ThreadCtx {
    zpb_ctx *c = nullptr;
    zpack_u8 *pin_in = nullptr, *pin_out = nullptr;     // pinned staging of zpack_write_files
    size_t pin_in_cap = 0, pin_out_cap = 0;
    ~ThreadCtx() {
        zpb_host_free(pin_in); zpb_host_free(pin_out);
        if (c) zpb_destroy(c);
    }
    bool ensure_pins(size_t in_bytes, size_t out_bytes) {
        if (in_bytes > pin_in_cap) { zpb_host_free(pin_in); pin_in = (zpack_u8 *)zpb_host_alloc(in_bytes); pin_in_cap = pin_in ? in_bytes : 0; }
        if (out_bytes > pin_out_cap) { zpb_host_free(pin_out); pin_out = (zpack_u8 *)zpb_host_alloc(out_bytes); pin_out_cap = pin_out ? out_bytes : 0; }
        return pin_in && pin_out;
    }
};
thread_local ThreadCtx t_ctx;
zpb_ctx *gpu() {
    if (!t_ctx.c) {
        const char *dev = getenv("ZPACK_GPU_DEVICE");
        if (dev) t_ctx.c = zpb_create(atoi(dev));
        else {
            // round-robin over the devices that exist: probe upwards from the next index, wrap to 0 on failure
            const int k = g_next_device.fetch_add(1);
            static std::atomic<int> ndev{0};
            int n = ndev.load();
            if (n == 0) {
                n = zpb_device_count();
                ndev.store(n > 0 ? n : 1);
                n = ndev.load();
            }
            t_ctx.c = zpb_create(k % n);
        }
        if (!t_ctx.c) {
            // No CPU fallback exists.  Callers get ZPACK_ERROR_* codes, but the reference CLI drops some of them
            // (programs/commands.c:155 ignores zpack_write_file_stream_end), so say it once where a user will see it.
            static std::atomic<bool> told{false};
            if (!told.exchange(true))
                fprintf(stderr, "zpack-b200: no usable CUDA device (%s); every (de)compression call fails, there is no CPU path\n",
                        zpb_last_error(nullptr));
        }
    }
    return t_ctx.c;
}
std::mutex g_group_lock;
zpb_group *g_group = nullptr;
zpb_group *gpu_group() {      // call with g_group_lock held
    if (!g_group) {
        const char *dev = getenv("ZPACK_GPU_DEVICE");
        if (dev) { int d = atoi(dev); g_group = zpb_group_create(&d, 1); }
        else g_group = zpb_group_create(nullptr, 0);
    }
    return g_group;
}
int g_ctx_token;  // zpack_create_cctx / _dctx hand out its address: contexts are opaque to callers
std::atomic<uint64_t> g_reader_gen{1};   // bumped whenever a reader is opened or closed: every read-ahead cache is stale

bool read_at(FILE *fp, zpack_u64 off, void *dst, size_t n, int *err) {
    if (fseeko(fp, (off_t)off, SEEK_SET) != 0) { *err = ZPACK_ERROR_SEEK_FAILED; return false; }
    if (n && fread(dst, 1, n, fp) != n) { *err = ZPACK_ERROR_READ_FAILED; return false; }
    return true;
}

zpack_u64 pow2_at_least(zpack_u64 n) { zpack_u64 b = 1; while (b < n) b <<= 1; return b; }

// append `n` bytes at the writer's cursor, to its FILE* or its growing heap (lib/zpack_common.c:72-104)
int sink_append(zpack_writer *w, const zpack_u8 *src, size_t n) {
    if (w->file) {
        if (fseeko(w->file, (off_t)w->write_offset, SEEK_SET) != 0) return ZPACK_ERROR_SEEK_FAILED;
        if (n && fwrite(src, 1, n, w->file) != n) return ZPACK_ERROR_WRITE_FAILED;
    } else if (w->buffer) {
        zpack_u64 need = (zpack_u64)w->file_size + n;
        if (w->buffer_capacity < need) {
            zpack_u64 cap = pow2_at_least(need);
            zpack_u8 *nb = (zpack_u8 *)realloc(w->buffer, (size_t)cap);
            if (!nb) return ZPACK_ERROR_MALLOC_FAILED;
            w->buffer = nb;
            w->buffer_capacity = (size_t)cap;
        }
        if (n) memcpy(w->buffer + w->write_offset, src, n);
    } else {
        return ZPACK_ERROR_WRITER_NOT_OPENED;
    }
    w->write_offset += n;
    w->file_size += n;
    return ZPACK_OK;
}

zpack_file_entry *push_entry(zpack_writer *w) {
    if (w->file_count + 1 > w->fe_capacity) {
        zpack_u64 cap = pow2_at_least(w->file_count + 1);
        zpack_file_entry *ne = (zpack_file_entry *)realloc(w->file_entries, (size_t)(cap * sizeof(zpack_file_entry)));
        if (!ne) return nullptr;
        w->file_entries = ne;
        w->fe_capacity = cap;
    }
    zpack_file_entry *e = w->file_entries + w->file_count++;
    memset(e, 0, sizeof *e);
    return e;
}

char *dup_name(const char *s) {
    size_t n = strlen(s) + 1;
    char *d = (char *)malloc(n);
    if (d) memcpy(d, s, n);
    return d;
}

// the staging a GPU-backed stream needs; lives behind zpack_stream.xxh3_state
struct StreamState {
    std::vector<zpack_u8> data;   // read: the decoded entry; write: the file's bytes so far
    size_t pos = 0;               // read: bytes already handed out
    int verdict = ZPACK_OK;       // read: status of the GPU decode (reported when the stream is done)
    bool loaded = false;
};
StreamState *state_of(zpack_stream *s) { return (StreamState *)s->xxh3_state; }

bool known_method(int m) { return m == ZPACK_COMPRESSION_NONE || m == ZPACK_COMPRESSION_ZSTD || m == ZPACK_COMPRESSION_LZ4; }

// Bytes of an entry's start that zstd_framed_head looks at
constexpr size_t ZSTD_HEAD_BYTES = 7;

// Whether a zstd entry starts the way this library's writer starts one of 64 KB frames: a single-segment frame of at
// most 64 KB, no checksum, no dictionary.  Anything else — the reference's one frame of dependent blocks, this
// library's frames from before the 64 KB layout — has nothing for the frame-parallel path.
bool zstd_framed_head(const zpack_u8 *p, size_t n) {
    if (n < 6 || get32(p) != 0xFD2FB528u) return false;
    const unsigned fhd = p[4];
    if (!(fhd & 0x20) || (fhd & 0x0F)) return false;
    if ((fhd >> 6) == 0) return true;                                  // 1-byte Frame_Content_Size
    return (fhd >> 6) == 1 && n >= 7 && get16(p + 5) + 256u <= 65536u;  // 2 bytes, holding size - 256
}

// Entries gpu_unpack_one first offers to zpb_unpack_entry_blocks_host (`head`: the first bytes of the entry, n of
// them).  zstd is routed on decoded size: a highly compressible file can be small on disk, and one warp's decode time
// grows with the bytes it writes.
bool block_path_entry(const zpack_file_entry &e, const zpack_u8 *head, size_t n) {
    return (e.comp_method == ZPACK_COMPRESSION_LZ4 && e.comp_size >= ZPB_ZSTD_FRAMED_MIN) ||
           (e.comp_method == ZPACK_COMPRESSION_ZSTD && e.uncomp_size >= ZPB_ZSTD_FRAMED_MIN && zstd_framed_head(head, n));
}

// One entry through the GPU: compressed bytes `comp` -> dst[0..max_size).  Returns an enum zpack_result.
int gpu_unpack_one(const zpack_u8 *comp, zpack_u64 comp_size, zpack_u8 *dst, size_t max_size, const zpack_file_entry *e,
                   size_t *last_return) {
    zpb_ctx *g = gpu();
    if (!g) return ZPACK_ERROR_MALLOC_FAILED;
    zpb_entry d;
    memset(&d, 0, sizeof d);
    d.src_off = 0; d.comp_size = comp_size; d.dst_off = 0; d.dst_cap = max_size;
    d.uncomp_size = e->uncomp_size; d.hash = e->hash; d.method = e->comp_method;
    int32_t st = 0;
    uint64_t dg = 0;
    // a large LZ4 entry written with independent blocks, or a large zstd entry written as 64 KB frames (what this
    // library's writer emits), is decoded block-parallel, chunks pipelined over PCIe; anything else — and anything that
    // path declines — is one dependency chain
    if (block_path_entry(*e, comp, (size_t)std::min<zpack_u64>(comp_size, ZSTD_HEAD_BYTES))) {
        int rc = zpb_unpack_entry_blocks_host(g, comp, comp_size, dst, max_size, e->uncomp_size, e->hash, 0, &st, &dg);
        if (rc == ZPB_OK) {
            if (last_return) *last_return = (size_t)st;
            return st;
        }
        if (rc != ZPB_INDEX_UNSUPPORTED) return ZPACK_ERROR_DECOMPRESS_FAILED;
    }
    if (zpb_unpack_host(g, comp, comp_size, dst, max_size, &d, 1, &st, &dg) != ZPB_OK) return ZPACK_ERROR_DECOMPRESS_FAILED;
    if (last_return) *last_return = (size_t)st;
    return st;
}

}  // namespace

extern "C" {

// ------------------------------------------------------------------------------------------------
// section readers
int zpack_read_header_memory(const zpack_u8 *b, zpack_u16 *version) {
    if (get32(b) != ZPK_SIG_HEADER) return ZPACK_ERROR_SIGNATURE_INVALID;
    *version = get16(b + 4);
    return (*version < ZPK_VERSION_MIN || *version > ZPK_VERSION_MAX) ? ZPACK_ERROR_VERSION_INCOMPATIBLE : ZPACK_OK;
}
int zpack_read_header(FILE *fp, zpack_u16 *version) {
    zpack_u8 b[ZPK_HEADER_BYTES];
    int err;
    if (!read_at(fp, 0, b, sizeof b, &err)) return err;
    return zpack_read_header_memory(b, version);
}
int zpack_read_data_header_memory(const zpack_u8 *b) { return get32(b) == ZPK_SIG_DATA ? ZPACK_OK : ZPACK_ERROR_SIGNATURE_INVALID; }
int zpack_read_data_header(FILE *fp) {
    zpack_u8 b[ZPK_SIG_BYTES];
    int err;
    if (!read_at(fp, ZPK_HEADER_BYTES, b, sizeof b, &err)) return err;
    return zpack_read_data_header_memory(b);
}
int zpack_read_eocdr_memory(const zpack_u8 *b, zpack_u64 *cdr_offset) {
    if (get32(b) != ZPK_SIG_EOCDR) return ZPACK_ERROR_SIGNATURE_INVALID;
    *cdr_offset = get64(b + 4);
    return ZPACK_OK;
}
int zpack_read_eocdr(FILE *fp, zpack_u64 eocdr_offset, zpack_u64 *cdr_offset) {
    zpack_u8 b[ZPK_EOCDR_BYTES];
    int err;
    if (!read_at(fp, eocdr_offset, b, sizeof b, &err)) return err;
    return zpack_read_eocdr_memory(b, cdr_offset);
}
int zpack_read_cdr_header_memory(const zpack_u8 *b, zpack_u64 *count, zpack_u64 *block_size) {
    if (get32(b) != ZPK_SIG_CDR) return ZPACK_ERROR_SIGNATURE_INVALID;
    *count = get64(b + 4);
    *block_size = get64(b + 12);
    return ZPACK_OK;
}
int zpack_read_file_entry_memory(const zpack_u8 *b, zpack_u64 *size_left, zpack_file_entry *entry, size_t *entry_size) {
    const zpack_u16 nlen = get16(b);
    *entry_size = (size_t)ZPK_ENTRY_FIXED_BYTES + nlen;
    if (*entry_size > *size_left) return ZPACK_ERROR_BLOCK_SIZE_INVALID;
    *size_left -= *entry_size;
    entry->filename = (char *)malloc((size_t)nlen + 1);
    if (!entry->filename) return ZPACK_ERROR_MALLOC_FAILED;
    memcpy(entry->filename, b + 2, nlen);
    entry->filename[nlen] = 0;
    const zpack_u8 *f = b + 2 + nlen;
    entry->offset = get64(f);
    entry->comp_size = get64(f + 8);
    entry->uncomp_size = get64(f + 16);
    entry->hash = get64(f + 24);
    entry->comp_method = f[32];
    return ZPACK_OK;
}
int zpack_read_file_entries_memory(const zpack_u8 *b, zpack_file_entry **entries, zpack_u64 header_count, zpack_u64 block_size,
                                   zpack_u64 *count, zpack_u64 *total_cs, zpack_u64 *total_us) {
    if (header_count > block_size / ZPK_ENTRY_FIXED_BYTES) return ZPACK_ERROR_BLOCK_SIZE_INVALID;
    const zpack_u64 bytes = header_count * sizeof(zpack_file_entry);
    zpack_file_entry *arr = (zpack_file_entry *)realloc(*entries, (size_t)bytes);
    if (!arr) return ZPACK_ERROR_MALLOC_FAILED;
    *entries = arr;
    memset(arr, 0, (size_t)bytes);
    for (zpack_u64 i = 0; i < header_count; ++i) {
        size_t used = 0;
        int rc = zpack_read_file_entry_memory(b, &block_size, arr + i, &used);
        if (rc) return rc;
        ++*count;
        *total_cs += arr[i].comp_size;
        *total_us += arr[i].uncomp_size;
        b += used;
    }
    return ZPACK_OK;
}
int zpack_read_cdr_memory(const zpack_u8 *b, size_t size_left, zpack_file_entry **entries, zpack_u64 *count, zpack_u64 *total_cs,
                          zpack_u64 *total_us) {
    zpack_u64 n = 0, block = 0;
    if (size_left < ZPK_CDR_HEADER_BYTES) return ZPACK_ERROR_BLOCK_SIZE_INVALID;   // the header itself must be inside the buffer
    int rc = zpack_read_cdr_header_memory(b, &n, &block);
    if (rc) return rc;
    if (block > size_left || ZPK_CDR_HEADER_BYTES > size_left - block) return ZPACK_ERROR_BLOCK_SIZE_INVALID;
    if (n == 0) return ZPACK_OK;
    return zpack_read_file_entries_memory(b + ZPK_CDR_HEADER_BYTES, entries, n, block, count, total_cs, total_us);
}
int zpack_read_cdr(FILE *fp, zpack_u64 cdr_offset, zpack_file_entry **entries, zpack_u64 *count, zpack_u64 *total_cs,
                   zpack_u64 *total_us) {
    zpack_u8 hdr[ZPK_CDR_HEADER_BYTES];
    int err;
    if (!read_at(fp, cdr_offset, hdr, sizeof hdr, &err)) return err;
    zpack_u64 n = 0, block = 0;
    int rc = zpack_read_cdr_header_memory(hdr, &n, &block);
    if (rc) return rc;
    if (n == 0) return ZPACK_OK;
    // `block` is an untrusted 64-bit field: it cannot exceed what the file holds behind the CDR header
    if (fseeko(fp, 0, SEEK_END) != 0) return ZPACK_ERROR_SEEK_FAILED;
    const zpack_u64 fsize = (zpack_u64)ftello(fp);
    if (cdr_offset > fsize || fsize - cdr_offset < ZPK_CDR_HEADER_BYTES || block > fsize - cdr_offset - ZPK_CDR_HEADER_BYTES)
        return ZPACK_ERROR_BLOCK_SIZE_INVALID;
    std::vector<zpack_u8> body;
    try { body.resize((size_t)block); } catch (const std::exception &) { return ZPACK_ERROR_MALLOC_FAILED; }
    if (!read_at(fp, cdr_offset + ZPK_CDR_HEADER_BYTES, body.data(), (size_t)block, &err)) return err;
    return zpack_read_file_entries_memory(body.data(), entries, n, block, count, total_cs, total_us);
}

// ------------------------------------------------------------------------------------------------
// reader
int zpack_read_archive_memory(zpack_reader *r) {
    g_reader_gen.fetch_add(1);
    if (!r->buffer) return ZPACK_ERROR_ARCHIVE_NOT_LOADED;
    if (r->file_size < ZPK_MIN_ARCHIVE_BYTES) return ZPACK_ERROR_FILE_TOO_SMALL;
    int rc;
    if ((rc = zpack_read_header_memory(r->buffer, &r->version))) return rc;
    if ((rc = zpack_read_data_header_memory(r->buffer + ZPK_HEADER_BYTES))) return rc;
    r->eocdr_offset = r->file_size - ZPK_EOCDR_BYTES;
    if ((rc = zpack_read_eocdr_memory(r->buffer + r->eocdr_offset, &r->cdr_offset))) return rc;
    if (r->cdr_offset >= r->file_size) return ZPACK_ERROR_READ_FAILED;
    return zpack_read_cdr_memory(r->buffer + r->cdr_offset, (size_t)(r->file_size - r->cdr_offset), &r->file_entries,
                                 &r->file_count, &r->comp_size, &r->uncomp_size);
}
int zpack_read_archive(zpack_reader *r) {
    g_reader_gen.fetch_add(1);
    if (!r->file) return ZPACK_ERROR_ARCHIVE_NOT_LOADED;
    if (fseeko(r->file, 0, SEEK_END) != 0) return ZPACK_ERROR_SEEK_FAILED;
    if (!r->file_size) r->file_size = (size_t)ftello(r->file);
    if (r->file_size < ZPK_MIN_ARCHIVE_BYTES) return ZPACK_ERROR_FILE_TOO_SMALL;
    int rc;
    if ((rc = zpack_read_header(r->file, &r->version))) return rc;
    if ((rc = zpack_read_data_header(r->file))) return rc;
    r->eocdr_offset = r->file_size - ZPK_EOCDR_BYTES;
    if ((rc = zpack_read_eocdr(r->file, r->eocdr_offset, &r->cdr_offset))) return rc;
    return zpack_read_cdr(r->file, r->cdr_offset, &r->file_entries, &r->file_count, &r->comp_size, &r->uncomp_size);
}
int zpack_read_raw_file(zpack_reader *r, zpack_file_entry *e, zpack_u8 *buffer, size_t max_size) {
    if (e->offset > r->file_size || e->comp_size > r->file_size - e->offset) return ZPACK_ERROR_FILE_OFFSET_INVALID;
    const size_t n = (size_t)(max_size < e->comp_size ? max_size : e->comp_size);
    if (r->file) {
        int err;
        if (!read_at(r->file, e->offset, buffer, n, &err)) return err;
    } else if (r->buffer) {
        memcpy(buffer, r->buffer + e->offset, n);
    } else {
        return ZPACK_ERROR_ARCHIVE_NOT_LOADED;
    }
    return ZPACK_OK;
}

// ---- read-ahead.  The reference's API hands out one entry per call (its CLI's `t` and `x` walk reader->file_entries
// in order, programs/commands.c), and a GPU call costs about the same for one entry as for a thousand.  When a thread
// asks for entry i of a reader's own CDR array right after entry i-1, the entries behind it — up to
// ZPACK_GPU_READAHEAD_MB of decoded bytes (default 128, 0 = off) — are decoded by the same call into a per-thread
// cache, and the following calls are served from it.  What a call returns (bytes, status, last_return) is what the
// individual call would have returned: same kernels, same entry fields (a cached result is only used while the
// entry's fields are what they were when it was decoded).
struct ReadAhead {
    const zpack_reader *owner = nullptr;
    uint64_t gen = 0;
    zpack_u64 last_idx = ~0ull;                 // entry index of this thread's previous zpack_read_file on `owner`
    zpack_u64 first = 0, count = 0;             // cached entries [first, first + count)
    zpack_u8 *out = nullptr;                    // pinned
    size_t out_cap = 0;
    std::vector<zpack_u64> off;
    std::vector<int32_t> st;
    std::vector<zpack_file_entry> seen;         // the entries' fields at decode time (filename unused)
    std::vector<zpb_entry> d;
    std::vector<zpack_u8> staged;
    ~ReadAhead() { zpb_host_free(out); }
};
thread_local ReadAhead t_ra;
size_t readahead_bytes() {
    static const size_t v = [] {
        const char *e = getenv("ZPACK_GPU_READAHEAD_MB");
        return (size_t)(e ? atoll(e) : 128) << 20;
    }();
    return v;
}
bool same_fields(const zpack_file_entry &a, const zpack_file_entry &b) {
    return a.offset == b.offset && a.comp_size == b.comp_size && a.uncomp_size == b.uncomp_size && a.hash == b.hash &&
           a.comp_method == b.comp_method;
}
bool plain_entry(const zpack_reader *r, const zpack_file_entry &e) {      // what zpack_read_file would hand to the GPU as one chain
    if (!e.comp_size || e.offset >= r->file_size || e.comp_size >= r->file_size - e.offset || !known_method(e.comp_method))
        return false;
    if (e.comp_method != ZPACK_COMPRESSION_ZSTD || e.uncomp_size < ZPB_ZSTD_FRAMED_MIN) return !block_path_entry(e, nullptr, 0);
    // a large zstd entry leaves the read-ahead batch only when it is 64 KB frames: its first bytes say so
    zpack_u8 head[ZSTD_HEAD_BYTES];
    const size_t n = (size_t)std::min<zpack_u64>(e.comp_size, sizeof head);
    int err;
    if (r->buffer) memcpy(head, r->buffer + e.offset, n);
    else if (!r->file || !read_at(r->file, e.offset, head, n, &err)) return true;   // the read that follows reports it
    return !block_path_entry(e, head, n);
}
// Decodes entries [idx, idx + k) into the cache; false = nothing cached (the caller takes the one-entry path).
bool readahead_fill(zpack_reader *r, zpack_u64 idx) {
    ReadAhead &c = t_ra;
    const size_t budget = readahead_bytes();
    zpack_u64 k = 0, bytes = 0;
    while (idx + k < r->file_count && k < 65536) {
        const zpack_file_entry &e = r->file_entries[idx + k];
        if (!plain_entry(r, e)) break;
        const zpack_u64 slot = (e.uncomp_size + 15) & ~15ull;
        if (bytes + slot > budget) break;
        bytes += slot;
        ++k;
    }
    c.count = 0;
    if (k < 2) return false;
    zpb_ctx *g = gpu();
    if (!g) return false;
    if (c.out_cap < bytes + 16) {
        zpb_host_free(c.out);
        c.out = (zpack_u8 *)zpb_host_alloc(budget + 16);
        c.out_cap = c.out ? budget + 16 : 0;
        if (!c.out) return false;
    }
    try {
        c.off.resize((size_t)k); c.st.assign((size_t)k, 0); c.seen.assign(r->file_entries + idx, r->file_entries + idx + k);
        c.d.resize((size_t)k);
        if (!r->buffer) {
            zpack_u64 total = 0;
            for (zpack_u64 i = 0; i < k; ++i) total += (c.seen[i].comp_size + 15) & ~15ull;
            c.staged.resize((size_t)total + 16);
        }
    } catch (const std::exception &) { return false; }
    zpack_u64 pos = 0, spos = 0;
    for (zpack_u64 i = 0; i < k; ++i) {
        const zpack_file_entry &e = c.seen[i];
        zpb_entry &d = c.d[i];
        memset(&d, 0, sizeof d);
        d.src_off = e.offset; d.comp_size = e.comp_size; d.dst_off = pos; d.dst_cap = e.uncomp_size;
        d.uncomp_size = e.uncomp_size; d.hash = e.hash; d.method = e.comp_method;
        if (!r->buffer) {
            int err;
            if (!read_at(r->file, e.offset, c.staged.data() + spos, (size_t)e.comp_size, &err)) return false;
            d.src_off = spos;
            spos += (e.comp_size + 15) & ~15ull;
        }
        c.off[i] = pos;
        pos += (e.uncomp_size + 15) & ~15ull;
    }
    const zpack_u8 *arch = r->buffer ? r->buffer : c.staged.data();
    const zpack_u64 asz = r->buffer ? r->file_size : c.staged.size();
    if (zpb_unpack_host(g, arch, asz, c.out, c.out_cap, c.d.data(), k, c.st.data(), nullptr) != ZPB_OK) return false;
    c.owner = r; c.gen = g_reader_gen.load(); c.first = idx; c.count = k;
    return true;
}

// zpack_read_file (lib/zpack_read.c:326-471) = a GPU batch of one
int zpack_read_file(zpack_reader *r, zpack_file_entry *e, zpack_u8 *buffer, size_t max_size, void *) {
    if (e->comp_size == 0) return ZPACK_OK;                                          // :328
    if (max_size < e->uncomp_size) return ZPACK_ERROR_BUFFER_TOO_SMALL;              // :329
    // :331 (strict: offset + comp_size < file_size), written so that it cannot wrap
    if (e->offset >= r->file_size || e->comp_size >= r->file_size - e->offset) return ZPACK_ERROR_FILE_OFFSET_INVALID;
    if (!known_method(e->comp_method)) return ZPACK_ERROR_COMP_METHOD_INVALID;       // :459-461
    if (!r->file && !r->buffer) return ZPACK_ERROR_ARCHIVE_NOT_LOADED;
    if (readahead_bytes() && r->file_entries && e >= r->file_entries && e < r->file_entries + r->file_count) {
        ReadAhead &c = t_ra;
        const zpack_u64 idx = (zpack_u64)(e - r->file_entries);
        const bool mine = c.owner == r && c.gen == g_reader_gen.load();
        const bool sequential = mine && c.last_idx + 1 == idx;
        if (!mine) { c.owner = r; c.gen = g_reader_gen.load(); c.count = 0; }
        c.last_idx = idx;
        bool hit = mine && idx >= c.first && idx < c.first + c.count && same_fields(*e, c.seen[(size_t)(idx - c.first)]);
        if (!hit && sequential && plain_entry(r, *e)) hit = readahead_fill(r, idx);
        if (hit) {
            const size_t k = (size_t)(idx - c.first);
            memcpy(buffer, c.out + c.off[k], (size_t)e->uncomp_size);
            r->last_return = (size_t)c.st[k];
            return c.st[k];
        }
    }
    if (r->file) {                                                                   // :336-344
        std::vector<zpack_u8> comp;
        try { comp.resize((size_t)e->comp_size); } catch (const std::exception &) { return ZPACK_ERROR_MALLOC_FAILED; }
        int rc = zpack_read_raw_file(r, e, comp.data(), comp.size());
        if (rc) return rc;
        return gpu_unpack_one(comp.data(), e->comp_size, buffer, max_size, e, &r->last_return);
    }
    if (!r->buffer) return ZPACK_ERROR_ARCHIVE_NOT_LOADED;
    return gpu_unpack_one(r->buffer + e->offset, e->comp_size, buffer, max_size, e, &r->last_return);   // :345-346
}

// The batched read (the extension SURVEY F7 asks for: the reference's API reads one entry per call): every entry of the
// batch decoded and verified by ONE call that uses every visible GPU (zpb_group_unpack_host).  Buffer-mode readers hand
// their archive over as it is; file-mode readers have the entries' compressed bytes read into one staging buffer first.
int zpack_read_files(zpack_reader *r, zpack_file_entry *entries, zpack_u64 n, zpack_u8 *out, zpack_u64 out_size,
                     const zpack_u64 *dst_off, const zpack_u64 *dst_cap, int *status) {
    if (!r->buffer && !r->file) return ZPACK_ERROR_ARCHIVE_NOT_LOADED;
    std::vector<zpb_entry> d;
    std::vector<int32_t> st;
    std::vector<zpack_u8> staged;
    try {
        d.resize((size_t)n); st.assign((size_t)n, 0);
        if (!r->buffer) {
            zpack_u64 total = 0;
            for (zpack_u64 i = 0; i < n; ++i)
                if (entries[i].comp_size && entries[i].offset < r->file_size && entries[i].comp_size < r->file_size - entries[i].offset)
                    total += (entries[i].comp_size + 15) & ~15ull;
            staged.resize((size_t)total + 16);
        }
    } catch (const std::exception &) { return ZPACK_ERROR_MALLOC_FAILED; }
    zpack_u64 pos = 0;
    for (zpack_u64 i = 0; i < n; ++i) {
        memset(&d[i], 0, sizeof(zpb_entry));
        const zpack_file_entry &e = entries[i];
        d[i].src_off = e.offset; d[i].comp_size = e.comp_size; d[i].dst_off = dst_off[i]; d[i].dst_cap = dst_cap[i];
        d[i].uncomp_size = e.uncomp_size; d[i].hash = e.hash; d[i].method = e.comp_method;
        if (e.comp_size && (e.offset >= r->file_size || e.comp_size >= r->file_size - e.offset)) { d[i].src_off = ~0ull; continue; }   // -> FILE_OFFSET_INVALID
        if (!r->buffer && e.comp_size) {
            int err;
            if (!read_at(r->file, e.offset, staged.data() + pos, (size_t)e.comp_size, &err)) return err;
            d[i].src_off = pos;
            pos += (e.comp_size + 15) & ~15ull;
        }
    }
    std::lock_guard<std::mutex> lk(g_group_lock);
    zpb_group *g = gpu_group();
    if (!g) return ZPACK_ERROR_MALLOC_FAILED;
    const zpack_u8 *arch = r->buffer ? r->buffer : staged.data();
    const zpack_u64 asz = r->buffer ? r->file_size : staged.size();
    if (zpb_group_unpack_host(g, arch, asz, out, out_size, d.data(), n, st.data(), nullptr) != ZPB_OK)
        return ZPACK_ERROR_DECOMPRESS_FAILED;
    int worst = ZPACK_OK;
    for (zpack_u64 i = 0; i < n; ++i) {
        if (status) status[i] = st[i];
        if (st[i] && !worst) worst = st[i];
    }
    return worst;
}

int zpack_read_raw_file_stream(zpack_reader *r, zpack_file_entry *e, zpack_stream *s, size_t *in_size) {
    if (e->comp_size == 0) return ZPACK_OK;
    if (e->offset > r->file_size || e->comp_size > r->file_size - e->offset) return ZPACK_ERROR_FILE_OFFSET_INVALID;
    if (!s->next_in || !s->avail_in || s->total_in > e->comp_size) return ZPACK_ERROR_STREAM_INVALID;
    zpack_u64 left = e->comp_size - s->total_in;
    size_t n = (size_t)(s->avail_in < left ? s->avail_in : left);
    if (n == 0) return ZPACK_OK;
    const zpack_u64 at = e->offset + s->total_in;
    if (r->file) {
        int err;
        if (!read_at(r->file, at, s->next_in, n, &err)) return err;
    } else if (r->buffer) {
        memcpy(s->next_in, r->buffer + at, n);
    } else {
        return ZPACK_ERROR_ARCHIVE_NOT_LOADED;
    }
    s->next_in += n; s->avail_in -= n; s->total_in += n;
    *in_size = n;
    return ZPACK_OK;
}

// zpack_read_file_stream (lib/zpack_read.c:515-640).  The GPU decodes whole entries, so the first call
// of an entry decodes it into the stream's staging buffer; every call then moves compressed bytes into
// the caller's input buffer and decoded bytes into its output buffer exactly as the field contract
// says (:502-513), keeps read_back > 0 while decoded bytes are still owed, and reports the digest verdict
// on the call that reaches ZPACK_READ_STREAM_DONE (:631-637).
int zpack_read_file_stream(zpack_reader *r, zpack_file_entry *e, zpack_stream *s, void *) {
    if (e->comp_size == 0 || zpack_read_stream_done(s, e)) return ZPACK_OK;
    if (!s->next_out || !s->avail_out) return ZPACK_ERROR_STREAM_INVALID;
    StreamState *st = state_of(s);
    if (!st) return ZPACK_ERROR_STREAM_INVALID;
    if (!known_method(e->comp_method)) return ZPACK_ERROR_COMP_METHOD_INVALID;
    if (s->total_in == 0) {   // a new entry starts (:524-525 resets the hash state here)
        st->loaded = false; st->pos = 0; st->verdict = ZPACK_OK;
        try { st->data.assign((size_t)e->uncomp_size, 0); } catch (const std::exception &) { return ZPACK_ERROR_MALLOC_FAILED; }
        int rc = zpack_read_file(r, e, st->data.data(), st->data.size(), nullptr);
        if (rc && rc != ZPACK_ERROR_FILE_HASH_MISMATCH) return rc;
        st->verdict = rc;
        st->loaded = true;
    }
    if (!st->loaded) return ZPACK_ERROR_STREAM_INVALID;
    size_t in_size = s->read_back;                        // leftover input sits at the front of next_in (:528-536)
    if (s->read_back) { s->next_in += s->read_back; s->avail_in -= s->read_back; s->read_back = 0; }
    if (s->total_in < e->comp_size) {
        size_t got = 0;
        int rc = zpack_read_raw_file_stream(r, e, s, &got);
        if (rc) return rc;
        in_size += got;
    }
    size_t owed = st->data.size() - st->pos;
    size_t n = owed < s->avail_out ? owed : s->avail_out;
    if (n) memcpy(s->next_out, st->data.data() + st->pos, n);
    st->pos += n;
    s->next_out += n; s->avail_out -= n; s->total_out += n;
    // all input handed over but output still owed: keep the stream open by asking for one byte back
    if (st->pos < st->data.size() && s->total_in == e->comp_size) s->read_back = in_size ? 1 : 0;
    if (zpack_read_stream_done(s, e)) return st->verdict;
    return ZPACK_OK;
}

int zpack_init_reader(zpack_reader *r, const char *path) {
    FILE *fp = fopen(path, "rb");
    if (!fp) return ZPACK_ERROR_OPEN_FAILED;
    if (r->file) fclose(r->file);
    r->file = fp;
    return zpack_read_archive(r);
}
int zpack_init_reader_cfile(zpack_reader *r, FILE *fp) { r->file = fp; return zpack_read_archive(r); }
int zpack_init_reader_memory(zpack_reader *r, const zpack_u8 *buffer, size_t size) {
    r->buffer = (zpack_u8 *)malloc(size ? size : 1);
    if (!r->buffer) return ZPACK_ERROR_MALLOC_FAILED;
    memcpy(r->buffer, buffer, size);
    r->file_size = size;
    r->buffer_shared = 0;
    return zpack_read_archive_memory(r);
}
int zpack_init_reader_memory_shared(zpack_reader *r, zpack_u8 *buffer, size_t size) {
    r->buffer = buffer;
    r->file_size = size;
    r->buffer_shared = 1;
    return zpack_read_archive_memory(r);
}
void zpack_reset_reader_dctx(zpack_reader *) {}   // GPU decodes are one-shot: nothing carries over between calls
void zpack_close_reader(zpack_reader *r) {
    g_reader_gen.fetch_add(1);
    if (r->file) fclose(r->file);
    if (!r->buffer_shared) free(r->buffer);
    if (r->file_entries) {
        for (zpack_u64 i = 0; i < r->file_count; ++i) free(r->file_entries[i].filename);
        free(r->file_entries);
    }
    memset(r, 0, sizeof *r);
}

// ------------------------------------------------------------------------------------------------
// writer
int zpack_init_writer(zpack_writer *w, const char *path) {
    w->file = fopen(path, "wb");
    return w->file ? ZPACK_OK : ZPACK_ERROR_OPEN_FAILED;
}
int zpack_init_writer_cfile(zpack_writer *w, FILE *fp) {
    if (!fp) return ZPACK_ERROR_OPEN_FAILED;
    w->file = fp;
    return ZPACK_OK;
}
int zpack_init_writer_heap(zpack_writer *w, size_t initial_size) {
    const size_t floor_ = ZPK_HEADER_BYTES + ZPK_SIG_BYTES;
    w->buffer_capacity = initial_size > floor_ ? initial_size : floor_;
    w->buffer = (zpack_u8 *)malloc(w->buffer_capacity);
    return w->buffer ? ZPACK_OK : ZPACK_ERROR_MALLOC_FAILED;
}
int zpack_write_header_ex(zpack_writer *w, zpack_u16 version) {
    zpack_u8 b[ZPK_HEADER_BYTES];
    put32(b, ZPK_SIG_HEADER);
    put16(b + 4, version);
    return sink_append(w, b, sizeof b);
}
int zpack_write_header(zpack_writer *w) { return zpack_write_header_ex(w, ZPK_VERSION_MAX); }
int zpack_write_data_header(zpack_writer *w) {
    zpack_u8 b[ZPK_SIG_BYTES];
    put32(b, ZPK_SIG_DATA);
    return sink_append(w, b, sizeof b);
}

// zpack_write_files (lib/zpack_write.c:280-343): the files of one call are compressed by ONE GPU batch
// (bounded staging: batches of <= 256 MiB of input), then appended in order; entry.offset is the running
// write cursor, i.e. the exclusive prefix sum of the compressed sizes — assembled here, on the host.
int zpack_write_files(zpack_writer *w, zpack_file *files, zpack_u64 file_count) {
    if (!w->file && !w->buffer) return ZPACK_ERROR_WRITER_NOT_OPENED;
    zpack_u64 i = 0;
    while (i < file_count) {
        zpack_u64 j = i, in_bytes = 0, out_bytes = 0;
        std::vector<zpb_file> d;
        while (j < file_count && (j == i || in_bytes + files[j].size <= (256ull << 20))) {
            const int m = files[j].options->method;
            if (!known_method(m)) { if (j == i) return ZPACK_ERROR_COMP_METHOD_INVALID; break; }
            zpb_file f;
            memset(&f, 0, sizeof f);
            f.src_off = in_bytes; f.size = files[j].size;
            f.dst_off = out_bytes; f.dst_cap = zpb_pack_bound((uint32_t)m, files[j].size);
            f.method = (uint32_t)m; f.level = files[j].options->level;
            in_bytes += (files[j].size + 15) & ~15ull;
            out_bytes += (f.dst_cap + 15) & ~15ull;
            d.push_back(f);
            ++j;
        }
        const size_t n = d.size();
        std::vector<uint64_t> csz(n), dig(n);
        std::vector<int32_t> st(n);
        zpb_ctx *g = gpu();
        if (!g) return ZPACK_ERROR_MALLOC_FAILED;
        // pinned staging owned by the calling thread (pageable buffers would make every copy of zpb_pack_host synchronous)
        if (!t_ctx.ensure_pins((size_t)in_bytes + 16, (size_t)out_bytes + 16)) return ZPACK_ERROR_MALLOC_FAILED;
        zpack_u8 *in = t_ctx.pin_in, *out = t_ctx.pin_out;
        for (size_t k = 0; k < n; ++k)
            if (files[i + k].size) memcpy(in + d[k].src_off, files[i + k].buffer, (size_t)files[i + k].size);
        if (zpb_pack_host(g, in, in_bytes + 16, out, out_bytes + 16, d.data(), n, csz.data(), dig.data(), st.data()) != ZPB_OK)
            return ZPACK_ERROR_COMPRESS_FAILED;
        for (size_t k = 0; k < n; ++k) {
            w->last_return = (size_t)st[k];
            if (st[k]) return st[k];                       // files before it are already in the archive, as in the reference
            zpack_file_entry *e = push_entry(w);
            if (!e) return ZPACK_ERROR_MALLOC_FAILED;
            if (!(e->filename = dup_name(files[i + k].filename))) return ZPACK_ERROR_MALLOC_FAILED;
            e->offset = w->write_offset;
            e->comp_size = csz[k];
            e->uncomp_size = files[i + k].size;
            e->hash = dig[k];                              // XXH3-64 of the input, fused into the pack kernel
            e->comp_method = (zpack_u8)files[i + k].options->method;
            int rc = sink_append(w, out + d[k].dst_off, (size_t)csz[k]);
            if (rc) return rc;
        }
        i = j;
    }
    return ZPACK_OK;
}

int zpack_write_files_from_archive(zpack_writer *w, zpack_reader *r, zpack_file_entry *entries, zpack_u64 file_count) {
    if (!w->file && !w->buffer) return ZPACK_ERROR_WRITER_NOT_OPENED;
    std::vector<zpack_u8> tmp;
    for (zpack_u64 i = 0; i < file_count; ++i) {
        const zpack_file_entry &s = entries[i];
        const zpack_u8 *src;
        if (r->file) {
            try { if (tmp.size() < s.comp_size) tmp.resize((size_t)s.comp_size); } catch (const std::exception &) { return ZPACK_ERROR_MALLOC_FAILED; }
            int rc = zpack_read_raw_file(r, entries + i, tmp.data(), tmp.size());
            if (rc) return rc;
            src = tmp.data();
        } else if (r->buffer) {
            if (s.offset >= r->file_size || s.comp_size > r->file_size - s.offset) return ZPACK_ERROR_FILE_OFFSET_INVALID;
            src = r->buffer + s.offset;
        } else {
            return ZPACK_ERROR_ARCHIVE_NOT_LOADED;
        }
        zpack_file_entry *e = push_entry(w);
        if (!e) return ZPACK_ERROR_MALLOC_FAILED;
        *e = s;
        if (!(e->filename = dup_name(s.filename))) return ZPACK_ERROR_MALLOC_FAILED;
        e->offset = w->write_offset;
        int rc = sink_append(w, src, (size_t)s.comp_size);
        if (rc) return rc;
    }
    return ZPACK_OK;
}

// Streaming writes (lib/zpack_write.c:461-685): chunks are staged; the file is compressed by the GPU in
// zpack_write_file_stream_end, which appends it and records the entry with
// offset = write_offset - total_out (:677), exactly as the reference computes it.
int zpack_write_file_stream(zpack_writer *w, zpack_compress_options *opt, zpack_stream *s, void *) {
    if (!s->next_in || !s->next_out || !s->avail_out) return ZPACK_ERROR_STREAM_INVALID;
    if (!known_method(opt->method)) return ZPACK_ERROR_COMP_METHOD_INVALID;
    if (!w->file && !w->buffer) return ZPACK_ERROR_WRITER_NOT_OPENED;
    StreamState *st = state_of(s);
    if (!st) return ZPACK_ERROR_STREAM_INVALID;
    if (s->total_in == 0) st->data.clear();
    try { st->data.insert(st->data.end(), s->next_in, s->next_in + s->avail_in); }
    catch (const std::exception &) { return ZPACK_ERROR_MALLOC_FAILED; }
    s->next_in += s->avail_in;
    s->total_in += s->avail_in;
    s->avail_in = 0;
    return ZPACK_OK;
}
int zpack_write_file_stream_end(zpack_writer *w, char *filename, zpack_compress_options *opt, zpack_stream *s, void *) {
    if (!s->next_out || !s->avail_out) return ZPACK_ERROR_STREAM_INVALID;
    if (!known_method(opt->method)) return ZPACK_ERROR_COMP_METHOD_INVALID;
    StreamState *st = state_of(s);
    if (!st) return ZPACK_ERROR_STREAM_INVALID;
    if (s->total_in == 0) st->data.clear();
    zpack_file f;
    f.filename = filename; f.buffer = st->data.data(); f.size = st->data.size(); f.options = opt; f.cctx = nullptr;
    const size_t before = w->write_offset;
    int rc = zpack_write_files(w, &f, 1);
    if (rc) return rc;
    s->total_out += w->write_offset - before;
    st->data.clear();
    return ZPACK_OK;
}

int zpack_write_cdr_ex(zpack_writer *w, zpack_file_entry *entries, zpack_u64 file_count) {
    zpack_u64 block = file_count * ZPK_ENTRY_FIXED_BYTES;
    std::vector<zpack_u16> nlen((size_t)file_count);
    for (zpack_u64 i = 0; i < file_count; ++i) {
        size_t l = strlen(entries[i].filename);
        if (l > ZPK_MAX_NAME) return ZPACK_ERROR_FILENAME_TOO_LONG;
        nlen[i] = (zpack_u16)l;
        block += l;
    }
    std::vector<zpack_u8> b;
    try { b.resize((size_t)(ZPK_CDR_HEADER_BYTES + block)); } catch (const std::exception &) { return ZPACK_ERROR_MALLOC_FAILED; }
    put32(b.data(), ZPK_SIG_CDR);
    put64(b.data() + 4, file_count);
    put64(b.data() + 12, block);
    zpack_u8 *p = b.data() + ZPK_CDR_HEADER_BYTES;
    for (zpack_u64 i = 0; i < file_count; ++i) {
        put16(p, nlen[i]);
        memcpy(p + 2, entries[i].filename, nlen[i]);
        p += 2 + nlen[i];
        put64(p, entries[i].offset); put64(p + 8, entries[i].comp_size); put64(p + 16, entries[i].uncomp_size);
        put64(p + 24, entries[i].hash); p[32] = entries[i].comp_method;
        p += 33;
    }
    const zpack_u64 at = w->write_offset;
    int rc = sink_append(w, b.data(), b.size());
    if (rc) return rc;
    w->cdr_offset = at;
    return ZPACK_OK;
}
int zpack_write_cdr(zpack_writer *w) { return zpack_write_cdr_ex(w, w->file_entries, w->file_count); }
int zpack_write_eocdr_ex(zpack_writer *w, zpack_u64 cdr_offset) {
    zpack_u8 b[ZPK_EOCDR_BYTES];
    put32(b, ZPK_SIG_EOCDR);
    put64(b + 4, cdr_offset);
    return sink_append(w, b, sizeof b);
}
int zpack_write_eocdr(zpack_writer *w) { return zpack_write_eocdr_ex(w, w->cdr_offset); }
int zpack_write_archive(zpack_writer *w, zpack_file *files, zpack_u64 file_count) {
    int rc;
    if ((rc = zpack_write_header(w))) return rc;
    if ((rc = zpack_write_data_header(w))) return rc;
    if ((rc = zpack_write_files(w, files, file_count))) return rc;
    if ((rc = zpack_write_cdr(w))) return rc;
    return zpack_write_eocdr(w);
}
void zpack_close_writer(zpack_writer *w) {
    if (w->file) fclose(w->file);
    free(w->buffer);
    if (w->file_entries) {
        for (zpack_u64 i = 0; i < w->file_count; ++i) free(w->file_entries[i].filename);
        free(w->file_entries);
    }
    memset(w, 0, sizeof *w);
}

// ------------------------------------------------------------------------------------------------
// stream + utils
int zpack_init_stream(zpack_stream *s) {
    if (!s->xxh3_state) {
        s->xxh3_state = new (std::nothrow) StreamState();
        if (!s->xxh3_state) return ZPACK_ERROR_MALLOC_FAILED;
    }
    return ZPACK_OK;
}
void zpack_reset_stream(zpack_stream *s) { s->total_in = 0; s->total_out = 0; s->read_back = 0; }
void zpack_close_stream(zpack_stream *s) { delete state_of(s); s->xxh3_state = nullptr; }

// buffer sizes callers size their loops from (lib/zpack_read.c:719-758, lib/zpack_write.c:858-897): the values
// the reference returns (ZSTD_DStreamInSize() etc.), NONE falling through to the zstd ones
size_t zpack_get_dstream_in_size(zpack_compression_method m) { return m <= 1 ? 131075 : m == 2 ? 65551 : 0; }
size_t zpack_get_dstream_out_size(zpack_compression_method m) { return m <= 1 ? 131072 : m == 2 ? 65536 : 0; }
size_t zpack_get_cstream_in_size(zpack_compression_method m) { return m <= 1 ? 131072 : m == 2 ? 65536 : 0; }
size_t zpack_get_cstream_out_size(zpack_compression_method m) { return m <= 1 ? 131591 : m == 2 ? 65551 : 0; }

zpack_file_entry *zpack_get_file_entry(const char *filename, zpack_file_entry *entries, zpack_u64 n) {
    for (zpack_u64 i = 0; i < n; ++i)
        if (strcmp(entries[i].filename, filename) == 0) return entries + i;
    return nullptr;
}
zpack_bool zpack_read_stream_done(zpack_stream *s, zpack_file_entry *e) { return s->total_in == e->comp_size && s->read_back == 0; }

void *zpack_create_cctx(zpack_compression_method m) { return (m == ZPACK_COMPRESSION_ZSTD || m == ZPACK_COMPRESSION_LZ4) ? &g_ctx_token : nullptr; }
void *zpack_create_dctx(zpack_compression_method m) { return zpack_create_cctx(m); }
void zpack_free_cctx(zpack_compression_method, void *) {}
void zpack_free_dctx(zpack_compression_method, void *) {}

}  // extern "C"
