/* include/zpack_b200.h — the thin C-ABI between ZPack's host library and the sm_100a kernels.
 *
 * Plain C: pointers and sizes only, no torch / C++ types.  This is the layer that the
 * per-entry loops of the reference host library are rerouted through:
 *
 *   zpack_read_file        (/root/reference/lib/zpack_read.c:326-471)   -> zpb_unpack_host  (batch of 1)
 *   zpack_read_file_stream (/root/reference/lib/zpack_read.c:515-640)   -> zpb_unpack_host  (+ host doling)
 *   zpack_write_files      (/root/reference/lib/zpack_write.c:280-343)  -> zpb_pack_host
 *   zpack_compress_file    (/root/reference/lib/zpack_write.c:161-224)  -> zpb_pack_host    (per entry)
 *   XXH3_64bits call sites (zpack_read.c:466, zpack_write.c:256, zpack_stream.c) -> zpb_xxh3_*
 *
 * The *_device variants are the same operations with the archive / corpus already resident in
 * HBM (the configuration BASELINE.json's metric is quoted on).  Every function returns 0
 * (ZPB_OK) or a negative ZPB_E_* library error; per-entry outcomes are reported in `status[]`
 * using the reference's `enum zpack_result` numbering (lib/zpack.h:189-218).
 *
 * There is no CPU fallback: without a CUDA device zpb_create() fails and nothing else works.
 */
#ifndef ZPACK_B200_H
#define ZPACK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZPB_ABI_VERSION 1

/* library-level return codes */
#define ZPB_OK              0
#define ZPB_E_NO_DEVICE    -1   /* no CUDA device / driver                   */
#define ZPB_E_CUDA         -2   /* a CUDA call failed; see zpb_last_error()  */
#define ZPB_E_ARG          -3   /* bad argument (NULL, misaligned, overflow) */
#define ZPB_E_NOMEM        -4   /* device or pinned allocation failed        */
#define ZPB_E_IO           -5   /* pread / pwrite failed or the file is short */

/* compression methods — values of zpack_compression_method (lib/zpack.h:60-66) */
#define ZPB_METHOD_NONE 0
#define ZPB_METHOD_ZSTD 1
#define ZPB_METHOD_LZ4  2

/* per-entry status: the subset of enum zpack_result the hot path can produce */
#define ZPB_ST_OK                  0
#define ZPB_ST_BUFFER_TOO_SMALL   12
#define ZPB_ST_DECOMPRESS_FAILED  13
#define ZPB_ST_COMPRESS_FAILED    14
#define ZPB_ST_HASH_MISMATCH      15
#define ZPB_ST_OFFSET_INVALID     16
#define ZPB_ST_FILE_INCOMPLETE    17
#define ZPB_ST_FILE_SIZE_INVALID  18
#define ZPB_ST_METHOD_INVALID     19
#define ZPB_ST_NOT_AVAILABLE      24

/* One archive entry to unpack: the hot-path view of zpack_file_entry (lib/zpack.h:71-80)
 * plus where its output goes.  64 bytes, uploaded to the device as-is. */
typedef struct zpb_entry {
    uint64_t src_off;      /* entry.offset: byte offset of the compressed bytes in the archive */
    uint64_t comp_size;    /* entry.comp_size                                                  */
    uint64_t dst_off;      /* where to put the output inside the output buffer (16 B aligned)  */
    uint64_t dst_cap;      /* max_size of zpack_read_file (>= uncomp_size or BUFFER_TOO_SMALL)  */
    uint64_t uncomp_size;  /* entry.uncomp_size: the digest covers dst[0 .. uncomp_size)       */
    uint64_t hash;         /* entry.hash: expected XXH3-64                                     */
    uint32_t method;       /* entry.comp_method                                                */
    uint32_t flags;        /* ZPB_F_*                                                          */
    uint64_t reserved;
} zpb_entry;

#define ZPB_F_NO_VERIFY 1u  /* compute the digest but do not compare it (raw / hash-only use) */
#define ZPB_F_DISCARD   2u  /* zpb_unpack_host only: decode + verify on the device, do not copy the bytes back —
                             * the archive integrity test (`zpack t`, programs/commands.c) needs the verdict only */

/* One file to pack: the hot-path view of zpack_file (lib/zpack.h:125-134). */
typedef struct zpb_file {
    uint64_t src_off;      /* offset of the file's bytes inside the input buffer (16 B aligned) */
    uint64_t size;         /* zpack_file.size                                                   */
    uint64_t dst_off;      /* offset of this file's output slot in the output buffer            */
    uint64_t dst_cap;      /* slot capacity, >= zpb_pack_bound(method, size)                    */
    uint32_t method;       /* options->method                                                   */
    int32_t  level;        /* options->level (LZ4: < 3 = fast path, negative = acceleration)    */
    uint64_t reserved[3];
} zpb_file;

typedef struct zpb_ctx zpb_ctx;

/* lifecycle ------------------------------------------------------------------------------- */
int         zpb_abi_version(void);
zpb_ctx    *zpb_create(int device);              /* NULL on failure; zpb_last_error(NULL) says why */
void        zpb_destroy(zpb_ctx *ctx);
const char *zpb_last_error(const zpb_ctx *ctx);  /* never NULL */
int         zpb_device_info(const zpb_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor);
/* counts every kernel this library has launched on this context (bench "gpu_launches") */
uint64_t    zpb_launch_count(const zpb_ctx *ctx);

/* unpack + verify ------------------------------------------------------------------------- */
/* Device-resident batch.  d_archive/d_out are device pointers; entries/status/digest are HOST
 * arrays of n elements (descriptor upload and result download are part of the call).
 * `stream` is a cudaStream_t (NULL = the context's own stream).  Synchronous on return. */
int zpb_unpack_device(zpb_ctx *ctx, const uint8_t *d_archive, uint64_t archive_size,
                      uint8_t *d_out, uint64_t out_size, const zpb_entry *entries, uint64_t n,
                      int32_t *status, uint64_t *digest, void *stream);

/* Same with host buffers: copies [lo,hi) of the archive that the entries touch to the device,
 * unpacks, copies each entry's uncomp_size bytes back into h_out + dst_off.  Batches of more than a few
 * hundred MB are pipelined in chunks over several streams (H2D, kernels and D2H of different chunks
 * overlap); pinned host buffers are needed for the copies to be asynchronous. */
int zpb_unpack_host(zpb_ctx *ctx, const uint8_t *h_archive, uint64_t archive_size,
                    uint8_t *h_out, uint64_t out_size, const zpb_entry *entries, uint64_t n,
                    int32_t *status, uint64_t *digest);

/* one large entry, sharded by blocks ------------------------------------------------------- */
/* Intra-entry parallelism (BASELINE config C5): an LZ4 entry whose frame has INDEPENDENT 64 KB blocks
 * (FLG B.Indep = 1 — what zpb_pack_* writes; the reference reader accepts both modes,
 * /root/reference/externals/lz4/lib/lz4frame.c:1151,1676) is decoded one warp per block, and a contiguous
 * run of its blocks can be given to each GPU.  Replaces, for such an entry, the LZ4F_decompress loop and the
 * XXH3_64bits pass of zpack_read_file (/root/reference/lib/zpack_read.c:396-468).  Reference-written
 * (block-linked) and zstd entries are one dependency chain each and stay on zpb_unpack_*. */
typedef struct zpb_block {
    uint64_t src_off;      /* archive offset of the block payload (after its 4-byte header) */
    uint32_t comp_size;    /* payload bytes                                                */
    uint32_t flags;        /* ZPB_BLK_STORED: payload is the data itself (header bit 31)    */
} zpb_block;
#define ZPB_BLK_STORED 1u
#define ZPB_INDEX_UNSUPPORTED 1   /* zpb_lz4_frame_index: not a single checksum-free B.Indep frame of 64 KB blocks */

/* Host-side framing walk (no codec work): header checks of LZ4F_decodeHeader (lz4frame.c:1113-1205) and the
 * block-header chain (lz4frame.c:1503-1531) of the frame at h_frame[0..comp_size).  `archive_off` is added to
 * every src_off (the entry's offset in the archive).  Writes up to `cap` blocks, always sets *n_blocks.
 * *content_size = the frame's content-size field or ~0 if absent.  Returns ZPB_OK, ZPB_INDEX_UNSUPPORTED
 * (use zpb_unpack_* instead), or ZPB_E_ARG. */
int zpb_lz4_frame_index(const uint8_t *h_frame, uint64_t comp_size, uint64_t archive_off, zpb_block *blocks,
                        uint64_t cap, uint64_t *n_blocks, uint32_t *block_size, uint64_t *content_size);

/* Decode blocks[0..n) — a contiguous run of one entry's blocks — into d_out + k * block_size.
 * shard_uncomp_size = decoded bytes of the run: every block but the run's last must decode to exactly
 * block_size (LZ4F writers fill blocks, lz4frame.c:873-882); only the entry's last shard may end short.
 * *status: 0, ZPB_ST_OFFSET_INVALID, or ZPB_ST_NOT_AVAILABLE = this path declines the shard (a block is
 * malformed or has a shape only the general decoder judges) — re-read the entry with zpb_unpack_device for
 * the reference's verdict.  The shard's per-KiB XXH3 stripe sums stay in the context for zpb_blocks_digest. */
int zpb_unpack_blocks_device(zpb_ctx *ctx, const uint8_t *d_archive, uint64_t archive_size, uint8_t *d_out,
                             uint64_t out_size, const zpb_block *blocks, uint64_t n, uint32_t block_size,
                             uint64_t shard_uncomp_size, int32_t *status, void *stream);

/* XXH3-64 scramble chain (xxhash.h:3527-3534, 3698) over the last decoded shard, which covers entry bytes
 * [shard_pos, shard_pos + shard_uncomp_size) of total_size.  acc_in: the 8 accumulators the previous shard
 * ended with (HOST pointer; NULL = first shard, XXH3_INIT_ACC); acc_out (HOST, may be NULL) receives the
 * state to hand to the next shard — 64 bytes is the only data that ever moves between GPUs.  For the
 * entry's last shard, d_out (its decoded bytes, device) and digest (HOST) are required: the tail stripes
 * and the merge (xxhash.h:3701-3747) run there. */
int zpb_blocks_digest(zpb_ctx *ctx, const uint64_t *acc_in, uint64_t *acc_out, uint64_t shard_pos,
                      uint64_t total_size, const uint8_t *d_out, uint64_t *digest, void *stream);
/* zpack_read_file for ONE large block-independent LZ4 entry with host buffers: frame index, then chunks of
 * blocks pipelined over the context's worker streams (H2D / decode / chain / D2H overlap), the XXH3 state
 * relayed chunk to chunk.  Returns ZPB_OK with *status = the entry's zpack_result, or ZPB_INDEX_UNSUPPORTED
 * when the entry is not eligible (linked blocks, checksums, sizes that do not add up, a block the fast
 * kernels decline) — the caller then uses zpb_unpack_host, which decodes anything.  flags: ZPB_F_*. */
int zpb_unpack_entry_blocks_host(zpb_ctx *ctx, const uint8_t *h_entry, uint64_t comp_size, uint8_t *h_out,
                                 uint64_t out_cap, uint64_t uncomp_size, uint64_t expect_hash, uint32_t flags,
                                 int32_t *status, uint64_t *digest);
/* device time of xxh3_chain_kernel in the last zpb_blocks_digest (ms) */
int zpb_last_chain_ms(const zpb_ctx *ctx, float *ms);

/* XXH3-64 (seed 0) of n independent ranges ------------------------------------------------- */
int zpb_xxh3_device(zpb_ctx *ctx, const uint8_t *d_data, const uint64_t *offsets,
                    const uint64_t *lengths, uint64_t n, uint64_t *digest, void *stream);
int zpb_xxh3_host(zpb_ctx *ctx, const uint8_t *h_data, uint64_t length, uint64_t *digest);

/* pack ------------------------------------------------------------------------------------ */
/* worst-case output bytes for one file (LZ4: frame header + per-block headers + EndMark) */
uint64_t zpb_pack_bound(uint32_t method, uint64_t size);

/* Compress n files that are resident in HBM into their slots; returns per-file compressed
 * size, XXH3-64 of the input and status.  The compressed-size prefix sum / entry.offset
 * assignment is the caller's (host) job, as in zpack_write_files. */
int zpb_pack_device(zpb_ctx *ctx, const uint8_t *d_in, uint64_t in_size, uint8_t *d_out,
                    uint64_t out_size, const zpb_file *files, uint64_t n, uint64_t *comp_size,
                    uint64_t *digest, int32_t *status, void *stream);
/* The same with host buffers: large batches are cut into chunks over worker streams (H2D of a chunk's input, kernel,
 * on-device gather of the frames, one D2H, host scatter into the slots at files[i].dst_off); bytes of h_out outside
 * [dst_off, dst_off + comp_size[i]) are not written. */
int zpb_pack_host(zpb_ctx *ctx, const uint8_t *h_in, uint64_t in_size, uint8_t *h_out,
                  uint64_t out_size, const zpb_file *files, uint64_t n, uint64_t *comp_size,
                  uint64_t *digest, int32_t *status);
/* LZ4 levels 3 and above (LZ4 HC in the reference, lz4frame.c:799-807).  0 (the default; env ZPB_LZ4HC=1 turns it on
 * at zpb_create): such files get ZPB_ST_NOT_AVAILABLE.  1: they are compressed by the HC block compressor — hash chains
 * searched up to a level-dependent depth and a cost-based parse per 64 KB block; levels above 12 act as 12.  The frames
 * have the same layout as the fast path's (block-independent, 64 KB blocks).  Levels below 3, zstd and stored files are
 * the same either way.  Like every setting of a context, it reaches the worker contexts of the pipelined host calls
 * (zpb_unpack_host, zpb_pack_host, zpb_unpack_entry_blocks_host) at the start of every call. */
int zpb_set_lz4hc(zpb_ctx *ctx, int enabled);

/* last kernel timing (CUDA events on the launching stream), for bench.py's roofline block */
int zpb_last_kernel_ms(const zpb_ctx *ctx, float *unpack_ms, float *pack_ms);
/* The last zpb_pack_device call by stage, summed over its rounds: the block compressors (lz4_pack_blocks_kernel, the
 * role of LZ4_compress_fast_extState under lz4frame.c:735-760, and the HC kernels lz4hc_match_kernel + lz4hc_parse_kernel)
 * and the framing + XXH3 kernel (lz4_pack_kernel). */
int zpb_last_pack_stage_ms(const zpb_ctx *ctx, float *blocks_ms, float *frames_ms);

/* per-stage device time of the last unpack (ms): scan, parse, exec, general-fallback.  With the overlap on (the
 * default, zpb_set_overlap) parse and exec run concurrently, so the two intervals overlap and exec's includes the time
 * its early grid had to share the SMs with the parse kernel; zpb_last_kernel_ms is first launch to last either way. */
int zpb_last_stage_ms(const zpb_ctx *ctx, float *ms4);
/* device time of zstd_unpack_kernel in the last unpack (ms; 0 when the batch had no zstd entry) */
int zpb_last_zstd_ms(const zpb_ctx *ctx, float *ms);
/* 1 (default): LZ4 / stored entries go through the scan -> parse -> exec pipeline and only what it
 * declines reaches the general decoder; 0: general decoder for everything (A/B and test use). */
int zpb_set_fast_path(zpb_ctx *ctx, int enabled);
/* 1 (default; env ZPB_OVERLAP): the execute kernel starts as soon as the scan has finished and overlaps the tail of the
 * parse kernel (separate streams, entries whose blocks are not parsed yet are put aside for a last pass);
 * 0: scan, parse, execute back to back on one stream — what per-kernel timings (zpb_last_stage_ms) are meaningful for. */
int zpb_set_overlap(zpb_ctx *ctx, int enabled);

/* several GPUs of one box, one call ------------------------------------------------------------ */
/* What a multi-GPU caller of the reference's read / write loops binds: the per-entry loop of a batch reader
 * (zpack_read_file over the entries of an archive, /root/reference/lib/zpack_read.c:326-471, which the reference allows from
 * several threads with one context each, lib/zpack.h:335-341) and zpack_write_files (lib/zpack_write.c:280-343), spread over
 * the GPUs of the box.  Entries / files are independent: a batch is cut into contiguous runs in archive order, balanced by
 * decoded bytes, one run per device, each driven from its own host thread through zpb_unpack_host / zpb_pack_host.
 * No collective, no peer traffic (there is nothing to reduce); every device copies only the archive range it needs. */
typedef struct zpb_group zpb_group;
int         zpb_device_count(void);                            /* visible CUDA devices (0: none, or no driver) */
zpb_group  *zpb_group_create(const int *devices, int n);        /* devices == NULL or n <= 0: every visible device */
void        zpb_group_destroy(zpb_group *g);
int         zpb_group_size(const zpb_group *g);
zpb_ctx    *zpb_group_ctx(zpb_group *g, int k);                  /* the k-th device's context (tuning, timings) */
const char *zpb_group_last_error(const zpb_group *g);
/* order[n]: the entries in archive order; cuts[world + 1]: device k takes order[cuts[k] .. cuts[k+1]) */
int zpb_group_partition(const zpb_entry *entries, uint64_t n, int world, uint64_t *order, uint64_t *cuts);
int zpb_group_unpack_host(zpb_group *g, const uint8_t *h_archive, uint64_t archive_size, uint8_t *h_out,
                          uint64_t out_size, const zpb_entry *entries, uint64_t n, int32_t *status, uint64_t *digest);
int zpb_group_pack_host(zpb_group *g, const uint8_t *h_in, uint64_t in_size, uint8_t *h_out, uint64_t out_size,
                        const zpb_file *files, uint64_t n, uint64_t *comp_size, uint64_t *digest, int32_t *status);
/* zpb_group_unpack_host and zpb_group_pack_host both record it, on a group of one device too */
int zpb_group_last_ms(const zpb_group *g, float *ms, int cap);   /* wall time of each device's share of the last call */
/* pinned host memory for the *_host entry points (pageable buffers make their copies synchronous) */
void *zpb_host_alloc(uint64_t bytes);
void  zpb_host_free(void *p);

/* the container level on the device -------------------------------------------------------------- */
/* SURVEY §8(f) rows 1 and 4: an archive image that stays in HBM is opened, assembled and copied entry by entry without a
 * host pass over its bytes.  The host side of each call touches only the per-entry table it is given (argument checks and
 * two sums) and the 42 fixed bytes of an archive.
 *
 *   zpb_archive_open_device   zpack_read_archive_memory -> zpack_read_cdr_memory -> zpack_read_file_entries_memory
 *                             (/root/reference/lib/zpack_read.c:225-260, 168-188, 109-166), without its malloc per entry
 *   zpb_archive_build_device  the offset table of zpack_write_files (ZPACK_ADD_OFFSET_AND_SIZE, lib/zpack_write.c:280-343),
 *                             zpack_write_header / _data_header, zpack_write_cdr_ex, zpack_write_eocdr
 *                             (lib/zpack_write.c:640-685, 713-776, 778-800) and the payload moves in between
 *   zpb_copy_entries_device   the memcpy loop of zpack_write_files_from_archive (lib/zpack_write.c:345-428) */
typedef struct zpb_arc_entry {
    uint64_t src_off;      /* where the entry's compressed bytes are in the source buffer (a pack slot, or entry.offset of the
                            * archive it is copied from); open: = offset                                                  */
    uint64_t comp_size;    /* entry.comp_size                                                                            */
    uint64_t uncomp_size;  /* entry.uncomp_size                                                                          */
    uint64_t hash;         /* entry.hash                                                                                 */
    uint64_t name_off;     /* of the file name inside the names blob (not NUL-terminated)                                */
    uint32_t name_len;     /* <= 65535 (ZPACK_MAX_FILENAME_LENGTH, lib/zpack.h:48)                                       */
    uint32_t method;       /* entry.comp_method                                                                          */
    uint64_t offset;       /* entry.offset in the archive: written by build, read by copy (the destination), = src_off after open */
    uint64_t reserved;
} zpb_arc_entry;

/* Parse the central directory of the archive image at d_archive (device).  *result = the zpack_result the reference's open
 * returns for these bytes (0, FILE_TOO_SMALL 5, SIGNATURE_INVALID 6, READ_FAILED 7, BLOCK_SIZE_INVALID 8,
 * VERSION_INCOMPATIBLE 9); *n = the directory's file count as soon as its header is readable.  entries (HOST, cap elements)
 * receives one row per file; names (HOST, optional, names_cap >= *names_size) receives the directory block that name_off
 * points into.  ZPB_E_ARG when cap < *n (call again with a larger table) or the directory is >= 4 GB. */
int zpb_archive_open_device(zpb_ctx *ctx, const uint8_t *d_archive, uint64_t archive_size, zpb_arc_entry *entries, uint64_t cap,
                            uint64_t *n, uint8_t *names, uint64_t names_cap, uint64_t *names_size, int32_t *result, void *stream);
/* Write a whole archive into d_archive (device): header, the n payloads back to back in table order (read from d_src +
 * src_off: pack slots, or another archive), central directory, end record.  entries / names are HOST arrays; offset of every
 * entry is assigned on the device and returned in the table.  d_src and d_archive must not overlap. */
int zpb_archive_build_device(zpb_ctx *ctx, const uint8_t *d_src, uint64_t src_size, zpb_arc_entry *entries, uint64_t n,
                             const uint8_t *names, uint64_t names_size, uint8_t *d_archive, uint64_t archive_cap,
                             uint64_t *archive_size, void *stream);
/* d_dst[offset .. offset + comp_size) = d_src[src_off .. src_off + comp_size) for every entry; ranges of different entries
 * must not overlap in d_dst, and d_dst must not overlap d_src. */
int zpb_copy_entries_device(zpb_ctx *ctx, const uint8_t *d_src, uint64_t src_size, uint8_t *d_dst, uint64_t dst_size,
                            const zpb_arc_entry *entries, uint64_t n, void *stream);
/* device time (ms) of the last call's kernels: [0] offset table + directory + copy work items, [1] the payload copy kernel, [2] directory parse */
int zpb_last_archive_ms(const zpb_ctx *ctx, float *ms3);
/* File <-> HBM for a device-resident archive: bytes [file_off, file_off + size) of the open file descriptor fd to / from
 * device memory, read / written by several host threads through pinned buffers on their own streams (pread, H2D and the next
 * pread overlap; no GPUDirect-Storage driver is assumed).  Replaces the reference's fread of entry and directory bytes
 * (/root/reference/lib/zpack_read.c:298-324, 190-223) and its seek + fwrite (lib/zpack_common.c:72-81) when the other side of
 * the transfer is the device.  ZPB_E_IO when the file is shorter than the range or a system call fails. */
int zpb_file_read_device(zpb_ctx *ctx, int fd, uint64_t file_off, uint64_t size, uint8_t *d_dst);
int zpb_file_write_device(zpb_ctx *ctx, int fd, uint64_t file_off, uint64_t size, const uint8_t *d_src);

/* tuning knobs: lanes per dependency chain (4, 8, 16, 32; 0 = keep) and resident CTAs per SM
 * (0 = occupancy API, -1 = keep).  Defaults can also come from ZPB_GROUP / ZPB_CTAS_PER_SM. */
int zpb_set_tuning(zpb_ctx *ctx, int group_lanes, int ctas_per_sm);

#ifdef __cplusplus
}
#endif
#endif /* ZPACK_B200_H */
