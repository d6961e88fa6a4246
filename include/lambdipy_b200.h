/*
 * lambdipy_b200.h -- C ABI of the B200 (sm_100a) ELF strip library, liblambdipy_b200.so.
 *
 * What it replaces.  The reference (customink/lambdipy) has no FFI for this step: it strips the
 * build tree by running one shell line inside a generated script,
 *
 *     find {install_dir}/ -name "*.so" | xargs strip        /root/reference/lambdipy/project_build.py:260
 *
 * executed by install_non_resolved_requirements() (project_build.py:234-277; Popen at :268, docker
 * exec at :274) before the script is removed (:277).  The entry points below are what a ctypes
 * binding placed at that spot calls instead (see INTEGRATION.md for the reference-side stub):
 *
 *   lb2_strip_tree()          == the whole shell line: select basename "*.so" under a root
 *                                (find, :260), strip each regular ELF in place (strip, :260) the way
 *                                GNU strip 2.42 does: new contents written into the EXISTING inode
 *                                (mode, owner and other hard links kept; mtime not).
 *   lb2_strip_host()          == `strip` over a batch of files already read into host memory
 *                                (what xargs hands to one strip process), results to host memory.
 *   lb2_strip_device_async()  == the same batch with input and output arenas resident in HBM
 *                                (benchmark / pipeline building block).
 *
 * Result contract: for every file with status LB2_ST_OK the output bytes are identical to
 * `strip --strip-unneeded -o OUT IN` of GNU Binutils 2.42 (== flagless `strip` for ET_DYN/ET_EXEC).
 * Files the device planner does not cover get a positive status and no output; lb2_strip_tree can
 * hand exactly those to the host `strip` binary (LB2_TREE_FALLBACK_HOST_STRIP) so the tree ends up
 * identical to the reference's, and reports how many took that route.
 *
 * Conventions: plain C types; the caller owns every buffer it passes; the library keeps no pointer
 * past a call except where stated (async call: until lb2_batch_results); functions return 0 on
 * success or a negative LB2_E_* code and never throw; one context per thread and device.
 * There is no CPU implementation behind this ABI: without a CUDA device lb2_ctx_create fails.
 */
#ifndef LAMBDIPY_B200_H
#define LAMBDIPY_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct lb2_ctx lb2_ctx;

/* library return codes */
enum {
  LB2_OK = 0,
  LB2_E_CUDA = -1,        /* CUDA runtime error; text in lb2_last_error */
  LB2_E_ARG = -2,         /* bad argument (NULL, unaligned offsets, ...) */
  LB2_E_CAPACITY = -3,    /* output arena too small; stats.out_bytes_needed says how much */
  LB2_E_IO = -4,          /* filesystem error in lb2_strip_tree */
  LB2_E_NODEVICE = -5,    /* no usable CUDA device */
  LB2_E_STATE = -6        /* call out of order (no batch in flight, ...) */
};

/* per-file status written by the plan kernel */
enum {
  LB2_ST_OK = 0,
  LB2_ST_NOT_ELF = 1,            /* GNU strip: "file format not recognized" */
  LB2_ST_NOT_ELF64LE = 2,
  LB2_ST_BAD_TYPE = 3,           /* ET_REL, ET_CORE ... */
  LB2_ST_NO_SECTIONS = 4,        /* GNU strip: "has no sections" */
  LB2_ST_XINDEX = 5,
  LB2_ST_UNSUPPORTED_LAYOUT = 6, /* a layout rule the planner does not implement */
  LB2_ST_BAD_NOTES = 7,          /* corrupt .gnu.build.attributes (objcopy refuses too) */
  LB2_ST_PLANNER_LIMIT = 8,      /* > 64 sections, > 32 phdrs, > 2 KB of section names, > 8 KB notes */
  LB2_ST_MALFORMED = -1
};

/* flags for the strip calls */
#define LB2_F_NO_MERGE_NOTES 1u /* behave like `strip --no-merge-notes` */

/* flags for lb2_strip_tree */
#define LB2_TREE_FALLBACK_HOST_STRIP 0x100u /* unsupported ELF files: run the host `strip` on them  */
#define LB2_TREE_TOLERATE_NON_ELF    0x200u /* non-ELF "*.so": leave untouched (reference: rc 123)   */
#define LB2_TREE_DRY_RUN             0x400u /* plan + compact, write nothing                         */
#define LB2_TREE_CLEANUP             0x800u /* also do the script's rm lines (project_build.py:256-259) on the walk */

typedef struct lb2_stats {
  uint32_t n_files, n_ok, n_unsupported, overflow;
  uint64_t in_bytes;          /* input bytes of the n_ok files                                  */
  uint64_t out_bytes;         /* OUT: stripped bytes written                                    */
  uint64_t copy_bytes;        /* C:   extent bytes read (input arena + regenerated literals)    */
  uint64_t header_bytes;      /* H:   header/table/note bytes the planner parsed                */
  uint64_t n_tiles;
  uint64_t out_bytes_needed;  /* 256-byte-rounded arena bytes the batch needs                   */
  float plan_ms;              /* plan + offset scan kernels, CUDA events on the call's stream   */
  float compact_ms;           /* compaction kernel                                              */
  float h2d_ms, d2h_ms;       /* lb2_strip_host only: summed copy time                          */
  uint64_t h2d_bytes;         /* lb2_strip_host only: bytes that crossed the bus upwards (DMA'd ranges, or what the   */
  uint64_t d2h_bytes;         /*   kernels pulled in zero-copy mode) and downwards                                    */
} lb2_stats;

typedef struct lb2_tree_stats {
  uint32_t n_selected;        /* paths whose basename ends in the suffix                        */
  uint32_t n_gpu;             /* replaced with GPU-produced bytes                               */
  uint32_t n_fallback;        /* handed to the host `strip`                                     */
  uint32_t n_skipped;         /* symlinks, directories, tolerated non-ELF                       */
  uint32_t n_failed;          /* would make the reference's script exit non-zero                */
  uint32_t n_removed;         /* LB2_TREE_CLEANUP: *.egg-info, *.dist-info, __pycache__, tests entries removed */
  uint64_t in_bytes, out_bytes;
  double walk_read_s;         /* directory walk + stat                                          */
  double gpu_s;               /* kernels + result fetch, summed over batches                    */
  double write_s;             /* file reads/uploads and downloads/writes (overlapped), wall     */
  double fallback_s;          /* host `strip` on the files the planner refused                  */
  double read_cpu_s;          /* summed over the I/O threads: time inside pread                 */
  double write_cpu_s;         /* ... inside pwrite / truncate                                   */
  double dma_wait_s;          /* ... issuing and waiting for the slot DMAs                      */
  uint32_t io_threads, n_batches;
  lb2_stats batch;
} lb2_tree_stats;

/* ---- context ---------------------------------------------------------------------------- */
int lb2_ctx_create(int device, lb2_ctx **ctx);
void lb2_ctx_destroy(lb2_ctx *ctx);
const char *lb2_last_error(const lb2_ctx *ctx); /* ctx may be NULL: error of the failed create */
const char *lb2_version(void);
int lb2_sm_count(const lb2_ctx *ctx);

/* ---- device / pinned memory for callers without their own CUDA runtime (ctypes) ---------- */
void *lb2_dev_alloc(lb2_ctx *ctx, uint64_t bytes);
void lb2_dev_free(lb2_ctx *ctx, void *p);
void *lb2_pinned_alloc(lb2_ctx *ctx, uint64_t bytes); /* pinned + device-mapped, on the GPU's NUMA node (LB2_NUMA=0: anywhere) */
void lb2_pinned_free(lb2_ctx *ctx, void *p);
int lb2_memcpy_h2d(lb2_ctx *ctx, void *d_dst, const void *h_src, uint64_t bytes);
int lb2_memcpy_d2h(lb2_ctx *ctx, void *h_dst, const void *d_src, uint64_t bytes);
int lb2_memset_d(lb2_ctx *ctx, void *d_dst, int value, uint64_t bytes);

/* ---- strip a batch resident in HBM ------------------------------------------------------ */
/* d_in: input arena; file f occupies [h_in_off[f], h_in_off[f+1]) minus padding -- offsets must be
 * multiples of 16 and h_in_sizes[f] gives the exact byte length (NULL: use the offset difference).
 * d_out: output arena of out_capacity bytes; file f lands at out_off[f] (multiples of 256).
 * Enqueues upload of the offsets, the plan kernel, the offset scan and the compaction kernel on
 * `stream` (a cudaStream_t; NULL = the context's own stream) and returns without synchronising.  Up to TWO
 * batches may be in flight (the second is queued behind the first on the stream, so the GPU does not idle while the
 * host collects); lb2_batch_results collects them in order.  Batches that share an output arena overwrite it. */
int lb2_strip_device_async(lb2_ctx *ctx, const void *d_in, const uint64_t *h_in_off, const uint64_t *h_in_sizes,
                           uint32_t n_files, void *d_out, uint64_t out_capacity, uint32_t flags, void *stream);
/* Waits for the OLDEST batch in flight, copies its offsets/status back.  Any pointer may be NULL. */
int lb2_batch_results(lb2_ctx *ctx, uint64_t *h_out_off /* n+1 */, uint64_t *h_out_sizes /* n */,
                      int32_t *h_status /* n */, lb2_stats *stats);

/* ---- strip a shard whose input + output do not fit side by side in HBM ------------------------- */
/* Input arena resident (as above); the output is streamed through a ring of TWO slots of slot_capacity
 * bytes each at d_out_ring: consecutive files are grouped into chunks of <= max_chunk_bytes of arena span
 * (0 = slot_capacity), chunk k is written to slot k % 2 and handed to on_chunk (may be NULL) before the
 * slot is reused two chunks later -- the consumer owns the slot only for the duration of the callback.
 * Offsets passed to the callback are relative to the slot.  h_out_sizes / h_status (n_files each, may be
 * NULL) receive the per-file results; *total sums the chunks (plan_ms / compact_ms: summed kernel times).
 * This is what one `strip` process does to an argument list longer than memory: SURVEY.md D7, the
 * 10 000-file corpus of BASELINE config 4 on one GPU (/root/reference/lambdipy/project_build.py:260). */
typedef int (*lb2_chunk_fn)(void *user, uint32_t chunk, uint32_t first_file, uint32_t n_files, const void *d_out_slot,
                            const uint64_t *out_off, const uint64_t *out_sizes, const int32_t *status,
                            const lb2_stats *chunk_stats);
int lb2_strip_device_chunked(lb2_ctx *ctx, const void *d_in, const uint64_t *h_in_off, const uint64_t *h_in_sizes,
                             uint32_t n_files, void *d_out_ring, uint64_t slot_capacity, uint64_t max_chunk_bytes,
                             uint32_t flags, void *stream, lb2_chunk_fn on_chunk, void *user, uint64_t *h_out_sizes,
                             int32_t *h_status, lb2_stats *total);

/* ---- strip a batch held in host memory ---------------------------------------------------- */
/* h_out_off[f] (multiples of 256) and h_out_sizes[f] describe where file f was written in h_out.
 * When both arenas are pinned and device-mapped (lb2_pinned_alloc, cudaHostAlloc, cudaHostRegister) the
 * kernels run on them directly over PCIe (zero-copy: only headers and kept extents are pulled, stripped
 * files are pushed straight back; LB2_HOST_ZEROCOPY=0 disables).  LB2_HOST_DMA=1 selects the copy-engine
 * variant instead: plan over the mapping, DMA of the kept ranges into a device slot, compaction in HBM, DMA
 * of the output (same bytes on the bus, measured within 3 % of zero-copy).  Otherwise, or when both are
 * disabled: explicit H2D of whole files -> kernels -> D2H, pipelined in <= LB2_CHUNK_MB (256) MB chunks of
 * whole files on three streams.  stats->h2d_bytes / d2h_bytes say what crossed the bus. */
int lb2_strip_host(lb2_ctx *ctx, const void *h_in, const uint64_t *h_in_off, const uint64_t *h_in_sizes,
                   uint32_t n_files, void *h_out, uint64_t out_capacity, uint64_t *h_out_off, uint64_t *h_out_sizes,
                   int32_t *h_status, uint32_t flags, lb2_stats *stats);

/* ---- strip a directory tree in place (the reference's shell line) ------------------------ */
int lb2_strip_tree(lb2_ctx *ctx, const char *root, const char *suffix /* ".so" */, uint32_t flags,
                   lb2_tree_stats *stats);
/* The same with the sibling clean-up lines of the reference's script folded into the directory walk
 * (flag LB2_TREE_CLEANUP; /root/reference/lambdipy/project_build.py:256-259):
 *     rm -rf ROOT/{glob}.egg-info ROOT/{glob}.dist-info          (top level only, shell glob: no dot files)
 *     find ROOT/ -name __pycache__ | xargs rm -rf
 *     find ROOT/ -name tests | grep -v "KEEP" | xargs rm -rf      KEEP = keep_tests_regex, a grep basic regex on
 *                                                                the printed path; the reference passes "*" when
 *                                                                --keep-tests is not given, 'a\|b' otherwise (:249)
 * They run before the selection, as in the script: objects under a removed directory are not stripped. */
int lb2_strip_tree_ex(lb2_ctx *ctx, const char *root, const char *suffix, uint32_t flags, const char *keep_tests_regex,
                      lb2_tree_stats *stats);
/* Only the clean-up lines (no GPU, no context needed). */
int lb2_tree_cleanup(const char *root, const char *keep_tests_regex, uint32_t *n_removed);
/* Optional: pay lb2_strip_tree's first-use costs (pinned slot ring, I/O streams, device workspaces) now,
 * e.g. on a helper thread while the reference's script is still running pip
 * (/root/reference/lambdipy/project_build.py:266-268).  expected_tree_bytes sizes the ring (0 = default). */
int lb2_tree_prepare(lb2_ctx *ctx, uint64_t expected_tree_bytes);

/* ---- plan only: per-file output sizes and status, nothing copied (tests) ------------------ */
int lb2_plan_device(lb2_ctx *ctx, const void *d_in, const uint64_t *h_in_off, const uint64_t *h_in_sizes,
                    uint32_t n_files, uint32_t flags, uint64_t *h_out_sizes, int32_t *h_status, lb2_stats *stats);

/* ---- synthetic corpus: fill payload regions of an HBM arena with counter-based random bytes - */
typedef struct lb2_fill_region {
  uint64_t offset; /* byte offset in the arena */
  uint64_t len;
} lb2_fill_region;
/* byte at arena offset o = byte (o & 7) of splitmix64(seed + (o >> 3)); independent of the region
 * split, so host and device generators agree. */
int lb2_corpus_fill(lb2_ctx *ctx, void *d_arena, const lb2_fill_region *h_regions, uint32_t n_regions,
                    uint64_t seed, void *stream);

/* Copies n host-built blobs (ELF headers, notes, string tables) into the arena:
 * arena[h_dst[i] .. +h_len[i]) = h_data[h_src[i] .. +h_len[i]).  Synchronous. */
int lb2_corpus_scatter(lb2_ctx *ctx, void *d_arena, const void *h_data, uint64_t data_bytes, const uint64_t *h_dst,
                       const uint64_t *h_src, const uint64_t *h_len, uint32_t n);

/* ---- gzip release tarballs (DEFLATE on the GPU) ------------------------------------------ */
/* Replaces the compression of
 *     with tarfile.open(tarball_path, "w:gz") as tar: tar.add(path, arcname=...)
 *                                              /root/reference/lambdipy/package_build.py:165-172
 * (zlib level 9, one CPU core).  The stream is cut into 64 KiB chunks compressed independently by one CTA
 * each (back-references reach 32 KiB into the preceding input); every non-final chunk ends with an empty
 * stored block.  The result inflates to exactly the input; its bytes differ from zlib's.  The output is a
 * pure function of the input bytes (and, for lb2_gzip_segments, independent of the window size). */
typedef struct lb2_gzip_stats {
  uint64_t in_bytes, out_bytes;  /* uncompressed input, compressed output (deflate stream only)                 */
  float kernel_ms;               /* deflate kernel + concatenation, CUDA events, summed over windows             */
  double read_s;                 /* lb2_gzip_segments: pread + memcpy into the pinned slots, summed over workers  */
  double upload_s;               /* wall time spent waiting for window uploads (window 0, then what compressing
                                    the previous window did not hide)                                           */
  double download_s, write_s;    /* D2H of the compressed output, pwrite of header / stream / trailer, wall       */
  double setup_s;                /* buffer allocation inside this call (0 once the context's buffers are large enough) */
  uint64_t n_chunks;
  uint32_t n_windows, io_threads;
  uint64_t phase_cycles[6];      /* SM cycles summed over CTAs: hash sort, scatter, match search, lazy parse,
                                    Huffman + header, emit                                                      */
} lb2_gzip_stats;

/* Raw DEFLATE of n bytes at d_in (HBM) into d_out (cap bytes).  `hist` bytes before d_in (at most 32768
 * are used) are history: back-references may reach into them, they are not emitted.  final != 0: the last
 * block has BFINAL=1; final == 0: the stream ends with a sync flush and may be continued by a later call
 * whose history is this call's last 32 KiB.  *crc32 = CRC-32 of the n bytes.  Synchronous on `stream`
 * (NULL: the context's stream).  cap too small: LB2_E_CAPACITY, *out_len = bytes needed.  A bound for cap:
 * ceil(n / 65536) * 66560 (or 66560 when n == 0). */
int lb2_deflate_device(lb2_ctx *ctx, const void *d_in, uint64_t n, uint32_t hist, uint32_t final, void *d_out,
                       uint64_t cap, uint64_t *out_len, uint32_t *crc32, lb2_gzip_stats *stats, void *stream);

/* One piece of the uncompressed stream: `data` != NULL: len literal bytes; else the first len bytes of
 * the regular file `path`. */
typedef struct lb2_gz_segment {
  const void *data;
  const char *path;
  uint64_t len;
} lb2_gz_segment;
/* Writes out_path = gz_header (gz_header_len bytes, as given), the DEFLATE stream of the concatenated
 * segments, CRC-32 and ISIZE (little-endian, ISIZE mod 2^32).  The stream is processed in windows of
 * LB2_GZ_WINDOW_MB (default 1024) MB, each primed with the previous window's last 32 KiB; reading window
 * k+1 overlaps compressing and writing window k.  File bodies are read by lb2_strip_tree's I/O workers into its
 * pinned slot ring (lb2_tree_prepare) and DMA'd into the window; the window buffers stay allocated with the
 * context and are reused by later calls.  A file shorter than its segment (or unreadable) gives
 * LB2_E_IO and out_path is removed. */
int lb2_gzip_segments(lb2_ctx *ctx, const lb2_gz_segment *segs, uint32_t n_segs, const char *out_path,
                      const void *gz_header, uint32_t gz_header_len, lb2_gzip_stats *stats);

#ifdef __cplusplus
}
#endif
#endif
