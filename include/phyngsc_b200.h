/*
 * phyngsc_b200.h -- C ABI of the B200-native phyNGSC subblock compressor.
 *
 * The reference (pcdslab/PHYNGSC) has no plugin / FFI seam: the path is the body of the
 * `while (p_bytes_read < p_working_region)` loop in main() (phyNGSC.cpp:168-840).  This header cuts
 * that seam.  Each entry point names the reference lines it replaces; INTEGRATION.md shows the
 * patch to phyNGSC.cpp a maintainer would apply.
 *
 * Plain pointers and sizes only; no C++ or torch types.  All compute runs in hand-written sm_100a
 * CUDA kernels; there is no CPU fallback -- every compute call fails with PHY_ERR_CUDA when no
 * device or no kernel image is usable.
 *
 * Threading: one phy_ctx per rank / GPU, calls on a ctx serialised by the caller.  The library
 * never calls MPI (the reference initialises MPI_THREAD_FUNNELED, phyNGSC.cpp:57).
 */
#ifndef PHYNGSC_B200_H
#define PHYNGSC_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PHY_ABI_VERSION 3 /* 3: phy_stream_prepare, emit callbacks come from a library thread */

enum {
  PHY_OK = 0,
  PHY_ERR_MALFORMED = -1,   /* line 3 is not "+", or quality length != sequence length (reference: UB)      */
  PHY_ERR_FIELDS = -2,      /* separator count differs between titles (reference: warning then UB, :417-421) */
  PHY_ERR_COLORSPACE = -3,  /* colour-space reads (phyNGSC.cpp:473-547) are not implemented                  */
  PHY_ERR_UNSUPPORTED = -4, /* outside the reference's defined domain: >32 title fields, token >512 B,
                               field max_len == 128 (Q11), Huffman code > 32 bits, NUL bytes; or beyond the
                               kernels' limits: a read of 512 bases or more (the per-position quality table
                               has 512 rows) fails its subblock, and so do 32 records of more than 24 KiB
                               whose packed quality tables exceed 24 KiB (e.g. 511 bp reads with more than
                               24 quality symbols)                                                            */
  PHY_ERR_CAPACITY = -5,    /* a ctx buffer (batch bytes, records, arena, output) is too small               */
  PHY_ERR_CUDA = -6,        /* CUDA runtime error / no device; see phy_last_error()                          */
  PHY_ERR_ARG = -7
};

typedef struct phy_ctx phy_ctx;

/* Region geometry, exactly the reference's (phyNGSC.cpp:113-124): region = file_size / np, rank r
 * owns [r*region, r*region + region + overlap - 1] (last rank: to EOF). */
typedef struct {
  uint64_t file_size;     /* FASTQ_size                                                     */
  int32_t np;             /* g_size (>= 1; the reference itself refuses np < 2, :91-97)     */
  int32_t rank;           /* p_rank                                                         */
  uint64_t window_bytes;  /* READ_BUFFER_SIZE, 8 MiB in the reference (defs.h:20)           */
  uint32_t overlap;       /* 500 (phyNGSC.cpp:48)                                           */
  uint32_t record_cap;    /* records a window can hold: 100000 (records_per_th x threads, phyNGSC.cpp:51,82,321) */
  uint32_t threads;       /* the reference's third CLI argument (0 is read as 1).  It only moves where the stop rule
                             of phyNGSC.cpp:315 starts to apply: threads before the last take every record whose title
                             ends in their slice of the window (:261-266, :303), so windows shorter than
                             threads x overlap keep more records than with one thread                         */
  uint32_t reserved;      /* 0 */
} phy_region_params;

/* One subblock as the reference's loop body produces it. */
typedef struct {
  uint64_t win_off;        /* window start relative to the region start (r_buffer_curr_pos - p_wr_start) */
  uint64_t win_len;        /* r_buffer_size used for this window                             */
  uint32_t rec_start;      /* rec_start_pos (non-zero only in the first window of rank > 0)  */
  int32_t overlap;         /* overlap in force (500 or 0, phyNGSC.cpp:123,751)               */
  uint32_t n_records;      /* no_records                                                     */
  uint32_t warnings;       /* bit0: record cap hit (phyNGSC.cpp:321-326)                     */
  uint64_t bytes_consumed; /* the increment of p_bytes_read (phyNGSC.cpp:745)                */
  uint32_t sec_len[4];     /* info, title, quality, dna stream lengths                       */
  uint64_t out_off;        /* offset of this payload in the output buffer (16-byte aligned)  */
  uint32_t out_len;        /* p_bytes_to_copy (phyNGSC.cpp:799)                              */
  int32_t status;          /* PHY_OK or the error raised for this subblock                   */
} phy_subblock_desc;

typedef struct {
  uint32_t n_subblocks;
  uint32_t n_batches;
  uint64_t bytes_in;         /* sum of bytes_consumed                                       */
  uint64_t bytes_out;        /* sum of out_len                                              */
  uint64_t out_used;         /* bytes of the output buffer used (payloads are 16-byte aligned) */
  int32_t wr_overlap;        /* wr_ov_used, for the footer (phyNGSC.cpp:160)                */
  uint32_t kernel_launches;  /* kernels launched by the call                                */
  float kernel_ms;           /* CUDA-event time of the kernel legs (first launch to last kernel done, per batch, summed) */
  float h2d_ms, d2h_ms;      /* CUDA-event time of the copies (0 if resident)               */
} phy_region_result;

/* Create a context on cuda_device.  max_batch_bytes bounds the region bytes resident per batch
 * (< 4 GiB: positions inside a batch are 32-bit); max_subblocks bounds the windows per batch.
 * 0 picks defaults (1 GiB + 16 MiB / 192). */
int phy_ctx_create(phy_ctx **out, int cuda_device, uint64_t max_batch_bytes, uint32_t max_subblocks);
int phy_device_count(void); /* CUDA devices visible to the process (0 when there is none) */
void phy_ctx_destroy(phy_ctx *ctx);

/* Replaces phyNGSC.cpp:168-840 for a whole working region: partition sync (:131-156), window chaining
 * (:744-755), record split, tokenise, analyse, Huffman, emit, section concat.
 *   region      host bytes starting at file offset rank*region (p_wr_start); region_len bytes are
 *               readable (at least up to p_wr_end + 1; more is fine and gives the read-slack
 *               semantics for records longer than `overlap`, SURVEY.md Q4)
 *   out         host buffer receiving the subblock payloads (info|title|quality|dna), payload i at
 *               out + descs[i].out_off
 *   descs       receives one descriptor per subblock, in order; *inout_n_descs = capacity in, count out
 * Host buffers may be pageable or pinned (phy_host_alloc; pinned makes the copies asynchronous). */
int phy_compress_region(phy_ctx *ctx, const uint8_t *region, uint64_t region_len, const phy_region_params *params,
                        uint8_t *out, uint64_t out_cap, phy_subblock_desc *descs, uint32_t *inout_n_descs,
                        phy_region_result *result);

/* Streamed variant for callers that are still filling `region` (a reader thread pulling the rank's byte range from
 * the file, phyNGSC.cpp:128/:249 done ahead of the GPU): before the library touches region[0, upto) it calls
 * wait(user, upto), which returns once those bytes are in place.  Batches are uploaded in order, so the file read of
 * batch b+1 overlaps the upload and the kernels of batch b.  Everything else is phy_compress_region. */
typedef void (*phy_wait_fn)(void *user, uint64_t upto);
int phy_compress_region_streamed(phy_ctx *ctx, const uint8_t *region, uint64_t region_len, const phy_region_params *params,
                                 phy_wait_fn wait, void *user, uint8_t *out, uint64_t out_cap, phy_subblock_desc *descs,
                                 uint32_t *inout_n_descs, phy_region_result *result);

/* The region is not in memory at all: the library pulls it through `read` (called from its own reader threads, in 16 MiB
 * pieces, straight into pinned staging memory -- no copy of the region is ever pinned or held by the caller) and hands
 * every batch of finished subblocks to `emit`, in order, from one library thread (never two emit calls at a time) while
 * later batches are still being read, uploaded and compressed.
 * Replaces the per-subblock MPI_File_read_at / compress / copy-to-write-buffer loop of phyNGSC.cpp:168-906 for one rank.
 *   read(user, off, dst, n)      fill dst with region bytes [off, off + n); return n, anything else is an error.
 *                                Must be thread-safe (pread is) and must not call MPI (MPI_THREAD_FUNNELED, phyNGSC.cpp:57).
 *   emit(user, descs, n, bytes)  n subblocks in order; payload i is bytes + descs[i].out_off (valid until emit returns);
 *                                a non-zero return stops the call with PHY_ERR_ARG. */
typedef int64_t (*phy_read_fn)(void *user, uint64_t off, void *dst, uint64_t n);
typedef int (*phy_emit_fn)(void *user, const phy_subblock_desc *descs, uint32_t n, const uint8_t *payloads);
int phy_compress_stream(phy_ctx *ctx, uint64_t region_len, const phy_region_params *params, phy_read_fn read, void *read_user,
                        phy_emit_fn emit, void *emit_user, phy_region_result *result);
/* Allocates what phy_compress_stream needs (pinned staging ring, pinned payload slots, second device buffers, copy streams)
 * ahead of the call, so that a driver can keep that one-off cost out of its timed region -- the analogue of MPI_Init
 * preceding p_timer_start in the reference (phyNGSC.cpp:57,111).  Optional: phy_compress_stream does it on first use. */
int phy_stream_prepare(phy_ctx *ctx);

/* The same work split into its three legs, for callers that keep data resident (and for kernel-only
 * timing): upload copies host bytes into the ctx input buffer; compress_resident runs the kernels over
 * what is resident (single batch: region_len <= max_batch_bytes) leaving payloads in device memory
 * (descs[i].out_off is then an offset into the device output buffer); download copies them out. */
int phy_upload(phy_ctx *ctx, const uint8_t *region, uint64_t region_len);
int phy_compress_resident(phy_ctx *ctx, uint64_t region_len, const phy_region_params *params,
                          phy_subblock_desc *descs, uint32_t *inout_n_descs, phy_region_result *result);
int phy_download(phy_ctx *ctx, uint8_t *out, uint64_t out_cap, uint64_t *out_len);

/* First record of a rank > 0 region: the '@' ... '\n' heuristic of phyNGSC.cpp:131-156.  Returns the
 * offset inside `region`, or a negative error. */
int64_t phy_find_first_record(const uint8_t *region, uint64_t region_len);

/* Raw device pointers of the ctx buffers (for zero-copy producers) and pinned host memory. */
void *phy_device_input(phy_ctx *ctx, uint64_t *capacity);
void *phy_device_output(phy_ctx *ctx, uint64_t *capacity);
void *phy_host_alloc(uint64_t bytes);
void phy_host_free(void *p);

/* Block header exactly as MakeHeader writes it (tasks.cpp:1179-1200); returns bytes written or 0. */
uint32_t phy_make_block_header(int32_t wrid, int32_t bewr, int32_t bhs, int32_t beso, int32_t bcss,
                               const uint32_t *sbol, uint32_t nosb, uint8_t *out, uint32_t cap);
/* Footer exactly as MakeFooter writes it (tasks.cpp:1104-1176) for the given block order. */
int32_t phy_make_footer(int32_t np, uint64_t fastq_size, uint32_t n_blocks, uint32_t n_subblocks,
                        const int32_t *overlaps, const int32_t *block_order, const uint32_t *lb_sizes,
                        uint8_t *out, uint32_t cap);

/* Stage dumps for the parity tests: copies `bytes` bytes at byte offset `offset` of a named device
 * buffer of the last batch ("te", "se", "rstart", "kx", "qoff", "doff", "plans", "acc", "cls", "arena",
 * "hdr", "sbout") to dst.  Returns bytes copied or a negative error. */
int64_t phy_debug_read(phy_ctx *ctx, const char *name, uint64_t offset, void *dst, uint64_t bytes);

/* Per-stage timing for bench.py: with profiling enabled every batch records one CUDA event after each
 * kernel launch (and synchronises at the end of the batch); phy_profile_read returns the stage names and
 * their mean duration in ms per batch since profiling was enabled.  Returns the number of stages. */
int phy_profile(phy_ctx *ctx, int enable);
int phy_profile_read(phy_ctx *ctx, const char **names, float *ms, int cap);

/* Decoder of one subblock payload (info | title | quality | dna) back to FASTQ text: the inverse of the path above
 * (host code, phyngsc_b200/host/phy_decode.hpp; replaces the Fetch* chain of tasks.cpp:625-1101, whose driver
 * phyNGSD.cpp the reference does not ship).  Needs no device and no context; reentrant.  Returns the number of bytes
 * written to `out`, PHY_ERR_CAPACITY if `cap` is too small, PHY_ERR_MALFORMED for a payload that is not a subblock. */
int64_t phy_decode_subblock(const uint8_t *payload, uint64_t len, uint8_t *out, uint64_t cap);

const char *phy_strerror(int code);
const char *phy_last_error(phy_ctx *ctx); /* detail of the last failure on ctx (may be "") */
int phy_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif
