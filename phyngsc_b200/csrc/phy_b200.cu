/*
 * phy_b200.cu -- context, batch scheduling and the C ABI (include/phyngsc_b200.h) of the B200-native
 * phyNGSC subblock compressor.  Kernels live in phy_kernels.cuh, format logic in phy_core.cuh.
 * There is no CPU path: every compute entry point needs a CUDA device.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/phyngsc_b200.h"
#include "phy_kernels.cuh"
#include "phy_encode.cuh"
#include "phy_seqstat.cuh"
#include "phy_title.cuh"

using namespace phy;

#define NKERN 20
#define GROUPS_MAX 8

static_assert(sizeof(phy_subblock_desc) == 72, "phy_subblock_desc layout is part of the ABI");
static_assert(sizeof(phy_region_params) == 40, "phy_region_params layout is part of the ABI");

/* Owning handles of a context's CUDA resources.  Each is complete or empty, never half made, and its destructor releases
 * it: phy_ctx_destroy (and a failed ctx_init) only has to delete the context. */
template <class T, bool Pinned> struct Buf { /* `cap` bytes of device memory, or of pinned host memory */
  T *p = nullptr;
  u64 cap = 0;
  Buf() = default;
  Buf(const Buf &) = delete;
  Buf &operator=(const Buf &) = delete;
  ~Buf() { release(); }
  operator T *() const { return p; }
  T *operator->() const { return p; }
  void swap(Buf &o) { std::swap(p, o.p); std::swap(cap, o.cap); }
  void release() {
    if (p) { if (Pinned) cudaFreeHost(p); else cudaFree(p); }
    p = nullptr; cap = 0;
  }
  /* At least `bytes`.  Growing frees the old buffer first (never two at a time) and leaves the buffer empty if it fails;
   * `zero` clears a new buffer. */
  cudaError_t ensure(u64 bytes, bool zero = false) {
    if (cap >= bytes) return cudaSuccess;
    release();
    void *q = nullptr;
    cudaError_t e = Pinned ? cudaHostAlloc(&q, bytes, cudaHostAllocDefault) : cudaMalloc(&q, bytes);
    if (e != cudaSuccess) return e;
    p = (T *)q; cap = bytes;
    if (zero && (e = cudaMemset(p, 0, bytes)) != cudaSuccess) release();
    return e;
  }
};
template <class T> using DevBuf = Buf<T, false>;
template <class T> using PinBuf = Buf<T, true>;

static cudaError_t create(cudaStream_t *s, int priority) { return cudaStreamCreateWithPriority(s, cudaStreamNonBlocking, priority); }
static cudaError_t create(cudaEvent_t *e, unsigned flags) { return cudaEventCreateWithFlags(e, flags); }
static void destroy(cudaStream_t s) { cudaStreamDestroy(s); }
static void destroy(cudaEvent_t e) { cudaEventDestroy(e); }
template <class H, class Arg> struct Handle { /* a stream (ensure(priority)) or an event (ensure(flags)) */
  H h = nullptr;
  Handle() = default;
  Handle(const Handle &) = delete;
  Handle &operator=(const Handle &) = delete;
  ~Handle() { if (h) destroy(h); }
  operator H() const { return h; }
  cudaError_t ensure(Arg a) {
    if (h) return cudaSuccess;
    H x = nullptr;
    cudaError_t e = create(&x, a);
    if (e == cudaSuccess) h = x;
    return e;
  }
};
using Stream = Handle<cudaStream_t, int>;
using Event = Handle<cudaEvent_t, unsigned>;

/* pinned staging of phy_compress_stream */
static const u64 RING_CHUNK = 16ull << 20;
static const int RING_SLOTS = 8;
static const int HOUT_SLOTS = 4; /* pinned payload slots: one being filled by the copy engine, the others with the emitter thread */
static const int READERS = 6;    /* reader threads */

struct phy_ctx {
  int device = 0;
  int prio_hi = 0; /* the back part's streams outrank the front part's: a front part running ahead only fills gaps */
  u64 max_batch = 0; u32 max_sb = 0; u32 maxrec = 0; u32 arena_words = 0; u64 out_cap = 0; u32 slack = 0;
  u32 max_tiles = 0;
  Stream stream, s_prefix;
  Event ev_prefix;    /* the front part launched last is done */
  Event ev_k0, ev_k1; /* begin and end of a walk's kernel leg (phy_region_result::kernel_ms) */
  /* subblock groups of a batch: own stream, header (device + pinned mirror) and events */
  Stream gstream[GROUPS_MAX]; Event ev_rb[GROUPS_MAX], ev_scan[GROUPS_MAX], ev_done[GROUPS_MAX];
  DevBuf<BatchHdr> hdr_g; PinBuf<BatchHdr> h_hdr_g;
  /* device buffers */
  DevBuf<u8> in; DevBuf<u32> te, se, rstart; DevBuf<u16> kx; DevBuf<u32> qoff, doff, toff, chunk_first, chunk_last;
  DevBuf<u32> tile_cnt, tile_off; DevBuf<uint2> nl_mask;
  DevBuf<u32> blk_mask, tv, tc, tp, v0; /* parsed titles (k_stat1 -> k_stat2 / k_enc_title); tv / tp / tc grow on demand */
  DevBuf<PlanState> plan_state; DevBuf<SbPlan> plans; DevBuf<BatchHdr> hdr;
  DevBuf<SbAcc> acc; DevBuf<SbClass> cls; DevBuf<SbOut> sbout; DevBuf<u32> arena; DevBuf<u8> out;
  DevBuf<u32> tmp; DevBuf<u64> tmp_used; /* temporary buffer of the single-walk encoder (words) */
  /* second input / output buffers and copy streams of the pipelined region call (allocated on first use) */
  DevBuf<u8> in2, out2;
  Stream s_in, s_out;
  Event ev_in[2], ev_c[2], ev_out[2], ev_h0[2], ev_d0[2];
  /* pinned host mirrors */
  PinBuf<BatchHdr> h_hdr; PinBuf<SbPlan> h_plans; PinBuf<SbOut> h_sbout; PinBuf<PlanState> h_state;
  /* Front part of a batch (record splitter + window plan) ahead of its back part: the front part writes the "next" set of its
   * outputs (record table, window plans, header, host mirrors); prefix_finish() swaps that set with the current one, which the
   * back part (every other kernel) reads.  So the front part of batch b + 1 can run beside the back part of batch b. */
  struct PrefixSet { DevBuf<u32> te, se, rstart; DevBuf<SbPlan> plans; DevBuf<BatchHdr> hdr;
                     PinBuf<BatchHdr> h_hdr; PinBuf<SbPlan> h_plans; PinBuf<PlanState> h_state; } nxt;
  struct BatchArgs { const u8 *in = nullptr; u32 len = 0, start_pos = 0; i64 batch_base = 0, region_len = 0; bool is_final = false; } cur_args, nxt_args;
  int pi = 0; /* next profiling event of the batch */
  u32 launches = 0;
  u64 resident_len = 0, resident_out = 0;
  PinBuf<u8> ring, hout[HOUT_SLOTS]; Event ev_ring[RING_SLOTS], ev_hout[HOUT_SLOTS]; /* pinned staging of phy_compress_stream */
  DevBuf<u8> big_in, big_out; /* resident regions larger than one batch (phy_upload) */
  u32 last_S = 0;
  u32 qcode_hint = 0; /* longest quality code the previous batch saw */
  u32 nq_hint = 0, prev_groups = 0, prev_max_len = 0; /* quality alphabet size seen by the previous batch (sizes the packed tables' shared memory without a readback) */
  /* per-kernel timing (phy_profile): one event after every launch of run_batch */
  bool profile = false;
  Event pev[NKERN + 1];
  float pms[NKERN] = {};
  u32 pcount = 0;
  std::string err;
};

#define CK(call)                                                                                       \
  do {                                                                                                 \
    cudaError_t e_ = (call);                                                                           \
    if (e_ != cudaSuccess) {                                                                           \
      char buf_[512];                                                                                  \
      snprintf(buf_, sizeof buf_, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));  \
      ctx->err = buf_;                                                                                 \
      return PHY_ERR_CUDA;                                                                             \
    }                                                                                                  \
  } while (0)

static const u32 SPAN_MAX = 96 * 1024;
static const u32 ENC_STAGE_MAX = 24 * 1024; /* a warp's stage in the encoder kernels: 32 records of up to 768 bytes on average */
static const u32 ENC_DYN_MAX = 200 * 1024;  /* dynamic shared memory of the single-walk encoder kernels */
static const u32 PK_SMEM_MAX = 24 * 1024; /* packed quality code tables kept in shared memory by k_lengths / k_emit */

static const char *KERNEL_NAMES[NKERN] = {"nl_count", "nl_scan", "nl_emit", "plan", "plan_readback", "stat1", "seqstat", "classify", "zero_hist",
                                          "stat2", "huff", "slots", "enc_title", "enc_qd", "lengths", "layout", "outscan", "zero_out", "place", "emit"};

extern "C" int phy_abi_version(void) { return PHY_ABI_VERSION; }

extern "C" int phy_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

extern "C" const char *phy_strerror(int code) {
  switch (code) {
    case PHY_OK: return "ok";
    case PHY_ERR_MALFORMED: return "malformed FASTQ record";
    case PHY_ERR_FIELDS: return "title field count differs between records";
    case PHY_ERR_COLORSPACE: return "colour-space reads are not implemented";
    case PHY_ERR_UNSUPPORTED: return "input outside the reference's defined domain";
    case PHY_ERR_CAPACITY: return "context buffer too small";
    case PHY_ERR_CUDA: return "CUDA error";
    case PHY_ERR_ARG: return "bad argument";
  }
  return "unknown error";
}

extern "C" const char *phy_last_error(phy_ctx *ctx) { return ctx ? ctx->err.c_str() : ""; }

extern "C" void *phy_host_alloc(uint64_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
extern "C" void phy_host_free(void *p) { if (p) cudaFreeHost(p); }

extern "C" void phy_ctx_destroy(phy_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device); /* the handles release their resources on the context's device */
  delete ctx;
}

static int ctx_init(phy_ctx *ctx, int device, u64 max_batch, u32 max_sb) {
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) { ctx->err = "no such CUDA device"; return PHY_ERR_CUDA; }
  CK(cudaSetDevice(device));
  ctx->device = device;
  ctx->max_batch = max_batch ? max_batch : ((1ull << 30) + (16ull << 20));
  if (ctx->max_batch >= (1ull << 32) - (1u << 20)) { ctx->err = "max_batch_bytes must be < 4 GiB"; return PHY_ERR_ARG; }
  ctx->max_sb = max_sb ? max_sb : 192;
  ctx->maxrec = (u32)(ctx->max_batch / 32) + 1024;
  ctx->arena_words = (2u << 20) / 4 + RAW_WORDS; /* coding scratch + the raw quality table */
  ctx->out_cap = ctx->max_batch / 2 + (1u << 20);
  ctx->slack = 64 * 1024;
  ctx->max_tiles = (u32)((ctx->max_batch + TILE - 1) / TILE) + 1;
  int prio_lo = 0;
  CK(cudaDeviceGetStreamPriorityRange(&prio_lo, &ctx->prio_hi));
  CK(ctx->stream.ensure(ctx->prio_hi));
  CK(ctx->s_prefix.ensure(prio_lo));
  CK(ctx->ev_prefix.ensure(cudaEventDisableTiming));
  CK(ctx->hdr_g.ensure(sizeof(BatchHdr) * GROUPS_MAX));
  CK(ctx->h_hdr_g.ensure(sizeof(BatchHdr) * GROUPS_MAX));
  CK(ctx->ev_rb[0].ensure(cudaEventDisableTiming));
  CK(ctx->ev_k0.ensure(cudaEventDefault));
  CK(ctx->ev_k1.ensure(cudaEventDefault));
  CK(ctx->in.ensure(ctx->max_batch + 4096, true));
  const size_t rec4 = (size_t)(ctx->maxrec + 4) * 4;
  for (DevBuf<u32> *b : {&ctx->te, &ctx->se, &ctx->rstart, &ctx->nxt.te, &ctx->nxt.se, &ctx->nxt.rstart, &ctx->qoff, &ctx->doff, &ctx->toff})
    CK(b->ensure(rec4));
  CK(ctx->kx.ensure((size_t)(ctx->maxrec + 4) * 2));
  {
    size_t rows = (size_t)ctx->maxrec / CH + ctx->max_sb + 2; /* every subblock rounds its chunk count up */
    CK(ctx->chunk_first.ensure(rows * MAXF * 4));
    CK(ctx->chunk_last.ensure(rows * MAXF * 4));
    CK(ctx->blk_mask.ensure(rows * (CH / 32) * 4));
    CK(ctx->v0.ensure((size_t)ctx->max_sb * MAXF * 4));
  }
  CK(ctx->tile_cnt.ensure((size_t)ctx->max_tiles * 4));
  CK(ctx->tile_off.ensure((size_t)ctx->max_tiles * 4));
  CK(ctx->nl_mask.ensure((size_t)ctx->max_tiles * NLT * sizeof(uint2)));
  CK(ctx->plan_state.ensure(sizeof(PlanState)));
  CK(ctx->plans.ensure(sizeof(SbPlan) * ctx->max_sb));
  CK(ctx->hdr.ensure(sizeof(BatchHdr)));
  CK(ctx->nxt.plans.ensure(sizeof(SbPlan) * ctx->max_sb));
  CK(ctx->nxt.hdr.ensure(sizeof(BatchHdr)));
  CK(ctx->acc.ensure(sizeof(SbAcc) * ctx->max_sb));
  CK(ctx->cls.ensure(sizeof(SbClass) * ctx->max_sb));
  CK(ctx->sbout.ensure(sizeof(SbOut) * ctx->max_sb));
  CK(ctx->arena.ensure((size_t)ctx->arena_words * 4 * ctx->max_sb));
  CK(ctx->out.ensure(ctx->out_cap + 64));
  CK(ctx->tmp.ensure(((ctx->max_batch + ctx->max_batch / 2) / 4 + (1u << 20)) * 4)); /* 1.5 bytes per input byte: slots are sized by bounds, not by what is written */
  CK(ctx->tmp_used.ensure(sizeof(u64)));
  CK(ctx->h_hdr.ensure(sizeof(BatchHdr)));
  CK(ctx->h_plans.ensure(sizeof(SbPlan) * ctx->max_sb));
  CK(ctx->h_sbout.ensure(sizeof(SbOut) * ctx->max_sb));
  CK(ctx->h_state.ensure(sizeof(PlanState)));
  CK(ctx->nxt.h_hdr.ensure(sizeof(BatchHdr)));
  CK(ctx->nxt.h_plans.ensure(sizeof(SbPlan) * ctx->max_sb));
  CK(ctx->nxt.h_state.ensure(sizeof(PlanState)));
  {
    u8 lut[256];
    fill_char_lut(lut);
    CK(cudaMemcpyToSymbol(g_char_lut, lut, sizeof lut));
    for (u32 c = 0; c < 256; ++c) { u32 a = amb_code((u8)c); lut[c] = a > 1 ? (u8)(79u + 8u * a) : (u8)0; }
    CK(cudaMemcpyToSymbol(g_xq_lut, lut, sizeof lut));
  }
  CK(cudaFuncSetAttribute(k_stat1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_dnacount, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SPAN_MAX));
  CK(cudaFuncSetAttribute(k_seqstat<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_seqstat<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_seqstat<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_seqstat<8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_seqstat<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_seqstat<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_seqstat<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_seqstat<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_lengths<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(EW * ENC_STAGE_MAX + PK_SMEM_MAX)));
  CK(cudaFuncSetAttribute(k_lengths<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(EP * ENC_STAGE_MAX + PK_SMEM_MAX)));
  CK(cudaFuncSetAttribute(k_emit<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(EW * ENC_STAGE_MAX + PK_SMEM_MAX)));
  CK(cudaFuncSetAttribute(k_emit<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(EP * ENC_STAGE_MAX + PK_SMEM_MAX)));
  CK(cudaFuncSetAttribute(k_huff, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HUFF_SMEM));
  CK(cudaFuncSetAttribute(k_enc_title, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_enc_qd<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_enc_qd<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_enc_qd<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  CK(cudaFuncSetAttribute(k_enc_qd<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENC_DYN_MAX));
  return PHY_OK;
}

extern "C" int phy_ctx_create(phy_ctx **out, int cuda_device, uint64_t max_batch_bytes, uint32_t max_subblocks) {
  if (!out) return PHY_ERR_ARG;
  phy_ctx *ctx = new phy_ctx();
  int rc = ctx_init(ctx, cuda_device, max_batch_bytes, max_subblocks);
  if (rc) { fprintf(stderr, "phyngsc_b200: %s\n", ctx->err.c_str()); phy_ctx_destroy(ctx); *out = nullptr; return rc; }
  *out = ctx;
  return PHY_OK;
}

extern "C" void *phy_device_input(phy_ctx *ctx, uint64_t *capacity) { if (capacity) *capacity = ctx->max_batch; return ctx->in; }
extern "C" void *phy_device_output(phy_ctx *ctx, uint64_t *capacity) { if (capacity) *capacity = ctx->out_cap; return ctx->out; }

/* phyNGSC.cpp:131-156 */
extern "C" int64_t phy_find_first_record(const uint8_t *b, uint64_t lim) {
  uint64_t c = 0;
  while (c < lim && b[c] != '@') ++c;
  uint64_t first_at = c;
  while (c < lim && b[c] != '\n') ++c;
  if (c + 1 >= lim) return PHY_ERR_MALFORMED;
  return (int64_t)((b[c + 1] == '@') ? c + 1 : first_at);
}

/* Switches of the environment, read once per process:
 *   PHY_GROUPS      subblock groups of a batch (1..GROUPS_MAX, default 3; the profiling scripts set 1)
 *   PHY_ENC=0       every subblock through the two-walk encoder (k_lengths + k_emit) instead of the single-walk kernels
 *   PHY_DEBUG_SYNC  fault isolation: synchronise after every launch (also runs one group and no front part ahead) */
static int env_int(const char *name, int dflt) { const char *v = getenv(name); return v ? atoi(v) : dflt; }
static const struct {
  int groups = env_int("PHY_GROUPS", 3); /* measured on 1 GB: 3.25 / 3.13 / 3.01 / 3.05 ms for 1..4 groups */
  bool enc = env_int("PHY_ENC", 1) != 0;
  bool debug_sync = getenv("PHY_DEBUG_SYNC") != nullptr;
} sw;

#define PMARK()                                                                                                   \
  do {                                                                                                            \
    if (ctx->profile) cudaEventRecord(ctx->pev[ctx->pi], st);                                                     \
    if (sw.debug_sync) {                                                                                          \
      cudaError_t e_ = cudaStreamSynchronize(st);                                                                 \
      if (e_ == cudaSuccess) e_ = cudaGetLastError();                                                             \
      if (e_ != cudaSuccess) {                                                                                    \
        ctx->err = std::string("after stage ") + (ctx->pi ? KERNEL_NAMES[ctx->pi - 1] : "start") + ": " + cudaGetErrorString(e_); \
        return PHY_ERR_CUDA;                                                                                      \
      }                                                                                                           \
    }                                                                                                             \
    ++ctx->pi;                                                                                                    \
  } while (0)

/* Where the batch walk over a region stands; every entry point walks a region by these rules.  A batch is the region's
 * bytes [base, base + blen); its window chain starts at next_pos. */
struct Walk {
  PlanState st;           /* the reference's plan state at the region's start (walk_init) */
  u64 len = 0;            /* region bytes */
  u64 max_batch = 0;
  u64 back = 0;           /* how far before a batch's end the next one starts: a window that does not fit the rest of a batch
                           * (with the slack for records longer than the overlap) is left to the next batch */
  u64 base = 0, blen = 0;
  bool final = false;     /* the batch ends at the region's end */
  bool nl = false;        /* last rank whose file does not end in a newline: the reference's arithmetic still places the next
                           * record start one byte past the end; a virtual newline behind the final batch gives the splitter
                           * the same view (written by a one-byte memset behind the region's bytes on the device) */
  u64 next_pos = 0;       /* PlanState::bytes_read at the start of the batch */
  u32 nb = 0;             /* batches finished */

  u64 len_at(u64 b) const { return len - b < max_batch ? len - b : max_batch; }
  void place(u64 b) { base = b; blen = len_at(b); final = b + blen == len; }
  /* start of the batch after a non-final one */
  u64 candidate() const { return (base + blen - back) & ~(u64)255; }
  u32 kernel_len() const { return (u32)(blen + (final && nl ? 1 : 0)); }
  u32 start_pos() const { return (u32)(next_pos - base) + (nb == 0 ? st.rec_start : 0u); }
  /* After a batch whose front part made S windows and left the chain at hs: `done` once the working region is covered,
   * else `move` says whether the next round runs the candidate batch or -- the chain stopped early because the batch's
   * subblock capacity was used up -- the same bytes again.  A chain that made no progress is an error. */
  int after(phy_ctx *ctx, const PlanState &hs, u32 S, bool &done, bool &move) {
    ++nb;
    move = false;
    if (hs.status) { ctx->err = std::string("window chaining failed: ") + phy_strerror(hs.status); return hs.status; }
    done = hs.done != 0;
    if (done) return PHY_OK;
    const u64 stopped = (u64)hs.bytes_read;
    if (S == 0 && stopped == next_pos && (final || stopped < candidate())) {
      ctx->err = final ? "region exhausted before the working region was covered" : "a window does not fit one batch (raise max_batch_bytes)";
      return final ? PHY_ERR_MALFORMED : PHY_ERR_CAPACITY;
    }
    next_pos = stopped;
    move = !final && next_pos >= candidate();
    return PHY_OK;
  }
};

/* Front part of the walk's batch on stream `st` (`in`: the batch's first byte on the device): record splitter, window chain,
 * sizes; its results go to the "next" set and are copied to that set's host mirrors.  Does not wait. */
static int prefix_launch(phy_ctx *ctx, cudaStream_t st, const u8 *in, const Walk &w) {
  const u32 len = w.kernel_len();
  Dev d;
  memset(&d, 0, sizeof d);
  d.in = in; d.len = len; d.start_pos = w.start_pos();
  d.te = ctx->nxt.te; d.se = ctx->nxt.se; d.rstart = ctx->nxt.rstart; d.maxrec = ctx->maxrec;
  d.tile_cnt = ctx->tile_cnt; d.tile_off = ctx->tile_off; d.nl_mask = ctx->nl_mask; d.ntiles = (len + TILE - 1) / TILE;
  d.plan_state = ctx->plan_state; d.plans = ctx->nxt.plans; d.max_sb = ctx->max_sb; d.hdr = ctx->nxt.hdr;
  d.batch_base = (i64)w.base; d.region_len = (i64)w.len; d.batch_is_final = w.final ? 1 : 0; d.slack = ctx->slack;
  ctx->nxt_args.in = in; ctx->nxt_args.len = len; ctx->nxt_args.start_pos = d.start_pos; ctx->nxt_args.batch_base = d.batch_base;
  ctx->nxt_args.region_len = d.region_len; ctx->nxt_args.is_final = w.final;
  if (d.ntiles == 0) { ctx->err = "empty batch"; return PHY_ERR_ARG; }
  ctx->pi = 0;
  PMARK();
  CK(cudaMemsetAsync(ctx->tile_off, 0, (size_t)((d.ntiles + SUPER - 1) / SUPER) * 4, st));
  k_nl_count<<<d.ntiles, NLT, 0, st>>>(d); PMARK();
  k_nl_scan<<<1, 1024, 0, st>>>(d); PMARK();
  k_nl_emit<<<d.ntiles, NLT, 0, st>>>(d); PMARK();
  k_plan<<<1, 32, 0, st>>>(d);
  k_spanmax<<<dim3(8, ctx->max_sb), 256, 0, st>>>(d); PMARK();
  ctx->launches += 5;
  CK(cudaMemcpyAsync(ctx->nxt.h_hdr, ctx->nxt.hdr, sizeof(BatchHdr), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(ctx->nxt.h_state, ctx->plan_state, sizeof(PlanState), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(ctx->nxt.h_plans, ctx->nxt.plans, sizeof(SbPlan) * ctx->max_sb, cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(ctx->ev_prefix, st));
  return PHY_OK;
}

/* Waits for the front part launched last and makes its results the current set: h_hdr / h_state / h_plans describe the batch. */
static int prefix_finish(phy_ctx *ctx) {
  CK(cudaEventSynchronize(ctx->ev_prefix));
  ctx->te.swap(ctx->nxt.te); ctx->se.swap(ctx->nxt.se); ctx->rstart.swap(ctx->nxt.rstart);
  ctx->plans.swap(ctx->nxt.plans); ctx->hdr.swap(ctx->nxt.hdr);
  ctx->h_hdr.swap(ctx->nxt.h_hdr); ctx->h_plans.swap(ctx->nxt.h_plans); ctx->h_state.swap(ctx->nxt.h_state);
  ctx->cur_args = ctx->nxt_args;
  ctx->last_S = 0;
  const BatchHdr &H = *ctx->h_hdr;
  if (H.status) { ctx->err = std::string("batch failed while splitting records: ") + phy_strerror(H.status); return H.status; }
  ctx->last_S = H.S;
  return PHY_OK;
}

/* Back part of the current batch (everything after the window plan) on the context's main stream and its group streams.
 * On return (after the caller has synchronised the main stream) h_sbout and h_hdr->total_out describe the payloads. */
static int run_body(phy_ctx *ctx, u8 *out, u64 out_cap) {
  const phy_ctx::BatchArgs &A = ctx->cur_args;
  Dev d;
  memset(&d, 0, sizeof d);
  d.in = A.in; d.len = A.len; d.start_pos = A.start_pos;
  d.te = ctx->te; d.se = ctx->se; d.rstart = ctx->rstart; d.maxrec = ctx->maxrec;
  d.kx = ctx->kx; d.qoff = ctx->qoff; d.doff = ctx->doff; d.toff = ctx->toff; d.chunk_first = ctx->chunk_first; d.chunk_last = ctx->chunk_last;
  d.blk_mask = ctx->blk_mask; d.v0 = ctx->v0;
  d.tile_cnt = ctx->tile_cnt; d.tile_off = ctx->tile_off; d.nl_mask = ctx->nl_mask; d.ntiles = (A.len + TILE - 1) / TILE;
  d.plan_state = ctx->plan_state; d.plans = ctx->plans; d.max_sb = ctx->max_sb; d.hdr = ctx->hdr;
  d.acc = ctx->acc; d.cls = ctx->cls; d.sbout = ctx->sbout; d.arena = ctx->arena; d.arena_words = ctx->arena_words;
  d.out = out; d.out_cap = out_cap;
  d.batch_base = A.batch_base; d.region_len = A.region_len; d.batch_is_final = A.is_final ? 1 : 0; d.slack = ctx->slack;
  d.span_bytes = 0;
  d.tmp = ctx->tmp; d.tmp_cap = ctx->tmp.cap / 4; d.tmp_used = ctx->tmp_used;
  cudaStream_t st = ctx->stream;
  if (ctx->prev_groups) { /* the previous batch is complete (the callers synchronise): its alphabet is the hint for this one */
    u32 mx = 0, mq = 0;
    for (u32 g = 0; g < ctx->prev_groups; ++g) { mx = ctx->h_hdr_g[g].max_pk_bytes > mx ? ctx->h_hdr_g[g].max_pk_bytes : mx; mq = ctx->h_hdr_g[g].max_qcode > mq ? ctx->h_hdr_g[g].max_qcode : mq; }
    ctx->qcode_hint = mq;
    if (ctx->prev_max_len) ctx->nq_hint = mx / 2 / (ctx->prev_max_len + 1);
    ctx->prev_groups = 0;
  }
  CK(cudaMemsetAsync(ctx->tmp_used, 0, sizeof(u64), st));
  const BatchHdr H = *ctx->h_hdr;
  const u32 S = H.S;
  if (S == 0) return PHY_OK;
  u32 span = (H.max_span + 16 + 1023) & ~1023u; /* exact: every 128-record span of the batch fits (k_spanmax) */
  if (span > SPAN_MAX) span = SPAN_MAX;         /* longer spans fail their subblock with PHY_ERR_UNSUPPORTED */
  d.span_bytes = span;
  d.max_nf = H.max_nf < (u32)MAXF ? H.max_nf : (u32)MAXF;
  { /* parsed-title rows: one row of 32 entries per (block, field) in each of tv and tp; grown when a batch needs more */
    const SbPlan &PL = ctx->h_plans[S - 1];
    const u64 chunks = (u64)PL.chunk_base + (PL.n_records + CH - 1) / CH;
    d.nfs = d.max_nf ? d.max_nf : 1u;
    const u64 need = chunks * d.nfs * CH;
    for (DevBuf<u32> *b : {&ctx->tv, &ctx->tp, &ctx->tc})
      if (b->cap < need * 4) CK(b->ensure((need + need / 4) * 4));
    d.tv = ctx->tv; d.tp = ctx->tp; d.tc = ctx->tc;
  }
  /* launch geometry shared by all subblock groups of the batch */
  {
    u32 es = (H.max_span32 + 16 + 255) & ~255u;
    d.enc_stage = es > ENC_STAGE_MAX ? ENC_STAGE_MAX : es; /* wider blocks fail their subblock with PHY_ERR_UNSUPPORTED */
  }
  /* Single-walk encoder (phy_encode.cuh): G lanes share a record's quality / DNA codes so that a lane's run of read
   * positions stays short (its staging words and the records a warp keeps staged shrink with G); PHY_ENC=0 switches
   * the single-walk kernels off (every subblock then takes k_lengths + k_emit). */
  u32 encG = H.max_len <= 64 ? 1u : H.max_len <= 256 ? 4u : 8u; /* measured per shape (36 / 100 / 150 / 50-205 bp): 1, 4, 4, 4 */
  while (encG < 8 && seg_len(H.max_len, encG) > 64) encG *= 2; /* a lane keeps one bit per position of its run (k_seqstat) */
  d.fg.g = sw.enc ? encG : 0u;
  /* lane-private staging: a lane's run of positions times the longest quality code -- 12 bits unless the previous batch
   * of this context saw longer ones (subblocks that need more than the kernels were launched with take the two-walk path) */
  d.fg.lpw_q = (seg_len(H.max_len, encG) * (ctx->qcode_hint > 12 ? (ctx->qcode_hint > 24 ? 24u : ctx->qcode_hint) : 12u) + 31u) / 32u + 2u;
  d.fg.pk_bytes = 0;
  d.qd_stage = ((32u / encG) * H.max_rec + 32u + 255u) & ~255u;
  if (encG == 1) d.qd_stage = (H.max_span32 + 16 + 255) & ~255u;
  d.qd_nbuf = encG > 1 && d.qd_stage <= 2560 ? 2u : 1u; /* measured: a second stage only pays while it is small (100 bp: 0.86 vs 0.90 ms per GB, 150 bp: 0.89 vs 0.78) */
  d.ts = (((H.max_tlen + 16u + 15u) & ~15u) | 16u);
  const u32 max_tasks = (H.max_chunks * CH + TASK_RECORDS - 1) / TASK_RECORDS;
  /* statistics: k_seqstat uses the lane split and the record stages of k_enc_qd, k_stat1 / k_stat2 stage title lines only */
  d.sq_rows = H.max_len < 1 ? 1u : H.max_len > RAW_ROWS - 1 ? RAW_ROWS - 1 : H.max_len;
  d.sq_stage = d.qd_stage; d.sq_nbuf = 1; /* one stage: more resident CTAs hide the copy better (100 bp: 0.66 vs 0.76 ms per GB) */
  const bool sq_wide = d.sq_rows <= 126; /* 32-bit counters while the private table stays below 48 KB, else 16-bit pairs */
  const u32 sq_dyn = ((d.sq_rows * (sq_wide ? 97u : SQ_ROWW) * 4u + 15u) & ~15u) + SQ_WARPS * d.sq_nbuf * d.sq_stage;
  /* k_stat1: two stages of one title slot per lane for every warp; fewer warps per CTA when the title lines are long */
  u32 s1_warps = S1W;
  while (s1_warps > 1 && s1_warps * 2u * 32u * d.ts > ENC_DYN_MAX) s1_warps /= 2;
  const u32 title_stat_dyn = s1_warps * 2u * 32u * d.ts;
  if (sq_dyn > ENC_DYN_MAX || title_stat_dyn > ENC_DYN_MAX) { ctx->err = "records too long for the statistics kernels' shared memory"; return PHY_ERR_UNSUPPORTED; }
  /* Subblock groups: the subblocks of the batch are split into G consecutive groups that run the rest of the pipeline on
   * their own streams.  Several of its stages are latency-bound (one warp per subblock in k_classify, one warp per table
   * in k_huff, one CTA per subblock in k_layout): while one group sits in such a stage the other keeps the SMs busy.
   * A group sees its own slice of the per-subblock arrays (shifted base pointers) and its own header; the payloads of all
   * groups still lie back to back because a group's output scan starts at the previous group's end. */
  const u32 G = (ctx->profile || sw.debug_sync || S < 16) ? 1u : (u32)(sw.groups < 1 ? 1 : sw.groups > GROUPS_MAX ? GROUPS_MAX : sw.groups);
  if (G > 1)
    for (u32 g = 0; g < G; ++g) {
      if (g) CK(ctx->gstream[g].ensure(ctx->prio_hi));
      for (Event *e : {&ctx->ev_rb[g], &ctx->ev_scan[g], &ctx->ev_done[g]}) CK(e->ensure(cudaEventDisableTiming));
    }
  Dev dg[GROUPS_MAX];
  u32 s0[GROUPS_MAX + 1];
  for (u32 g = 0; g <= G; ++g) s0[g] = (u32)((u64)S * g / G);
  for (u32 g = 0; g < G; ++g) {
    Dev &e = dg[g];
    e = d;
    const u32 b = s0[g];
    e.plans += b; e.acc += b; e.cls += b; e.sbout += b; e.arena += (size_t)b * ctx->arena_words;
    e.hdr = ctx->hdr_g + g;
    e.prev_total = g ? &ctx->hdr_g[g - 1].total_out : nullptr;
    BatchHdr hg = H; /* device-side consumers read S and status; max_pk_bytes / max_qcode / total_out are produced per group */
    hg.S = s0[g + 1] - s0[g]; hg.max_pk_bytes = 0; hg.max_qcode = 0; hg.total_out = 0; hg.out_begin = 0;
    ctx->h_hdr_g[g] = hg;
  }
  /* phase 1 (statistics) of every group, then phase 2 (coding) once the group's packed-table size is known on the host */
  for (u32 g = 0; g < G; ++g) {
    const Dev &e = dg[g];
    const u32 Sg = s0[g + 1] - s0[g];
    cudaStream_t gs = g ? ctx->gstream[g] : st;
#define GMARK() do { if (G == 1) PMARK(); } while (0)
    CK(cudaMemcpyAsync(ctx->hdr_g + g, ctx->h_hdr_g + g, sizeof(BatchHdr), cudaMemcpyHostToDevice, gs));
    CK(cudaMemsetAsync(e.acc, 0, sizeof(SbAcc) * Sg, gs));
    GMARK();
    k_stat1<<<dim3((max_tasks + s1_warps - 1) / s1_warps, Sg), s1_warps * 32, title_stat_dyn, gs>>>(e);
    k_xdelta<<<Sg, 128, 0, gs>>>(e); GMARK();
    k_zero_raw<<<dim3(4, Sg), 256, 0, gs>>>(e);
    {
      const dim3 g_sq((max_tasks + SQ_WARPS - 1) / SQ_WARPS, Sg);
#define PHY_SQ(G_) do { if (sq_wide) k_seqstat<G_, true><<<g_sq, SQ_WARPS * 32, sq_dyn, gs>>>(e); else k_seqstat<G_, false><<<g_sq, SQ_WARPS * 32, sq_dyn, gs>>>(e); } while (0)
      switch (encG) {
        case 1: PHY_SQ(1); break;
        case 2: PHY_SQ(2); break;
        case 4: PHY_SQ(4); break;
        default: PHY_SQ(8); break;
      }
#undef PHY_SQ
    }
    GMARK();
    k_classify<<<Sg, 32, 0, gs>>>(e); GMARK();
    /* the group header now holds the exact size of the packed quality tables: the copy is ordered before the
     * statistics kernels that follow, so the host gets it while they keep the GPU busy (only waited for when the
     * previous batch left no hint, see below) */
    CK(cudaMemcpyAsync(ctx->h_hdr_g + g, ctx->hdr_g + g, sizeof(BatchHdr), cudaMemcpyDeviceToHost, gs));
    CK(cudaEventRecord(ctx->ev_rb[g], gs));
    k_zero_hist<<<dim3(8, Sg), 256, 0, gs>>>(e); GMARK();
    k_stat2<<<dim3((H.max_chunks * (CH / 32) + S2W * S2B - 1) / (S2W * S2B), Sg), S2W * 32, 0, gs>>>(e);
    k_dnacount<<<dim3((H.max_chunks + S2G - 1) / S2G, Sg), CH, span, gs>>>(e); /* returns at once unless the DNA is Huffman coded */
    GMARK();
  }
  const u32 nq_hint = ctx->nq_hint; /* quality alphabet of the previous batch of this context (0: none yet) */
  for (u32 g = 0; g < G; ++g) {
    Dev &e = dg[g];
    const u32 Sg = s0[g + 1] - s0[g];
    cudaStream_t gs = g ? ctx->gstream[g] : st;
    /* Shared memory for the packed quality tables: (longest read + 1) x alphabet x 2 bytes.  The alphabet size is known
     * on the device only; the first batch of a context waits for the readback, later batches reserve room for the
     * alphabet the previous batch had plus eight symbols, so the GPU never waits for the host here (a subblock whose
     * tables outgrow the reservation reads them from global memory instead -- slower, same bytes). */
    u32 pk;
    if (nq_hint) pk = ((H.max_len + 1) * (nq_hint + 8 > 256 ? 256u : nq_hint + 8) * 2u + 15u) & ~15u;
    else { CK(cudaEventSynchronize(ctx->ev_rb[g])); pk = (ctx->h_hdr_g[g].max_pk_bytes + 15u) & ~15u; }
    e.pk_bytes = pk <= PK_SMEM_MAX ? pk : 0u; /* larger tables stay in global memory (L1) */
    k_huff<<<dim3(HUFF_LARGE + 32, Sg), HUFF_WARPS * 32, HUFF_SMEM, gs>>>(e); GMARK();
    /* single-walk encoder: slots, then title + info and quality + DNA of every task into the temporary buffer */
    e.fg.pk_bytes = e.pk_bytes;
    const u32 title_dyn = ENC_WARPS * enc_title_warp_bytes();
    const u32 qd_dyn = e.fg.pk_bytes + ENC_WARPS * (e.qd_nbuf * e.qd_stage + (32u * e.fg.lpw_q + 2u * CCW) * 4u);
    if (e.fg.g && (title_dyn > ENC_DYN_MAX || qd_dyn > ENC_DYN_MAX || e.fg.pk_bytes == 0)) e.fg.g = 0; /* does not fit: two-walk kernels */
    k_slots<<<Sg, 32, 0, gs>>>(e); GMARK();
    const dim3 g_enc((max_tasks + ENC_WARPS - 1) / ENC_WARPS, Sg);
    if (e.fg.g) k_enc_title<<<g_enc, ENC_WARPS * 32, title_dyn, gs>>>(e);
    GMARK();
    switch (e.fg.g) {
      case 1: k_enc_qd<1><<<g_enc, ENC_WARPS * 32, qd_dyn, gs>>>(e); break;
      case 2: k_enc_qd<2><<<g_enc, ENC_WARPS * 32, qd_dyn, gs>>>(e); break;
      case 4: k_enc_qd<4><<<g_enc, ENC_WARPS * 32, qd_dyn, gs>>>(e); break;
      case 8: k_enc_qd<8><<<g_enc, ENC_WARPS * 32, qd_dyn, gs>>>(e); break;
      default: break;
    }
    GMARK();
    /* two-walk kernels for the subblocks the single-walk kernels could not take (bounds beyond their staging): one warp
     * per 32-record block while at least ~32 warps of such CTAs fit an SM, else warp pairs on a shared stage */
    const u32 solo_dyn = e.pk_bytes + EW * e.enc_stage, pair_dyn = e.pk_bytes + EP * e.enc_stage;
    const bool pair = (solo_dyn + 7 * 1024) * 4 > 227u * 1024;
    const dim3 ge_solo((4 * H.max_chunks + EW * EGW - 1) / (EW * EGW), Sg), ge_pair((4 * H.max_chunks + EP * EGW - 1) / (EP * EGW), Sg);
    if (pair) k_lengths<true><<<ge_pair, EW * 32, pair_dyn, gs>>>(e);
    else k_lengths<false><<<ge_solo, EW * 32, solo_dyn, gs>>>(e);
    GMARK();
    k_layout<<<Sg, 256, 0, gs>>>(e); GMARK();
    if (g) CK(cudaStreamWaitEvent(gs, ctx->ev_scan[g - 1], 0)); /* the previous group's end of output */
    k_outscan<<<1, 256, 0, gs>>>(e); GMARK();
    if (G > 1) CK(cudaEventRecord(ctx->ev_scan[g], gs));
    k_zero_out<<<148 * 4, 256, 0, gs>>>(e); GMARK();
    if (e.fg.g) k_place<<<dim3(64, Sg), 256, 0, gs>>>(e);
    GMARK();
    if (pair) k_emit<true><<<ge_pair, EW * 32, pair_dyn, gs>>>(e);
    else k_emit<false><<<ge_solo, EW * 32, solo_dyn, gs>>>(e);
    GMARK();
    ctx->launches += e.fg.g ? 19 : 16;
    CK(cudaMemcpyAsync(ctx->h_sbout + s0[g], e.sbout, sizeof(SbOut) * Sg, cudaMemcpyDeviceToHost, gs));
    CK(cudaMemcpyAsync(ctx->h_hdr_g + g, ctx->hdr_g + g, sizeof(BatchHdr), cudaMemcpyDeviceToHost, gs)); /* max_pk_bytes: the next batch's hint */
    if (g == G - 1) CK(cudaMemcpyAsync(ctx->h_hdr, ctx->hdr_g + g, sizeof(BatchHdr), cudaMemcpyDeviceToHost, gs)); /* total_out = the end of the last group */
    if (g) { CK(cudaEventRecord(ctx->ev_done[g], gs)); CK(cudaStreamWaitEvent(st, ctx->ev_done[g], 0)); } /* the caller waits on the main stream */
  }
  ctx->prev_groups = G; ctx->prev_max_len = H.max_len;
  CK(cudaGetLastError());
  if (ctx->profile) {
    CK(cudaStreamSynchronize(st));
    for (int i = 0; i < NKERN && i + 1 < ctx->pi; ++i) { float t = 0; cudaEventElapsedTime(&t, ctx->pev[i], ctx->pev[i + 1]); ctx->pms[i] += t; }
    ctx->pcount++;
  }
  return PHY_OK;
}

/* Front and back part of the walk's batch one after the other on the main stream (the pipelined region call). */
static int run_batch(phy_ctx *ctx, const u8 *in, u8 *out, u64 out_cap, const Walk &w) {
  int rc = prefix_launch(ctx, ctx->stream, in, w);
  if (rc) return rc;
  rc = prefix_finish(ctx);
  if (rc) return rc;
  return run_body(ctx, out, out_cap);
}

static void fill_descs(phy_ctx *ctx, u32 S, u64 out_base, phy_subblock_desc *descs) {
  for (u32 i = 0; i < S; ++i) {
    const SbPlan &P = ctx->h_plans[i];
    const SbOut &O = ctx->h_sbout[i];
    phy_subblock_desc &D = descs[i];
    D.win_off = P.win_off; D.win_len = P.win_len; D.rec_start = P.rec_start; D.overlap = P.overlap;
    D.n_records = P.n_records; D.warnings = P.warnings; D.bytes_consumed = P.bytes_consumed;
    for (int k = 0; k < 4; ++k) D.sec_len[k] = O.sec_len[k];
    D.out_off = out_base + O.out_off; D.out_len = O.out_len; D.status = O.status;
  }
}

static const u64 HEAD_BYTES = 1u << 20; /* the '@' heuristic of a rank > 0 looks at this much of the region's head */

/* Region set-up of every walk: the parameters, the first record of a rank > 0 (found in `head`, the region's first
 * min(region_len, HEAD_BYTES) bytes on the host), the reference's plan state (uploaded on the main stream) and the first
 * batch.  The caller decides Walk::nl. */
static int walk_init(phy_ctx *ctx, const u8 *head, u64 region_len, const phy_region_params *p, Walk &w) {
  if (!p || p->np < 1 || p->rank < 0 || p->rank >= p->np || p->window_bytes == 0 || p->file_size == 0) { ctx->err = "bad region parameters"; return PHY_ERR_ARG; }
  u32 first = 0;
  if (p->rank != 0) {
    int64_t f = phy_find_first_record(head, region_len < HEAD_BYTES ? region_len : HEAD_BYTES);
    if (f < 0) { ctx->err = "no record start found at the beginning of the region"; return (int)f; }
    first = (u32)f;
  }
  plan_init(w.st, p->file_size, p->np, p->rank, p->window_bytes, p->overlap, p->record_cap, first, p->threads);
  if ((u64)w.st.wr_len > region_len) { ctx->err = "region_len is shorter than the rank's working region"; return PHY_ERR_ARG; }
  w.len = region_len; w.max_batch = ctx->max_batch; w.back = (u64)p->window_bytes + ctx->slack;
  if (region_len > ctx->max_batch && ctx->max_batch < 2 * w.back + 4096) { ctx->err = "max_batch_bytes is too small for the window size"; return PHY_ERR_CAPACITY; }
  w.place(0);
  *ctx->h_state = w.st;
  ctx->launches = 0;
  CK(cudaMemcpyAsync(ctx->plan_state, ctx->h_state, sizeof(PlanState), cudaMemcpyHostToDevice, ctx->stream));
  return PHY_OK;
}

/* Totals of a walk's descriptors. */
struct Tally {
  u32 n = 0;
  u64 bytes_in = 0, bytes_out = 0;
  int worst = 0;
  void add(const phy_subblock_desc *d, u32 k) {
    for (u32 i = 0; i < k; ++i) { bytes_in += d[i].bytes_consumed; bytes_out += d[i].out_len; if (d[i].status < worst) worst = d[i].status; }
    n += k;
  }
};

/* Fills *r (if given) and returns the worst subblock status. */
static int walk_result(phy_ctx *ctx, const Walk &w, const Tally &t, u64 out_used, float kernel_ms, float h2d_ms, float d2h_ms, phy_region_result *r) {
  if (r) {
    memset(r, 0, sizeof *r);
    r->n_subblocks = t.n; r->n_batches = w.nb; r->wr_overlap = (int32_t)w.st.rec_start; r->kernel_launches = ctx->launches;
    r->out_used = out_used; r->kernel_ms = kernel_ms; r->h2d_ms = h2d_ms; r->d2h_ms = d2h_ms;
    r->bytes_in = t.bytes_in; r->bytes_out = t.bytes_out;
  }
  if (t.worst) ctx->err = std::string("a subblock failed: ") + phy_strerror(t.worst);
  return t.worst;
}

extern "C" int phy_upload(phy_ctx *ctx, const uint8_t *region, uint64_t region_len) {
  if (!ctx || !region || region_len == 0) return PHY_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  ctx->resident_len = ctx->resident_out = 0; /* until the new bytes are in place */
  u8 *dst = ctx->in;
  if (region_len > ctx->max_batch) { /* larger than one batch: its own device buffers, walked batch by batch */
    CK(ctx->big_in.ensure(region_len + 4096));
    CK(ctx->big_out.ensure(region_len / 2 + (1u << 20) + 64));
    dst = ctx->big_in;
  }
  for (u64 o = 0; o < region_len; o += 1ull << 30) { /* 1 GiB pieces: pageable sources are staged by the driver */
    const u64 n = region_len - o < (1ull << 30) ? region_len - o : (1ull << 30);
    CK(cudaMemcpyAsync(dst + o, region + o, n, cudaMemcpyHostToDevice, ctx->stream));
  }
  /* 64 bytes of zero padding behind the data: vector loads may run past the end */
  CK(cudaMemsetAsync(dst + region_len, 0, 64, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->resident_len = region_len;
  return PHY_OK;
}

extern "C" int phy_compress_resident(phy_ctx *ctx, uint64_t region_len, const phy_region_params *params,
                                     phy_subblock_desc *descs, uint32_t *inout_n_descs, phy_region_result *result) {
  if (!ctx || !descs || !inout_n_descs) return PHY_ERR_ARG;
  if (region_len == 0 || region_len != ctx->resident_len) { ctx->err = "resident bytes do not match region_len"; return PHY_ERR_ARG; }
  CK(cudaSetDevice(ctx->device));
  const bool big = region_len > ctx->max_batch;
  u8 *rin = big ? ctx->big_in : ctx->in, *rout = big ? ctx->big_out : ctx->out;
  const u64 rout_cap = big ? ctx->big_out.cap - 64 : ctx->out_cap;
  cudaStream_t s = ctx->stream;
  std::vector<u8> head;
  if (params && params->rank != 0) { /* the head of the region is needed on the host for the '@' heuristic */
    head.resize(region_len < HEAD_BYTES ? region_len : HEAD_BYTES);
    CK(cudaMemcpy(head.data(), rin, head.size(), cudaMemcpyDeviceToHost));
  }
  Walk w;
  int rc = walk_init(ctx, head.data(), region_len, params, w);
  if (rc) return rc;
  if (w.st.is_last) {
    u8 last_byte = '\n';
    CK(cudaMemcpy(&last_byte, rin + region_len - 1, 1, cudaMemcpyDeviceToHost));
    w.nl = last_byte != '\n';
    if (w.nl) CK(cudaMemsetAsync(rin + region_len, '\n', 1, s));
  }
  CK(cudaEventRecord(ctx->ev_k0, s));
  /* The front part of batch b + 1 (record splitter, window chain: bandwidth- and latency-bound, 0.5 ms per GB) runs on a
   * lower-priority stream beside the back part of batch b (issue-bound record kernels); it only needs to know where batch
   * b's chain stopped, which batch b's own front part has already told the host.  Profiling and PHY_DEBUG_SYNC run each
   * batch's front part on the main stream after the back part of the batch before. */
  const bool ahead = !ctx->profile && !sw.debug_sync;
  cudaStream_t sp = ahead ? ctx->s_prefix : s;
  if (ahead) CK(cudaStreamWaitEvent(sp, ctx->ev_k0, 0)); /* the plan state is on the device first */
  const u32 cap_descs = *inout_n_descs;
  Tally t;
  u64 out_used = 0;
  rc = prefix_launch(ctx, sp, rin, w);
  if (rc) return rc;
  for (bool done = false; !done;) {
    rc = prefix_finish(ctx);
    if (rc) return rc;
    const u32 S = ctx->last_S;
    bool move;
    rc = w.after(ctx, *ctx->h_state, S, done, move);
    if (rc) return rc;
    if (t.n + S > cap_descs) { ctx->err = "descriptor array too small"; return PHY_ERR_CAPACITY; }
    if (move) w.place(w.candidate());
    rc = run_body(ctx, rout + out_used, rout_cap - out_used); /* first, so that the GPU is busy again as early as possible ... */
    if (rc) return rc;
    if (!done && ahead) { rc = prefix_launch(ctx, sp, rin + w.base, w); if (rc) return rc; } /* ... the next front part fills in beside it */
    CK(cudaStreamSynchronize(s));
    fill_descs(ctx, S, out_used, descs + t.n);
    t.add(descs + t.n, S);
    if (S) out_used += ctx->h_hdr->total_out;
    if (!done && !ahead) { rc = prefix_launch(ctx, sp, rin + w.base, w); if (rc) return rc; }
  }
  CK(cudaEventRecord(ctx->ev_k1, s));
  CK(cudaStreamSynchronize(s));
  float kernel_ms = 0;
  CK(cudaEventElapsedTime(&kernel_ms, ctx->ev_k0, ctx->ev_k1));
  *inout_n_descs = t.n;
  ctx->resident_out = out_used;
  return walk_result(ctx, w, t, out_used, kernel_ms, 0, 0, result);
}

extern "C" int phy_download(phy_ctx *ctx, uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
  if (!ctx || !out) return PHY_ERR_ARG;
  if (ctx->resident_out > out_cap) { ctx->err = "output buffer too small"; return PHY_ERR_CAPACITY; }
  CK(cudaSetDevice(ctx->device));
  const u8 *src = ctx->resident_len > ctx->max_batch ? ctx->big_out : ctx->out;
  CK(cudaMemcpyAsync(out, src, ctx->resident_out, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (out_len) *out_len = ctx->resident_out;
  return PHY_OK;
}

/* Copy streams, events and second buffers of the pipelined region call; the second input buffer is only needed for regions
 * of several batches. */
static int copy_init(phy_ctx *ctx, bool second_input) {
  CK(ctx->s_in.ensure(0)); /* default priority */
  CK(ctx->s_out.ensure(0));
  for (int i = 0; i < 2; ++i) {
    for (Event *e : {&ctx->ev_in[i], &ctx->ev_out[i], &ctx->ev_h0[i], &ctx->ev_d0[i]}) CK(e->ensure(cudaEventDefault));
    CK(ctx->ev_c[i].ensure(cudaEventDisableTiming));
  }
  if (second_input) CK(ctx->in2.ensure(ctx->max_batch + 4096, true));
  CK(ctx->out2.ensure(ctx->out_cap + 64));
  return PHY_OK;
}

/* ---- streamed host I/O (phy_compress_stream) ------------------------------------------------------------------------- */
/* The caller's region is not in memory: reader threads pull it chunk by chunk through the caller's read callback into a
 * ring of pinned staging slots, the uploads consume the chunks in order, payloads come back into two pinned output slots and
 * are handed to the caller's emit callback one batch behind the kernels. */
struct StreamIO {
  phy_read_fn read = nullptr; void *ruser = nullptr; phy_emit_fn emit = nullptr; void *euser = nullptr;
  phy_ctx *ctx = nullptr; u64 region_len = 0, nchunks = 0;
  std::mutex m; std::condition_variable cv;
  u64 ready[RING_SLOTS] = {};     /* slot holds chunk ready - 1 (0: nothing yet)                        */
  u64 consumed[RING_SLOTS] = {};  /* uploads of chunk consumed - 1 from this slot have been enqueued       */
  bool failed = false, stop = false;
  std::vector<std::thread> readers;
  /* finished batches: the emitter thread waits for a batch's payloads to arrive in their pinned slot and hands them to the
   * caller's emit callback, in order, while the calling thread is already launching later batches */
  struct Item { std::vector<phy_subblock_desc> descs; int hslot; };
  std::deque<Item> items;
  bool hbusy[HOUT_SLOTS] = {};
  bool emit_failed = false, emit_done = false;
  std::thread emitter;

  void emitter_main() {
    cudaSetDevice(ctx->device);
    for (;;) {
      Item it;
      {
        std::unique_lock<std::mutex> g(m);
        cv.wait(g, [&] { return emit_done || !items.empty(); });
        if (items.empty()) return;
        it = std::move(items.front()); items.pop_front();
      }
      cudaEventSynchronize(ctx->ev_hout[it.hslot]);
      bool bad = false;
      { std::lock_guard<std::mutex> g(m); bad = emit_failed; }
      if (!bad && emit(euser, it.descs.data(), (uint32_t)it.descs.size(), ctx->hout[it.hslot])) bad = true;
      { std::lock_guard<std::mutex> g(m); hbusy[it.hslot] = false; if (bad) emit_failed = true; }
      cv.notify_all();
    }
  }
  /* a free pinned payload slot (waits for the emitter when all are in use); -1 once the callback has failed */
  int acquire_hslot() {
    std::unique_lock<std::mutex> g(m);
    int k = -1;
    cv.wait(g, [&] { if (emit_failed) return true; for (int i = 0; i < HOUT_SLOTS; ++i) if (!hbusy[i]) { k = i; return true; } return false; });
    if (emit_failed) return -1;
    hbusy[k] = true;
    return k;
  }
  void push_item(const phy_subblock_desc *d, u32 n, int hslot) {
    { std::lock_guard<std::mutex> g(m); items.push_back(Item{std::vector<phy_subblock_desc>(d, d + n), hslot}); }
    cv.notify_all();
  }
  /* all batches handed over: wait for the emitter; false when the callback stopped the call */
  bool finish_emit() {
    { std::lock_guard<std::mutex> g(m); emit_done = true; }
    cv.notify_all();
    if (emitter.joinable()) emitter.join();
    return !emit_failed;
  }

  void reader_main(int t, int nthreads) {
    cudaSetDevice(ctx->device);
    for (u64 k = (u64)t; k < nchunks; k += (u64)nthreads) {
      const int slot = (int)(k % RING_SLOTS);
      {
        std::unique_lock<std::mutex> g(m);
        cv.wait(g, [&] { return stop || k < (u64)RING_SLOTS || consumed[slot] == k - RING_SLOTS + 1; });
        if (stop) return;
      }
      if (k >= (u64)RING_SLOTS) cudaEventSynchronize(ctx->ev_ring[slot]); /* the copies out of the slot's previous chunk are done */
      const u64 off = k * RING_CHUNK, n = region_len - off < RING_CHUNK ? region_len - off : RING_CHUNK;
      const int64_t got = read(ruser, off, ctx->ring + (u64)slot * RING_CHUNK, n);
      {
        std::lock_guard<std::mutex> g(m);
        if (got != (int64_t)n) failed = true;
        ready[slot] = k + 1;
      }
      cv.notify_all();
      if (got != (int64_t)n) return;
    }
  }
  /* blocks until chunk k is in its slot; nullptr on a read failure */
  const u8 *chunk(u64 k) {
    const int slot = (int)(k % RING_SLOTS);
    std::unique_lock<std::mutex> g(m);
    cv.wait(g, [&] { return failed || ready[slot] == k + 1; });
    return failed ? nullptr : ctx->ring + (u64)slot * RING_CHUNK;
  }
  void release(u64 k) { { std::lock_guard<std::mutex> g(m); consumed[k % RING_SLOTS] = k + 1; } cv.notify_all(); }
  void shutdown() {
    { std::lock_guard<std::mutex> g(m); stop = true; emit_done = true; }
    cv.notify_all();
    for (auto &t : readers) if (t.joinable()) t.join();
    readers.clear();
    if (emitter.joinable()) emitter.join();
  }
  ~StreamIO() { shutdown(); }
};

/* Pipelined over batches: while batch b is compressed, batch b+1 streams host -> device on a second stream and
 * the payloads of batch b-1 stream device -> host on a third (double-buffered input and output).  The start of
 * batch b+1 does not depend on batch b's result: it is placed one window + slack before the end of batch b, which
 * is never past the point where the window chain stops in batch b. */
static int compress_region_impl(phy_ctx *ctx, const uint8_t *region, uint64_t region_len, const phy_region_params *params,
                                phy_wait_fn wait, void *wait_user, uint8_t *out, uint64_t out_cap, phy_subblock_desc *descs,
                                uint32_t *inout_n_descs, phy_region_result *result, StreamIO *io = nullptr) {
  if (!ctx || region_len == 0) return PHY_ERR_ARG;
  if (!io && (!region || !out || !descs || !inout_n_descs)) return PHY_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  /* `wait` (streamed variant): region[0, upto) is only valid after wait(user, upto) has returned */
  auto need = [&](u64 upto) { if (wait) wait(wait_user, upto < region_len ? upto : region_len); };
  if (params && params->rank != 0) need(HEAD_BYTES);
  const uint8_t *head = region;
  if (io) { /* streamed I/O: the head of the region is the head of chunk 0 */
    head = io->chunk(0);
    if (!head) { ctx->err = "reading the region failed"; return PHY_ERR_ARG; }
  }
  Walk w;
  int rc = walk_init(ctx, head, region_len, params, w);
  if (rc) return rc;
  cudaStream_t s = ctx->stream;
  CK(cudaStreamSynchronize(s));
  const bool multi = region_len > ctx->max_batch;
  rc = copy_init(ctx, multi);
  if (rc) return rc;
  u8 *inb[2] = {ctx->in, multi ? ctx->in2 : ctx->in}, *outb[2] = {ctx->out, ctx->out2};
  std::vector<phy_subblock_desc> batch_descs; /* streamed I/O: descriptors of one batch at a time */
  if (io) { batch_descs.resize(ctx->max_sb); descs = batch_descs.data(); }
  const u32 cap_descs = io ? ctx->max_sb : *inout_n_descs;
  Tally t;
  u32 nd = 0;
  u64 out_used = 0;
  float k_ms = 0, h2d_ms = 0, d2h_ms = 0;

  /* enqueue the upload of the batch that starts at `base` into input buffer `slot` (stream s_in).  Bytes that the
   * previous upload already brought to the device (the tail of the other buffer: consecutive batches overlap by one
   * window + slack) are copied device-to-device instead of crossing PCIe a second time. */
  u64 up_base = 0, up_blen = 0; int up_slot = -1; /* last upload issued on s_in */
  bool up_timed[2] = {false, false};
  auto upload = [&](u64 base, int slot) -> int {
    const u64 blen = w.len_at(base);
    if (up_timed[slot]) { float ms; CK(cudaEventSynchronize(ctx->ev_in[slot])); CK(cudaEventElapsedTime(&ms, ctx->ev_h0[slot], ctx->ev_in[slot])); h2d_ms += ms; up_timed[slot] = false; }
    CK(cudaEventRecord(ctx->ev_h0[slot], ctx->s_in));
    u64 carry = 0;
    if (up_slot >= 0 && up_slot != slot && base >= up_base && base < up_base + up_blen) {
      carry = up_base + up_blen - base;
      if (carry > blen) carry = blen;
      CK(cudaMemcpyAsync(inb[slot], inb[up_slot] + (base - up_base), carry, cudaMemcpyDeviceToDevice, ctx->s_in));
    }
    /* host bytes in pieces: with a reader still filling the region (streamed variants) a piece crosses PCIe as soon as it is
     * there; a region that is already complete goes in one copy per batch (every copy call costs the engine a few microseconds) */
    const u64 piece = (wait || io) ? (16ull << 20) : (1ull << 30);
    u8 last_byte = '\n';
    for (u64 o = carry; o < blen;) {
      u64 n = blen - o < piece ? blen - o : piece;
      const u8 *src;
      if (io) { /* the part of this piece that lies in one chunk of the ring */
        const u64 off = base + o, k = off / RING_CHUNK, in_chunk = off - k * RING_CHUNK;
        const u8 *c = io->chunk(k);
        if (!c) { ctx->err = "reading the region failed"; return PHY_ERR_ARG; }
        const u64 chunk_len = region_len - k * RING_CHUNK < RING_CHUNK ? region_len - k * RING_CHUNK : RING_CHUNK;
        if (n > chunk_len - in_chunk) n = chunk_len - in_chunk;
        src = c + in_chunk;
        CK(cudaMemcpyAsync(inb[slot] + o, src, n, cudaMemcpyHostToDevice, ctx->s_in));
        if (in_chunk + n == chunk_len) { /* the chunk has been consumed: its slot may be refilled once this copy is done */
          CK(cudaEventRecord(ctx->ev_ring[k % RING_SLOTS], ctx->s_in));
          io->release(k);
        }
      } else {
        need(base + o + n);
        src = region + base + o;
        CK(cudaMemcpyAsync(inb[slot] + o, src, n, cudaMemcpyHostToDevice, ctx->s_in));
      }
      if (base + o + n == region_len) last_byte = src[n - 1];
      o += n;
    }
    CK(cudaMemsetAsync(inb[slot] + blen, 0, 64, ctx->s_in)); /* zero padding: vector loads may run past the end */
    if (base + blen == region_len && w.st.is_last && last_byte != '\n') { /* see Walk::nl */
      w.nl = true;
      CK(cudaMemsetAsync(inb[slot] + blen, '\n', 1, ctx->s_in));
    }
    CK(cudaEventRecord(ctx->ev_in[slot], ctx->s_in));
    up_timed[slot] = true;
    up_base = base; up_blen = blen; up_slot = slot;
    return PHY_OK;
  };

  /* Batches: input buffer `cur` holds the batch being compressed, the other one receives the next batch meanwhile (its
   * start does not depend on this batch's result: one window + slack before this batch's end is never past the point
   * where the window chain stops here).  Output buffers alternate every round: the payloads of round r leave for the
   * host on s_out while round r + 1 runs. */
  int cur = 0, oslot = 0;
  rc = upload(0, cur);
  if (rc) return rc;
  bool have_next = false, done = false;
  bool have_d2h[2] = {false, false};
  auto speculate = [&]() -> int { /* the kernels of the batch before the previous one have left the other input buffer (the host synchronised on them) */
    if (w.final || have_next) return PHY_OK;
    int r = upload(w.candidate(), cur ^ 1);
    have_next = r == PHY_OK;
    return r;
  };
  const bool late = wait != nullptr || io != nullptr; /* bytes may not be there yet: waiting for them must not hold this batch's kernels back */
  while (!done) {
    if (!late) { rc = speculate(); if (rc) return rc; } /* region bytes are all there: the next upload is queued before this batch's kernels */
    CK(cudaStreamWaitEvent(s, ctx->ev_in[cur], 0));
    if (have_d2h[oslot]) CK(cudaStreamWaitEvent(s, ctx->ev_out[oslot], 0)); /* the payloads of the round before the previous one have left that buffer */
    CK(cudaEventRecord(ctx->ev_k0, s));
    rc = run_batch(ctx, inb[cur], outb[oslot], ctx->out_cap, w);
    if (rc) return rc;
    CK(cudaEventRecord(ctx->ev_k1, s));
    CK(cudaEventRecord(ctx->ev_c[oslot], s));
    if (late) { rc = speculate(); if (rc) return rc; }
    CK(cudaStreamSynchronize(s));
    const u32 S = ctx->last_S;
    bool move;
    rc = w.after(ctx, *ctx->h_state, S, done, move);
    if (rc) return rc;
    if (io) { nd = 0; out_used = 0; } /* every batch goes to its own pinned output slot and descriptor list */
    if (nd + S > cap_descs) { ctx->err = "descriptor array too small"; return PHY_ERR_CAPACITY; }
    const u64 tot = S ? ctx->h_hdr->total_out : 0;
    if (!io && out_used + tot > out_cap) { ctx->err = "output buffer too small"; return PHY_ERR_CAPACITY; }
    int hslot = -1;
    if (io) { hslot = io->acquire_hslot(); if (hslot < 0) { ctx->err = "the emit callback stopped the call"; return PHY_ERR_ARG; } }
    uint8_t *hdst = io ? ctx->hout[hslot] : out + out_used;
    if (have_d2h[oslot]) { float ms; CK(cudaEventElapsedTime(&ms, ctx->ev_d0[oslot], ctx->ev_out[oslot])); d2h_ms += ms; have_d2h[oslot] = false; }
    CK(cudaStreamWaitEvent(ctx->s_out, ctx->ev_c[oslot], 0));
    CK(cudaEventRecord(ctx->ev_d0[oslot], ctx->s_out));
    if (tot) CK(cudaMemcpyAsync(hdst, outb[oslot], tot, cudaMemcpyDeviceToHost, ctx->s_out));
    CK(cudaEventRecord(ctx->ev_out[oslot], ctx->s_out));
    if (io) CK(cudaEventRecord(ctx->ev_hout[hslot], ctx->s_out));
    have_d2h[oslot] = true;
    fill_descs(ctx, S, out_used, descs + nd);
    t.add(descs + nd, S);
    if (io) io->push_item(descs, S, hslot); /* the emitter thread hands the batch to the caller once its payloads have arrived */
    float ms;
    CK(cudaEventElapsedTime(&ms, ctx->ev_k0, ctx->ev_k1)); k_ms += ms;
    nd += S; out_used += tot; oslot ^= 1;
    if (move) { cur ^= 1; w.place(w.candidate()); have_next = false; } /* else the next round continues in the same bytes */
  }
  CK(cudaStreamSynchronize(ctx->s_in));
  CK(cudaStreamSynchronize(ctx->s_out));
  for (int i = 0; i < 2; ++i) {
    float ms;
    if (have_d2h[i]) { CK(cudaEventElapsedTime(&ms, ctx->ev_d0[i], ctx->ev_out[i])); d2h_ms += ms; }
    if (up_timed[i]) { CK(cudaEventElapsedTime(&ms, ctx->ev_h0[i], ctx->ev_in[i])); h2d_ms += ms; }
  }
  if (io && !io->finish_emit()) { ctx->err = "the emit callback stopped the call"; return PHY_ERR_ARG; }
  if (inout_n_descs) *inout_n_descs = t.n;
  return walk_result(ctx, w, t, io ? t.bytes_out : out_used, k_ms, h2d_ms, d2h_ms, result);
}

extern "C" int phy_stream_prepare(phy_ctx *ctx) {
  if (!ctx) return PHY_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  int rc = copy_init(ctx, true);
  if (rc) return rc;
  CK(ctx->ring.ensure(RING_CHUNK * RING_SLOTS));
  for (auto &h : ctx->hout) CK(h.ensure(ctx->out_cap + 64));
  for (auto &e : ctx->ev_ring) CK(e.ensure(cudaEventDisableTiming));
  for (auto &e : ctx->ev_hout) CK(e.ensure(cudaEventDisableTiming));
  return PHY_OK;
}

extern "C" int phy_compress_stream(phy_ctx *ctx, uint64_t region_len, const phy_region_params *params, phy_read_fn read, void *read_user,
                                   phy_emit_fn emit, void *emit_user, phy_region_result *result) {
  if (!ctx || !params || !read || !emit || region_len == 0) return PHY_ERR_ARG;
  int rc = phy_stream_prepare(ctx);
  if (rc) return rc;
  StreamIO io;
  io.read = read; io.ruser = read_user; io.emit = emit; io.euser = emit_user; io.ctx = ctx; io.region_len = region_len;
  io.nchunks = (region_len + RING_CHUNK - 1) / RING_CHUNK;
  for (int t = 0; t < READERS; ++t) io.readers.emplace_back([&io, t] { io.reader_main(t, READERS); });
  io.emitter = std::thread([&io] { io.emitter_main(); });
  rc = compress_region_impl(ctx, nullptr, region_len, params, nullptr, nullptr, nullptr, 0, nullptr, nullptr, result, &io);
  io.shutdown();
  cudaStreamSynchronize(ctx->s_in); /* a failed call may leave copies out of the ring in flight */
  return rc;
}

extern "C" int phy_compress_region(phy_ctx *ctx, const uint8_t *region, uint64_t region_len, const phy_region_params *params,
                                   uint8_t *out, uint64_t out_cap, phy_subblock_desc *descs, uint32_t *inout_n_descs,
                                   phy_region_result *result) {
  return compress_region_impl(ctx, region, region_len, params, nullptr, nullptr, out, out_cap, descs, inout_n_descs, result);
}

extern "C" int phy_compress_region_streamed(phy_ctx *ctx, const uint8_t *region, uint64_t region_len, const phy_region_params *params,
                                            phy_wait_fn wait, void *user, uint8_t *out, uint64_t out_cap, phy_subblock_desc *descs,
                                            uint32_t *inout_n_descs, phy_region_result *result) {
  return compress_region_impl(ctx, region, region_len, params, wait, user, out, out_cap, descs, inout_n_descs, result);
}

extern "C" int phy_profile(phy_ctx *ctx, int enable) {
  if (!ctx) return PHY_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  if (enable) for (auto &e : ctx->pev) CK(e.ensure(cudaEventDefault));
  ctx->profile = enable != 0;
  for (auto &m : ctx->pms) m = 0;
  ctx->pcount = 0;
  return PHY_OK;
}

extern "C" int phy_profile_read(phy_ctx *ctx, const char **names, float *ms, int cap) {
  if (!ctx) return PHY_ERR_ARG;
  int n = cap < NKERN ? cap : NKERN;
  for (int i = 0; i < n; ++i) { if (names) names[i] = KERNEL_NAMES[i]; if (ms) ms[i] = ctx->pcount ? ctx->pms[i] / ctx->pcount : 0.f; }
  return n;
}

extern "C" int64_t phy_debug_read(phy_ctx *ctx, const char *name, uint64_t offset, void *dst, uint64_t bytes) {
  if (!ctx || !name || !dst) return PHY_ERR_ARG;
  struct { const char *n; const void *p; u64 size; } tab[] = {
      {"te", ctx->te, (u64)ctx->maxrec * 4}, {"se", ctx->se, (u64)ctx->maxrec * 4}, {"rstart", ctx->rstart, (u64)ctx->maxrec * 4},
      {"kx", ctx->kx, (u64)ctx->maxrec * 2}, {"qoff", ctx->qoff, (u64)ctx->maxrec * 4}, {"doff", ctx->doff, (u64)ctx->maxrec * 4},
      {"toff", ctx->toff, (u64)ctx->maxrec * 4},
      {"plans", ctx->plans, sizeof(SbPlan) * ctx->max_sb}, {"acc", ctx->acc, sizeof(SbAcc) * ctx->max_sb},
      {"cls", ctx->cls, sizeof(SbClass) * ctx->max_sb}, {"arena", ctx->arena, (u64)ctx->arena_words * 4 * ctx->max_sb},
      {"hdr", ctx->hdr, sizeof(BatchHdr)}, {"sbout", ctx->sbout, sizeof(SbOut) * ctx->max_sb}, {"out", ctx->out, ctx->out_cap}};
  for (auto &e : tab)
    if (!strcmp(e.n, name)) {
      if (offset > e.size) return PHY_ERR_ARG;
      u64 n = bytes < e.size - offset ? bytes : e.size - offset;
      if (cudaMemcpy(dst, (const u8 *)e.p + offset, n, cudaMemcpyDeviceToHost) != cudaSuccess) { ctx->err = "debug read failed"; return PHY_ERR_CUDA; }
      return (int64_t)n;
    }
  /* sizes of the internal records, for test harnesses that want to decode the dumps */
  if (!strcmp(name, "sizeof")) {
    u32 v[6] = {(u32)sizeof(SbPlan), (u32)sizeof(SbAcc), (u32)sizeof(SbClass), (u32)sizeof(BatchHdr), (u32)sizeof(SbOut), ctx->arena_words};
    u64 n = bytes < sizeof v ? bytes : sizeof v;
    memcpy(dst, v, n);
    return (int64_t)n;
  }
  return PHY_ERR_ARG;
}
