// C ABI glue: validation, conv dispatch, workspace planning, and the DAG that enqueues a
// whole surrogate forward (NewFluidNet.forward, pytorch_networks_convae.py:1315-1388) and
// the TS time-stepping loop (:377-475) without any host synchronisation.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <string>

#include "common.cuh"

namespace pbmc {

static thread_local std::string g_last_cuda_error;
void set_last_cuda_error(cudaError_t e, const char* where) {
  g_last_cuda_error = std::string(where) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
  (void)cudaGetLastError();  // clear the sticky-less error so later launches are not blamed
}

int conv_ffma_dispatch(const pbmc_conv_desc& d, cudaStream_t st);
int conv_umma_dispatch(const pbmc_conv_desc& d, cudaStream_t st);  // conv_umma.cu
bool conv_umma_supported(const pbmc_conv_desc& d);
// pdl: launch with programmatic stream serialization (the kernel waits for its predecessor with griddepcontrol.wait)
int conv_row_dispatch(const pbmc_conv_desc& d, cudaStream_t st, bool pdl);  // conv_row.cu
bool conv_row_supported(const pbmc_conv_desc& d);
int conv_mux_dispatch(const pbmc_conv_desc& d, cudaStream_t st, bool pdl);  // conv_mux.cu
bool conv_mux_supported(const pbmc_conv_desc& d);
bool conv_mux_one_wave(const pbmc_conv_desc& d);
int conv_trunk_dispatch(const pbmc_trunk_desc& t, cudaStream_t st, bool pdl);  // conv_trunk.cu
bool conv_trunk_supported(const pbmc_trunk_desc& t);
double conv_trunk_layer_cost(int rpc);
int head_enqueue(const float* y, const double* chan_sum, const pbmc_member* members, float a_bound, int head_kind, int p_pred,
                 float* u, float* v, float* p, uint32_t* uvmax, int B, int H, int W, cudaStream_t st, bool pdl);  // head.cu
int build_input_enqueue(const float* T, const float* xc, const float* yc, const float* ycc, const pbmc_member* members, float* inp,
                        float* V, int B, int H, int W, void* zero, size_t zero_bytes, cudaStream_t st, bool pdl);  // pyramid.cu
int advect_diffuse_enqueue(const float* T, const float* u, const float* v, const float* x, const float* y,
                           const pbmc_member* members, const uint32_t* uvmax_in, int member_stride, double dx_min, double cn_max,
                           double dt_fixed, float* T_out, uint32_t* uvmax_out, double* dt_out, int B, int H, int W, cudaStream_t st,
                           bool pdl);  // stencil.cu
int clock_enqueue(pbmc_member_clock* clk, const float* Tin, float* Tout, const float* u, const float* v, const float* p,
                  double* dt_row, double* meanT_row, float* ring, double* meta, int slots, int B, int H, int W,
                  const pbmc_member_queue* queue, pbmc_member* members, int64_t* seq_row, const pbmc_diag_desc* diag,
                  const pbmc_member_chain* chain, cudaStream_t st);  // clock.cu

}  // namespace pbmc

using namespace pbmc;

struct pbmc_ctx {
  static constexpr int NSTREAM = PBMC_MAX_LEVELS;
  cudaStream_t s[NSTREAM];
  cudaEvent_t ev_fork[NSTREAM + 2];
  cudaEvent_t ev_join[NSTREAM];
  cudaEvent_t ev_in, ev_out;
};

extern "C" const char* pbmc_error_string(int st) {
  switch (st) {
    case PBMC_OK: return "ok";
    case PBMC_ERR_BAD_SHAPE: return "bad shape";
    case PBMC_ERR_UNSUPPORTED: return "unsupported configuration";
    case PBMC_ERR_NULL_POINTER: return "null pointer";
    case PBMC_ERR_MISALIGNED: return "pointer not 16-byte aligned";
    case PBMC_ERR_WORKSPACE: return "workspace too small";
    case PBMC_ERR_CUDA: return "CUDA error (see pbmc_last_cuda_error)";
    case PBMC_ERR_NOT_DEVICE_POINTER: return "pointer is not device memory";
    default: return "unknown status";
  }
}
extern "C" int pbmc_version(void) { return PBMC_VERSION; }
extern "C" const char* pbmc_last_cuda_error(void) { return g_last_cuda_error.c_str(); }
extern "C" size_t pbmc_sizeof(const char* name) {
  if (!name) return 0;
  if (!strcmp(name, "pbmc_member")) return sizeof(pbmc_member);
  if (!strcmp(name, "pbmc_src")) return sizeof(pbmc_src);
  if (!strcmp(name, "pbmc_conv_desc")) return sizeof(pbmc_conv_desc);
  if (!strcmp(name, "pbmc_layer")) return sizeof(pbmc_layer);
  if (!strcmp(name, "pbmc_net")) return sizeof(pbmc_net);
  if (!strcmp(name, "pbmc_slab_sync")) return sizeof(pbmc_slab_sync);
  if (!strcmp(name, "pbmc_trunk_desc")) return sizeof(pbmc_trunk_desc);
  if (!strcmp(name, "pbmc_edge9_desc")) return sizeof(pbmc_edge9_desc);
  if (!strcmp(name, "pbmc_member_clock")) return sizeof(pbmc_member_clock);
  if (!strcmp(name, "pbmc_member_queue")) return sizeof(pbmc_member_queue);
  if (!strcmp(name, "pbmc_diag_desc")) return sizeof(pbmc_diag_desc);
  if (!strcmp(name, "pbmc_member_chain")) return sizeof(pbmc_member_chain);
  return 0;
}

static int check_device_ptr(const void* p) {
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return PBMC_ERR_NOT_DEVICE_POINTER;
  }
  return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) ? PBMC_OK : PBMC_ERR_NOT_DEVICE_POINTER;
}

static int validate_conv(const pbmc_conv_desc& d) {
  if (d.nsrc <= 0 || d.nsrc > PBMC_MAX_SRC) return PBMC_ERR_BAD_SHAPE;
  if (d.B <= 0 || d.H <= 0 || d.W <= 0 || d.cout <= 0) return PBMC_ERR_BAD_SHAPE;
  if (d.ksize != 3 && d.ksize != 5) return PBMC_ERR_UNSUPPORTED;
  if (d.pad_mode < PBMC_PAD_ZEROS || d.pad_mode > PBMC_PAD_REFLECT) return PBMC_ERR_UNSUPPORTED;
  if (d.pad_mode == PBMC_PAD_REFLECT && (d.H <= d.ksize / 2 || d.W <= d.ksize / 2)) return PBMC_ERR_BAD_SHAPE;
  if (!d.wpk || !d.bias || !d.out) return PBMC_ERR_NULL_POINTER;
  if (!aligned16(d.wpk) || !aligned16(d.bias) || !aligned16(d.out)) return PBMC_ERR_MISALIGNED;
  for (int s = 0; s < d.nsrc; ++s) {
    const pbmc_src& S = d.src[s];
    if (!S.ptr) return PBMC_ERR_NULL_POINTER;
    if (!aligned16(S.ptr)) return PBMC_ERR_MISALIGNED;
    if (S.nblk <= 0) return PBMC_ERR_BAD_SHAPE;
    if ((S.xform == PBMC_XFORM_GN_GELU || S.xform == PBMC_XFORM_GN) && (!S.stats || !S.gamma || !S.beta))
      return PBMC_ERR_NULL_POINTER;
    if (S.xform < PBMC_XFORM_NONE || S.xform > PBMC_XFORM_SCALE) return PBMC_ERR_UNSUPPORTED;
    if (S.xform == PBMC_XFORM_SCALE && !S.stats) return PBMC_ERR_NULL_POINTER;
  }
  return PBMC_OK;
}

static int conv_enqueue(const pbmc_conv_desc& d, cudaStream_t st, bool pdl) {
  int rc = validate_conv(d);
  if (rc != PBMC_OK) return rc;
  int impl = d.impl;
  bool staged = false;
  for (int s = 0; s < d.nsrc; ++s) {
    if (d.src[s].layout != PBMC_LAYOUT_BLOCKED && d.src[s].layout != PBMC_LAYOUT_STAGED16) return PBMC_ERR_UNSUPPORTED;
    staged = staged || d.src[s].layout == PBMC_LAYOUT_STAGED16;
  }
  if (staged) {
    // operand images are only understood by the fp16 hi|lo row kernel (which checks the rest: 3x3, replicate, ...)
    if (impl != PBMC_CONV_AUTO && impl != PBMC_CONV_ROW_F16X2 && impl != PBMC_CONV_MUX_F16X2) return PBMC_ERR_UNSUPPORTED;
    impl = PBMC_CONV_ROW_F16X2;
  }
  if (impl == PBMC_CONV_AUTO)
    impl = (d.wpk_row && conv_mux_supported(d) && conv_mux_one_wave(d)) ? PBMC_CONV_MUX_F16X2
           : (d.wpk_row && conv_row_supported(d))   ? PBMC_CONV_ROW_F16X2
           : (d.wpk_umma && conv_umma_supported(d)) ? PBMC_CONV_UMMA_F16X2
                                                    : PBMC_CONV_FFMA;
  // a SCALE source is understood by the mux kernel only
  for (int s = 0; s < d.nsrc; ++s)
    if (d.src[s].xform == PBMC_XFORM_SCALE &&
        ((impl != PBMC_CONV_MUX_F16X2 && impl != PBMC_CONV_MUX_BF16) || !d.wpk_row || !conv_mux_supported(d)))
      return PBMC_ERR_UNSUPPORTED;
  if (impl == PBMC_CONV_MUX_F16X2 || impl == PBMC_CONV_MUX_BF16) {
    if (!d.wpk_row) return PBMC_ERR_UNSUPPORTED;
    if (conv_mux_supported(d)) {
      pbmc_conv_desc e = d;
      e.impl = impl;
      return conv_mux_dispatch(e, st, pdl);
    }
    impl = impl == PBMC_CONV_MUX_F16X2 ? PBMC_CONV_ROW_F16X2 : PBMC_CONV_ROW_BF16;  // multi-source / 5x5: row kernel
  }
  if (impl == PBMC_CONV_ROW_F16X2 || impl == PBMC_CONV_ROW_BF16) {
    if (!d.wpk_row || !conv_row_supported(d)) return PBMC_ERR_UNSUPPORTED;
    pbmc_conv_desc e = d;
    e.impl = impl;
    return conv_row_dispatch(e, st, pdl);
  }
  // FFMA and UMMA never take pdl: their kernels do not execute griddepcontrol.wait
  if (impl == PBMC_CONV_FFMA) return conv_ffma_dispatch(d, st);
  if (impl == PBMC_CONV_UMMA_3XTF32 || impl == PBMC_CONV_UMMA_BF16 || impl == PBMC_CONV_UMMA_F16X2) {
    if (!d.wpk_umma || !conv_umma_supported(d)) return PBMC_ERR_UNSUPPORTED;
    pbmc_conv_desc e = d;
    e.impl = impl;
    return conv_umma_dispatch(e, st);
  }
  return PBMC_ERR_UNSUPPORTED;
}

extern "C" int pbmc_conv_fwd(const pbmc_conv_desc* d, void* stream) {
  if (!d) return PBMC_ERR_NULL_POINTER;
  int rc = check_device_ptr(d->out);
  if (rc != PBMC_OK) return rc;
  return conv_enqueue(*d, (cudaStream_t)stream, false);
}

extern "C" int pbmc_trunk_fwd(const pbmc_trunk_desc* t, void* stream) {
  if (!t || !t->layers) return PBMC_ERR_NULL_POINTER;
  if (t->pad_mode < PBMC_PAD_ZEROS || t->pad_mode > PBMC_PAD_REFLECT) return PBMC_ERR_UNSUPPORTED;
  if (t->pad_mode == PBMC_PAD_REFLECT && (t->H <= 1 || t->W <= 1)) return PBMC_ERR_BAD_SHAPE;
  if (!t->ping[0]) return PBMC_ERR_NULL_POINTER;
  int rc = check_device_ptr(t->ping[0]);
  if (rc != PBMC_OK) return rc;
  return conv_trunk_dispatch(*t, (cudaStream_t)stream, false);
}
extern "C" int pbmc_trunk_supported(const pbmc_trunk_desc* t) { return t && t->layers && conv_trunk_supported(*t) ? 1 : 0; }

extern "C" int pbmc_ctx_create(pbmc_ctx** out) {
  if (!out) return PBMC_ERR_NULL_POINTER;
  pbmc_ctx* c = new pbmc_ctx();
  // s[0] carries the critical chain (conv0 -> level-0 trunk -> conv1..3 -> head) at the highest priority, the
  // coarse pyramid levels run on s[1..] at the lowest: a level-0 CTA never queues behind coarse-level work
  int prio_lo = 0, prio_hi = 0;
  PBMC_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  for (int i = 0; i < pbmc_ctx::NSTREAM; ++i) {
    PBMC_CUDA(cudaStreamCreateWithPriority(&c->s[i], cudaStreamNonBlocking, i == 0 ? prio_hi : prio_lo));
    PBMC_CUDA(cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming));
  }
  for (int i = 0; i < pbmc_ctx::NSTREAM + 2; ++i) PBMC_CUDA(cudaEventCreateWithFlags(&c->ev_fork[i], cudaEventDisableTiming));
  PBMC_CUDA(cudaEventCreateWithFlags(&c->ev_in, cudaEventDisableTiming));
  PBMC_CUDA(cudaEventCreateWithFlags(&c->ev_out, cudaEventDisableTiming));
  *out = c;
  return PBMC_OK;
}
extern "C" int pbmc_ctx_destroy(pbmc_ctx* c) {
  if (!c) return PBMC_OK;
  for (int i = 0; i < pbmc_ctx::NSTREAM; ++i) {
    cudaStreamDestroy(c->s[i]);
    cudaEventDestroy(c->ev_join[i]);
  }
  for (int i = 0; i < pbmc_ctx::NSTREAM + 2; ++i) cudaEventDestroy(c->ev_fork[i]);
  cudaEventDestroy(c->ev_in);
  cudaEventDestroy(c->ev_out);
  delete c;
  return PBMC_OK;
}

// ------------------------------------------------------------------ workspace plan
namespace {
struct Plan {
  int L, R, CB, CIB, COB3;
  int Hl[PBMC_MAX_LEVELS], Wl[PBMC_MAX_LEVELS];
  size_t inp, x0, pooled[PBMC_MAX_LEVELS], ping[PBMC_MAX_LEVELS][2], up[PBMC_MAX_LEVELS], h1, h2, h3;
  size_t stats, stats_bytes, chan_sum, sync, uvmax, total;  // sync: [L][B] grid-barrier counters of the persistent trunk kernels
  // stats slots: 0 = conv0, 1 + l*R + r = trunk, 1 + L*R = conv1, 2 + L*R = conv2
  size_t stat_off(int slot, int B) const { return stats + (size_t)slot * B * CB * 2 * sizeof(double); }
};

inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

int make_plan(const pbmc_net& n, int B, int H, int W, Plan& P) {
  if (n.levels < 1 || n.levels > PBMC_MAX_LEVELS || n.repeats < 1 || n.repeats > PBMC_MAX_REPEATS) return PBMC_ERR_UNSUPPORTED;
  if (n.c_h < 4 || n.c_h % 4 != 0 || n.c_i < 1 || n.c_o < 1 || n.c_o > 4) return PBMC_ERR_UNSUPPORTED;
  if (B <= 0 || H < 3 || W < 3) return PBMC_ERR_BAD_SHAPE;
  const bool learned = (n.flags & PBMC_NET_LEARNED) != 0;
  // learned 9-region convs: the ring kernel takes one 16-wide c_out tile and sources of <= 128 channels, and every level
  // must hold the reference's boundary strips (pbmc_conv_edge9; the reference's strips would overlap otherwise)
  const int strip = n.ksize == 5 ? 6 : n.ksize;
  if (learned && (n.c_h > 16 || n.c_i > 128 || (n.ksize != 3 && n.ksize != 5) || n.levels + 1 > PBMC_MAX_SRC))
    return PBMC_ERR_UNSUPPORTED;
  if (learned && (H < strip || W < strip)) return PBMC_ERR_UNSUPPORTED;
  P.L = n.levels; P.R = n.repeats; P.CB = n.c_h / 4; P.CIB = (n.c_i + 3) / 4; P.COB3 = (n.c_o + 3) / 4;
  P.Hl[0] = H; P.Wl[0] = W;
  for (int l = 1; l < P.L; ++l) {
    P.Hl[l] = P.Hl[l - 1] / 2; P.Wl[l] = P.Wl[l - 1] / 2;
    if (P.Hl[l] < 1 || P.Wl[l] < 1) return PBMC_ERR_BAD_SHAPE;
    if (learned && (P.Hl[l] < strip || P.Wl[l] < strip)) return PBMC_ERR_UNSUPPORTED;
    if (!learned && n.pad_mode == PBMC_PAD_REFLECT && (P.Hl[l] <= n.ksize / 2 || P.Wl[l] <= n.ksize / 2)) return PBMC_ERR_BAD_SHAPE;
  }
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes); return o; };
  const size_t px = (size_t)H * W;
  P.inp = take((size_t)B * P.CIB * px * 16);
  P.x0 = take((size_t)B * P.CB * px * 16);
  for (int l = 0; l < P.L; ++l) {
    const size_t pl = (size_t)P.Hl[l] * P.Wl[l];
    P.pooled[l] = l ? take((size_t)B * P.CB * pl * 16) : 0;
    P.ping[l][0] = take((size_t)B * P.CB * pl * 16);
    P.ping[l][1] = take((size_t)B * P.CB * pl * 16);
    P.up[l] = l ? take(std::max((size_t)B * P.CB * px * 16, pbmc_staged_bytes(B, H, W))) : 0;  // blocked fp32 or staged fp16 hi|lo
  }
  P.h1 = take((size_t)B * P.CB * px * 16);
  P.h2 = take((size_t)B * P.CB * px * 16);
  P.h3 = take((size_t)B * P.COB3 * px * 16);
  const int nslots = 3 + P.L * P.R;
  const size_t sync_bytes = ((size_t)P.L * B * sizeof(uint32_t) + 7) & ~(size_t)7;
  P.stats_bytes = (size_t)nslots * B * P.CB * 2 * sizeof(double) + (size_t)B * P.COB3 * 4 * sizeof(double) + sync_bytes +
                  (size_t)2 * B * sizeof(uint32_t);
  P.stats = take(P.stats_bytes);
  P.chan_sum = P.stats + (size_t)nslots * B * P.CB * 2 * sizeof(double);
  P.sync = P.chan_sum + (size_t)B * P.COB3 * 4 * sizeof(double);
  P.uvmax = P.sync + sync_bytes;
  P.total = off;
  return PBMC_OK;
}

inline pbmc_src make_src(const float* ptr, int nblk, int xform, const double* stats, const pbmc_layer* producer,
                         double inv_count) {
  pbmc_src s;
  s.ptr = ptr; s.nblk = nblk; s.xform = xform; s.stats = stats; s.layout = PBMC_LAYOUT_BLOCKED; s.reserved = 0;
  s.gamma = producer ? producer->gamma : nullptr;
  s.beta = producer ? producer->beta : nullptr;
  s.inv_count = inv_count;
  return s;
}

inline void fill_conv(pbmc_conv_desc& d, const pbmc_net& n, const pbmc_layer& L, int B, int H, int W, float* out,
                      double* ostats, double* ochan, int epi_act) {
  memset(&d, 0, sizeof(d));
  d.B = B; d.H = H; d.W = W;
  // a learned net's interior filters only produce the pixels whose window stays inside the image: zeros is the cheapest
  d.cout = L.cout; d.ksize = L.ksize; d.pad_mode = (n.flags & PBMC_NET_LEARNED) ? PBMC_PAD_ZEROS : n.pad_mode; d.epi_act = epi_act; d.impl = n.conv_impl;
  d.wpk = L.wpk; d.wpk_umma = L.wpk_umma; d.wpk_row = L.wpk_row; d.bias = L.bias; d.out = out; d.out_stats = ostats; d.out_chan_sum = ochan;
}

// Second launch of a learned 9-region conv: the ring kernel (pbmc_conv_edge9) over the conv `d` just enqueued -- same
// sources, output and statistics, which it repairs for the ring pixels
inline int ring_enqueue(const pbmc_conv_desc& d, const float* wedge, cudaStream_t st) {
  pbmc_edge9_desc e;
  memset(&e, 0, sizeof(e));
  for (int s = 0; s < d.nsrc; ++s) e.src[s] = d.src[s];
  e.nsrc = d.nsrc; e.B = d.B; e.H = d.H; e.W = d.W;
  e.cout = d.cout; e.ksize = d.ksize; e.epi_act = d.epi_act;
  e.wedge = wedge; e.bias = d.bias; e.out = d.out; e.out_stats = d.out_stats; e.out_chan_sum = d.out_chan_sum;
  return pbmc_conv_edge9(&e, st);
}
}  // namespace

extern "C" size_t pbmc_workspace_bytes(const pbmc_net* n, int B, int H, int W) {
  Plan P;
  if (!n || make_plan(*n, B, H, W, P) != PBMC_OK) return 0;
  return P.total;
}

#define RC(call)                 \
  do {                           \
    int _rc = (call);            \
    if (_rc != PBMC_OK) return _rc; \
  } while (0)

// Enqueue one surrogate forward.  `uv` points at the 2*B uint32 slots (uvmax of this step).
static int surrogate_enqueue_on(pbmc_ctx* ctx, const pbmc_net& n, const Plan& P, char* ws, const float* inp,
                                const pbmc_member* members, float* u, float* v, float* p, uint32_t* uvmax, int B, int H,
                                int W, cudaStream_t st, bool pre_zeroed = false);

// The forward runs on the context's high-priority stream, forked from / joined to the caller's stream.
static int surrogate_enqueue(pbmc_ctx* ctx, const pbmc_net& n, const Plan& P, char* ws, const float* inp,
                             const pbmc_member* members, float* u, float* v, float* p, uint32_t* uvmax, int B, int H,
                             int W, cudaStream_t caller) {
  PBMC_CUDA(cudaEventRecord(ctx->ev_in, caller));
  PBMC_CUDA(cudaStreamWaitEvent(ctx->s[0], ctx->ev_in, 0));
  const int rc = surrogate_enqueue_on(ctx, n, P, ws, inp, members, u, v, p, uvmax, B, H, W, ctx->s[0]);
  // join even on error so that a capture in progress is not left with a dangling fork
  cudaEventRecord(ctx->ev_out, ctx->s[0]);
  cudaStreamWaitEvent(caller, ctx->ev_out, 0);
  return rc;
}

// Per-level CTA budgets of one forward and whether the trunk runs as persistent kernels (one launch per pyramid level).
static bool level_cta_budgets(const pbmc_net& n, const Plan& P, int B, int H, int W, int* cta_budget) {
  const int L = P.L, R = P.R, CB = P.CB;
  {
    double tot = 0.0, w[PBMC_MAX_LEVELS];
    for (int l = 0; l < L; ++l) { w[l] = (double)B * ((P.Wl[l] + 127) / 128) * P.Hl[l]; tot += w[l]; }
    for (int l = 0; l < L; ++l) {
      const int strips = B * ((P.Wl[l] + 127) / 128);
      int share = (int)(148.0 * w[l] / tot);
      const int floor_ctas = strips * ((P.Hl[l] + 7) / 8);  // no need for more than one CTA per 8 rows
      int want = share < 2 ? 2 : share;
      if (want > floor_ctas) want = floor_ctas;
      if (want < strips) want = strips;
      // big batches: a level that needs more CTAs than its share even at 64 rows per CTA simply runs in waves
      if ((long)strips * ((P.Hl[l] + 63) / 64) > want) want = 0;
      cta_budget[l] = L > 1 ? want : 0;
    }
  }
  // Persistent trunk kernels (csrc/conv_trunk.cu: the R layers of a level in one launch, grid barrier between layers)
  // need EVERY CTA of EVERY level resident at once: taken only when all levels have a budget and the budgets fit 148 SMs.
  // Never for learned nets: the kernel consumes each layer's GroupNorm statistics at its grid barrier, before a ring
  // kernel could repair them.
  bool trunk_persistent = (n.flags & (PBMC_NET_TRUNK_PER_LAYER | PBMC_NET_LEARNED)) == 0 && CB == 4 && n.ksize == 3;
  // Their budgets are balanced on finish times, not on row counts: a level's kernel takes R x (the kernel's own per-layer
  // cost model, which moves in steps of a staging round of 5 rows), the coarse levels start after their pooling chain and
  // must still be up-sampled before conv[1] can begin.  Smallest common finish time whose CTA counts fit 148 SMs
  // (512^2: 100 / 32 / 8 / 4 / 2 / 2 instead of the row-proportional 108 / 26 / 6 / 3 / 2 / 2: 0.2135 -> 0.2065 ms per step,
  // the level-0 kernel keeps its five rounds and the up-sampling of the others no longer trails it).
  if (trunk_persistent && L > 1) {
    struct Opt { int ctas; double t; };
    Opt opts[PBMC_MAX_LEVELS][32];
    int nopt[PBMC_MAX_LEVELS];
    double cand[PBMC_MAX_LEVELS * 32];
    int ncand = 0;
    bool ok = true;
    for (int l = 0; l < L && ok; ++l) {
      const int units = B * ((P.Wl[l] + 127) / 128), Hl = P.Hl[l];
      const double start = 6000.0 * l, tail = l ? 2000.0 + 0.06 * (double)B * H * W : 0.0;
      nopt[l] = 0;
      double last = 1e30;
      const int rpc_min = Hl < 8 ? Hl : 8;  // no more than one CTA per 8 rows (2 of 10 staged rows are halo)
      for (int rpc = Hl < 22 ? Hl : 22; rpc >= rpc_min && nopt[l] < 32; --rpc) {  // fewest CTAs first
        const double c = conv_trunk_layer_cost(rpc);
        const long ctas = (long)units * ((Hl + rpc - 1) / rpc);
        if (c <= 0.0 || ctas > 148) continue;
        const double t = start + R * c + tail;
        if (t < last - 1e-9) { opts[l][nopt[l]++] = Opt{(int)ctas, t}; cand[ncand++] = t; last = t; }
      }
      ok = nopt[l] > 0;
    }
    if (ok) {
      double best_t = 1e30;
      int best_b[PBMC_MAX_LEVELS];
      for (int k = 0; k < ncand; ++k) {
        if (cand[k] >= best_t) continue;
        int sum = 0, bb[PBMC_MAX_LEVELS];
        bool feas = true;
        for (int l = 0; l < L && feas; ++l) {
          int pick = -1;
          for (int o = 0; o < nopt[l]; ++o)
            if (opts[l][o].t <= cand[k] + 1e-9) { pick = opts[l][o].ctas; break; }  // options are ordered by CTA count
          feas = pick > 0;
          bb[l] = pick;
          sum += pick;
        }
        if (feas && sum <= 148) { best_t = cand[k]; for (int l = 0; l < L; ++l) best_b[l] = bb[l]; }
      }
      if (best_t < 1e30) {
        // CTAs left over go to the levels in order (level 0 heads the chain that conv[1] waits on): each takes its fastest
        // option that still fits
        int sum = 0;
        for (int l = 0; l < L; ++l) sum += best_b[l];
        for (int l = 0; l < L; ++l)
          for (int o = nopt[l] - 1; o >= 0; --o)
            if (opts[l][o].ctas > best_b[l] && sum - best_b[l] + opts[l][o].ctas <= 148) {
              sum += opts[l][o].ctas - best_b[l];
              best_b[l] = opts[l][o].ctas;
              break;
            }
        for (int l = 0; l < L; ++l) cta_budget[l] = best_b[l];
      }
    }
  }
  {
    int total = 0;
    for (int l = 0; l < L && trunk_persistent; ++l) {
      const int bud = L > 1 ? cta_budget[l] : 148;
      pbmc_trunk_desc t;
      memset(&t, 0, sizeof(t));
      t.src0.nblk = CB; t.src0.layout = PBMC_LAYOUT_BLOCKED; t.src0.xform = PBMC_XFORM_NONE;
      t.layers = &n.trunk[l * PBMC_MAX_REPEATS];
      t.R = R; t.B = B; t.H = P.Hl[l]; t.W = P.Wl[l]; t.impl = n.conv_impl; t.max_ctas = bud;
      trunk_persistent = bud > 0 && conv_trunk_supported(t);
      total += bud;
    }
    trunk_persistent = trunk_persistent && total <= 148;
  }
  return trunk_persistent;
}

// pre_zeroed: the caller's previous kernel has already cleared the scratch region [P.stats, P.stats + P.stats_bytes)
static int surrogate_enqueue_on(pbmc_ctx* ctx, const pbmc_net& n, const Plan& P, char* ws, const float* inp,
                                const pbmc_member* members, float* u, float* v, float* p, uint32_t* uvmax, int B, int H,
                                int W, cudaStream_t st, bool pre_zeroed) {
  const int L = P.L, R = P.R, CB = P.CB;
  // Programmatic dependent launch (pdl) on the critical chain:
  //   conv[2], conv[3]   on: nothing else runs then; the next conv's set-up overlaps the previous one's drain
  //   conv[1]            on  (0.2348 -> 0.2331 -> 0.2311 ms/step at 512^2 with conv[2..3], then also conv[1])
  //   head kernel        on
  //   conv[0]            on in a rollout (behind the input-build kernel, no memset node in between)
  //   level-0 trunk      on for the persistent kernel (one launch behind conv[0]; its 96 CTAs leave the other levels
  //                      their SMs: 0.2011 -> 0.2003 ms/step in 10-step graphs); with one launch PER LAYER it cost
  //                      0.27 ms -- an early-resident CTA parked in griddepcontrol.wait took an SM from the other
  //                      levels' streams -- and stays off there
  //   ring kernels of conv[0..3] (learned nets), each directly behind its interior conv: OFF -- measured slower on B200
  //                      (paper network, 128x506, B = 1, 10-step graphs: 0.521 vs 0.474 ms/step; 32 x 256^2: 5.41 vs
  //                      5.41 ms), so the ring kernels launch in plain stream order
  const bool learned = (n.flags & PBMC_NET_LEARNED) != 0;
  auto F = [&](size_t off) { return reinterpret_cast<float*>(ws + off); };
  auto S = [&](int slot) { return reinterpret_cast<double*>(ws + P.stat_off(slot, B)); };
  double* chan_sum = reinterpret_cast<double*>(ws + P.chan_sum);
  // zero all statistics accumulators (GroupNorm sums, zero-mean sums) in one memset
  if (!pre_zeroed) {
    PBMC_CUDA(cudaMemsetAsync(ws + P.stats, 0, P.stats_bytes - (size_t)2 * B * sizeof(uint32_t), st));
    if (uvmax) PBMC_CUDA(cudaMemsetAsync(uvmax, 0, (size_t)B * sizeof(uint32_t), st));
  }

  pbmc_conv_desc d;
  // conv[0]: FluidLayer(c_i -> c_h), :1317
  fill_conv(d, n, n.conv0, B, H, W, F(P.x0), S(0), nullptr, PBMC_ACT_NONE);
  d.nsrc = 1;
  d.src[0] = make_src(inp, P.CIB, PBMC_XFORM_NONE, nullptr, nullptr, 0.0);
  RC(conv_enqueue(d, st, pre_zeroed));  // rollout: directly behind the input-build kernel
  if (learned) RC(ring_enqueue(d, n.wedge_conv0, st));
  PBMC_CUDA(cudaEventRecord(ctx->ev_fork[0], st));

  // pyramid levels (:1319-1327): level l runs on stream l (level 0 on the caller's stream)
  // The L level chains run side by side and a tensor-core conv CTA owns an SM, so each level gets a share of the
  // 148 SMs in proportion to its row-strip count (with a floor so that the small levels do not become the
  // longest chain): every level then needs about the same time per layer instead of each launch trying to
  // fill the GPU on its own and queueing behind the others.
  int cta_budget[PBMC_MAX_LEVELS];
  const bool trunk_persistent = level_cta_budgets(n, P, B, H, W, cta_budget);
  // conv[1] is the only reader of the up-sampled levels: when it runs on the fp16 hi|lo row kernel (3x3, replicate
  // padding, 16 hidden channels) they are written directly as its operand image and staged by bulk copies
  bool up_staged = n.pad_mode == PBMC_PAD_REPLICATE && CB == 4 && n.conv1.ksize == 3 && n.conv1.wpk_row != nullptr &&
                   (n.conv_impl == PBMC_CONV_AUTO || n.conv_impl == PBMC_CONV_ROW_F16X2 || n.conv_impl == PBMC_CONV_MUX_F16X2);
  if (up_staged) {
    pbmc_conv_desc t;
    memset(&t, 0, sizeof(t));
    t.nsrc = L + 1; t.ksize = 3; t.cout = n.conv1.cout;
    for (int l = 0; l < L; ++l) t.src[l].nblk = CB;
    for (int l = 1; l < L; ++l) t.src[l].layout = PBMC_LAYOUT_STAGED16;
    t.src[L].nblk = P.CIB;
    up_staged = L + 1 <= PBMC_MAX_SRC && conv_row_supported(t);
  }
  // Off by default: measured neutral-to-slower in the whole step (512^2: 0.244-0.260 vs 0.241 ms; 32 x 256^2: 1.47 vs
  // 1.445 ms) -- conv[1] is paced by its MMA issue loop, not by its producers, and the operand-image writer of the
  // bicubic kernel stores 2 x 8 B per thread.  pbmc_net.flags & PBMC_NET_UP_STAGED turns it on (results are bit-identical).
  up_staged = up_staged && (n.flags & PBMC_NET_UP_STAGED) != 0 && !learned;  // the ring kernel reads blocked sources only
  const float* level_in[PBMC_MAX_LEVELS];
  level_in[0] = F(P.x0);
  for (int l = 0; l < L; ++l) {
    cudaStream_t sl = l ? ctx->s[l] : st;
    const int Hl = P.Hl[l], Wl = P.Wl[l];
    if (l > 0) {
      // pool^l(x_in) computed incrementally from level l-1's pooled input (identical composition)
      PBMC_CUDA(cudaStreamWaitEvent(sl, ctx->ev_fork[l - 1], 0));
      pbmc_src ps = (l == 1) ? make_src(F(P.x0), CB, PBMC_XFORM_GN_GELU, S(0), &n.conv0, 1.0 / (4.0 * H * W))
                             : make_src(F(P.pooled[l - 1]), CB, PBMC_XFORM_NONE, nullptr, nullptr, 0.0);
      RC(pbmc_avgpool2(&ps, F(P.pooled[l]), B, P.Hl[l - 1], P.Wl[l - 1], sl));
      PBMC_CUDA(cudaEventRecord(ctx->ev_fork[l], sl));
      level_in[l] = F(P.pooled[l]);
    }
    const double invc = 1.0 / (4.0 * Hl * Wl);
    if (trunk_persistent) {
      pbmc_trunk_desc t;
      memset(&t, 0, sizeof(t));
      t.src0 = (l == 0) ? make_src(F(P.x0), CB, PBMC_XFORM_GN_GELU, S(0), &n.conv0, invc)
                        : make_src(level_in[l], CB, PBMC_XFORM_NONE, nullptr, nullptr, 0.0);
      t.layers = &n.trunk[l * PBMC_MAX_REPEATS];
      t.ping[0] = F(P.ping[l][0]); t.ping[1] = F(P.ping[l][1]);
      t.stats = S(1 + l * R);
      t.sync = reinterpret_cast<unsigned int*>(ws + P.sync) + (size_t)l * B;
      t.R = R; t.B = B; t.H = Hl; t.W = Wl; t.pad_mode = n.pad_mode; t.impl = n.conv_impl;
      t.max_ctas = L > 1 ? cta_budget[l] : 148;
      t.pre_zeroed = 1;  // the statistics / counter region was zeroed by the memset at the top of the forward
      t.loader = (n.flags & PBMC_NET_TRUNK_BULK_LOADER) ? PBMC_TRUNK_LOADER_BULK : PBMC_TRUNK_LOADER_THREADS;
      RC(conv_trunk_dispatch(t, sl, l == 0));  // level 0 runs on the main stream, directly behind conv[0]
    }
    for (int r = 0; r < R && !trunk_persistent; ++r) {
      const pbmc_layer& Lr = n.trunk[l * PBMC_MAX_REPEATS + r];
      fill_conv(d, n, Lr, B, Hl, Wl, F(P.ping[l][r & 1]), S(1 + l * R + r), nullptr, PBMC_ACT_NONE);
      d.max_ctas = cta_budget[l];
      d.nsrc = 1;
      if (r == 0) {
        d.src[0] = (l == 0) ? make_src(F(P.x0), CB, PBMC_XFORM_GN_GELU, S(0), &n.conv0, invc)
                            : make_src(level_in[l], CB, PBMC_XFORM_NONE, nullptr, nullptr, 0.0);
      } else {
        d.src[0] = make_src(F(P.ping[l][(r - 1) & 1]), CB, PBMC_XFORM_GN_GELU, S(1 + l * R + r - 1),
                            &n.trunk[l * PBMC_MAX_REPEATS + r - 1], invc);
      }
      RC(conv_enqueue(d, sl, false));  // one launch per layer: never (see above)
      if (learned) RC(ring_enqueue(d, n.wedge_trunk[l * PBMC_MAX_REPEATS + r], sl));
    }
    if (l > 0) {
      pbmc_src us = make_src(F(P.ping[l][(R - 1) & 1]), CB, PBMC_XFORM_GN_GELU, S(1 + l * R + R - 1),
                             &n.trunk[l * PBMC_MAX_REPEATS + R - 1], invc);
      if (up_staged)
        RC(pbmc_bicubic_up_staged(&us, ws + P.up[l], B, Hl, Wl, H, W, sl));
      else
        RC(pbmc_bicubic_up(&us, F(P.up[l]), B, Hl, Wl, H, W, sl));
      PBMC_CUDA(cudaEventRecord(ctx->ev_join[l], sl));
    }
  }
  for (int l = 1; l < L; ++l) PBMC_CUDA(cudaStreamWaitEvent(st, ctx->ev_join[l], 0));

  // conv[1] over cat(levels..., inputs) (:1332-1335): the concat is a source list
  fill_conv(d, n, n.conv1, B, H, W, F(P.h1), S(1 + L * R), nullptr, PBMC_ACT_NONE);
  if (L + 1 > PBMC_MAX_SRC) return PBMC_ERR_UNSUPPORTED;
  d.nsrc = L + 1;
  d.src[0] = make_src(F(P.ping[0][(R - 1) & 1]), CB, PBMC_XFORM_GN_GELU, S(1 + R - 1), &n.trunk[R - 1], 1.0 / (4.0 * H * W));
  for (int l = 1; l < L; ++l) {
    d.src[l] = make_src(F(P.up[l]), CB, PBMC_XFORM_NONE, nullptr, nullptr, 0.0);
    if (up_staged) d.src[l].layout = PBMC_LAYOUT_STAGED16;
  }
  d.src[L] = make_src(inp, P.CIB, PBMC_XFORM_NONE, nullptr, nullptr, 0.0);
  RC(conv_enqueue(d, st, true));
  if (learned) RC(ring_enqueue(d, n.wedge_conv1, st));
  // conv[3] (:1342) with per-channel sums for the zero-mean (:1343).  Its source is conv[2]'s GELU output, which no
  // GroupNorm brings to order 1: its scale follows conv[2]'s weights, and an fp16 hi|lo split of it loses relative
  // precision below 2^-3 (subnormal lo part) and overflows above 65504.  Where conv[3] runs on the fp16 mux kernel, conv[2]
  // also accumulates its sums of squares and conv[3] reads h2 as a SCALE source (times 2^-s per sample, s from h2's rms;
  // the epilogue multiplies by 2^s: exact).  Elsewhere, when the fp16 split was asked for, conv[3] runs on the 3xTF32
  // split, which has fp32's exponent range (FFMA where the tensor-core kernel does not take the shape).
  pbmc_conv_desc d3;
  fill_conv(d3, n, n.conv3, B, H, W, F(P.h3), nullptr, chan_sum, PBMC_ACT_NONE);
  d3.nsrc = 1;
  d3.src[0] = make_src(F(P.h2), CB, PBMC_XFORM_SCALE, S(2 + L * R), nullptr, 0.0);
  const bool conv3_scaled = !learned && d3.wpk_row && conv_mux_supported(d3) &&
                            (d3.impl == PBMC_CONV_MUX_F16X2 || (d3.impl == PBMC_CONV_AUTO && conv_mux_one_wave(d3)));
  if (conv3_scaled) {
    d3.impl = PBMC_CONV_MUX_F16X2;
  } else {
    d3.src[0].xform = PBMC_XFORM_NONE;
    d3.src[0].stats = nullptr;
    if (d3.impl == PBMC_CONV_AUTO || d3.impl == PBMC_CONV_UMMA_F16X2 || d3.impl == PBMC_CONV_ROW_F16X2 || d3.impl == PBMC_CONV_MUX_F16X2)
      d3.impl = (d3.wpk_umma && conv_umma_supported(d3)) ? PBMC_CONV_UMMA_3XTF32 : PBMC_CONV_FFMA;
  }
  // gn[0] + act folded into conv[2]'s load; conv[2] + act (:1336-1340)
  fill_conv(d, n, n.conv2, B, H, W, F(P.h2), conv3_scaled ? S(2 + L * R) : nullptr, nullptr, PBMC_ACT_GELU);
  d.nsrc = 1;
  d.src[0] = make_src(F(P.h1), CB, PBMC_XFORM_GN_GELU, S(1 + L * R), &n.conv1, 1.0 / (4.0 * H * W));
  RC(conv_enqueue(d, st, true));
  if (learned) RC(ring_enqueue(d, n.wedge_conv2, st));
  d = d3;
  RC(conv_enqueue(d, st, true));
  if (learned) RC(ring_enqueue(d, n.wedge_conv3, st));
  return head_enqueue(F(P.h3), chan_sum, members, n.a_bound, n.head_kind, n.p_pred, u, v, p, uvmax, B, H, W, st, true);
}

extern "C" int pbmc_trunk_cta_budgets(const pbmc_net* net, int B, int H, int W, int* budgets) {
  if (!net || !budgets) return PBMC_ERR_NULL_POINTER;
  Plan P;
  RC(make_plan(*net, B, H, W, P));
  for (int l = 0; l < PBMC_MAX_LEVELS; ++l) budgets[l] = 0;
  return level_cta_budgets(*net, P, B, H, W, budgets) ? 1 : 0;
}

extern "C" int pbmc_surrogate_forward(pbmc_ctx* ctx, const pbmc_net* net, const float* inp, const pbmc_member* members,
                                      float* u, float* v, float* p, uint32_t* uvmax, void* workspace,
                                      size_t workspace_bytes, int B, int H, int W, void* stream) {
  if (!ctx || !net || !inp || !u || !v || !workspace) return PBMC_ERR_NULL_POINTER;
  Plan P;
  RC(make_plan(*net, B, H, W, P));
  if (workspace_bytes < P.total) return PBMC_ERR_WORKSPACE;
  if (!aligned16(workspace) || !aligned16(inp)) return PBMC_ERR_MISALIGNED;
  RC(check_device_ptr(workspace));
  return surrogate_enqueue(ctx, *net, P, (char*)workspace, inp, members, u, v, p, uvmax, B, H, W, (cudaStream_t)stream);
}

namespace pbmc {
__global__ void uvmax_batch_reduce_kernel(uint32_t* uv, int B) {
  // ADNet's dt is ONE scalar over the whole batch (pytorch_networks_convae.py:556): fold members into slot 0
  uint32_t m = 0;
  for (int i = threadIdx.x; i < B; i += 32) m = max(m, uv[i]);
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (threadIdx.x == 0) uv[0] = m;
}
}  // namespace pbmc

namespace {
// The clock arguments of pbmc_rollout_clocked (clock == NULL: plain pbmc_rollout)
struct ClockArgs {
  pbmc_member_clock* clock;
  double* meanT_seq;
  float* snap_ring;
  double* snap_meta;
  int snap_slots;
};
}  // namespace

// pbmc_rollout, pbmc_rollout_clocked, pbmc_rollout_queued, pbmc_rollout_diagnosed and pbmc_rollout_chained: the same
// launches in the same order; a clock adds its two launches behind every step's stencil, a queue (NULL except for
// pbmc_rollout_queued / _diagnosed / _chained, whose members are mutable), a diagnostics descriptor (NULL except for
// pbmc_rollout_diagnosed / _chained) and chains (NULL except for pbmc_rollout_chained) none
static int rollout_impl(pbmc_ctx* ctx, const pbmc_net* net, const pbmc_member* members, const float* xc, const float* yc,
                        const float* ycc, const float* xcoef, const float* ycoef, double dx_min, double cn_max,
                        int per_member_dt, float* T_seq, int nslots, int first_step, int n_steps, double* dt_seq,
                        int dt_seq_rows, float* u, float* v, float* p, float* V, void* workspace, size_t workspace_bytes,
                        int B, int H, int W, const ClockArgs& clk, const pbmc_member_queue* queue, const pbmc_diag_desc* diag,
                        const pbmc_member_chain* chain, void* stream) {
  if (!ctx || !net || !members || !xc || !yc || !ycc || !xcoef || !ycoef || !T_seq || !u || !v || !workspace) return PBMC_ERR_NULL_POINTER;
  if (nslots < 2 || first_step < 1 || n_steps < 0 || !(dx_min > 0.0)) return PBMC_ERR_BAD_SHAPE;
  if (dt_seq != nullptr && dt_seq_rows < first_step + n_steps - 1) return PBMC_ERR_BAD_SHAPE;  // step i writes row i - 1
  if (net->c_i != 7) return PBMC_ERR_UNSUPPORTED;  // TS builds the 7-channel input (:390-407)
  Plan P;
  RC(make_plan(*net, B, H, W, P));
  if (workspace_bytes < P.total) return PBMC_ERR_WORKSPACE;
  if (!aligned16(workspace)) return PBMC_ERR_MISALIGNED;
  RC(check_device_ptr(workspace));
  RC(check_device_ptr(T_seq));
  cudaStream_t caller = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  uint32_t* uvmax = reinterpret_cast<uint32_t*>(ws + P.uvmax);
  const size_t field = (size_t)B * H * W;
  // All steps run on the context's high-priority stream, forked from / joined to the caller's stream ONCE: inside the
  // loop every link of the critical chain (input build -> conv[0] -> ... -> head -> stencil -> next input build) is a
  // plain same-stream dependency, and the scratch of each forward is cleared by its input-build kernel.
  cudaStream_t st = ctx->s[0];
  PBMC_CUDA(cudaEventRecord(ctx->ev_in, caller));
  PBMC_CUDA(cudaStreamWaitEvent(st, ctx->ev_in, 0));
  auto steps = [&]() -> int {
    for (int i = first_step; i < first_step + n_steps; ++i) {
      const float* Tin = T_seq + (size_t)((i - 1) % nslots) * field;
      float* Tout = T_seq + (size_t)(i % nslots) * field;
      const bool last = (i == first_step + n_steps - 1);
      // programmatic dependent launch: behind the previous step's stencil (not for the call's first step: whatever
      // precedes it in the stream is not ours)
      RC(build_input_enqueue(Tin, xc, yc, ycc, members, reinterpret_cast<float*>(ws + P.inp), last ? V : nullptr, B, H, W, ws + P.stats,
                             P.stats_bytes, st, i > first_step));
      RC(surrogate_enqueue_on(ctx, *net, P, ws, reinterpret_cast<float*>(ws + P.inp), members, u, v, p, uvmax, B, H, W, st, true));
      if (!per_member_dt && B > 1) {
        uvmax_batch_reduce_kernel<<<1, 32, 0, st>>>(uvmax, B);
        PBMC_CHECK_LAUNCH("uvmax_batch_reduce_kernel");
      }
      // programmatic dependent launch when the stencil is directly behind the head kernel (no batch reduction between)
      RC(advect_diffuse_enqueue(Tin, u, v, xcoef, ycoef, members, uvmax, per_member_dt ? 1 : 0, dx_min, cn_max, 0.0, Tout, nullptr,
                                dt_seq ? dt_seq + (size_t)(i - 1) * B : nullptr, B, H, W, st, per_member_dt || B == 1));
      // plain stream order behind the stencil; the next step's input build is PDL-launched behind the commit kernel
      pbmc_diag_desc dg;  // the descriptor with the step's rows of flux_seq / vrms_seq
      if (diag) {
        dg = *diag;
        dg.flux_seq += (size_t)(i - 1) * B * 2;
        dg.vrms_seq += (size_t)(i - 1) * B;
      }
      if (clk.clock)
        RC(clock_enqueue(clk.clock, Tin, Tout, u, v, p, dt_seq + (size_t)(i - 1) * B, clk.meanT_seq + (size_t)(i - 1) * B,
                         clk.snap_ring, clk.snap_meta, clk.snap_slots, B, H, W, queue, const_cast<pbmc_member*>(members),
                         queue ? queue->member_seq + (size_t)(i - 1) * B : nullptr, diag ? &dg : nullptr, chain, st));
    }
    return PBMC_OK;
  };
  const int rc = steps();
  // join even on error so that a capture in progress is not left with a dangling fork
  cudaEventRecord(ctx->ev_out, st);
  cudaStreamWaitEvent(caller, ctx->ev_out, 0);
  return rc;
}

extern "C" int pbmc_rollout(pbmc_ctx* ctx, const pbmc_net* net, const pbmc_member* members, const float* xc,
                            const float* yc, const float* ycc, const float* xcoef, const float* ycoef, double dx_min,
                            double cn_max,
                            int per_member_dt, float* T_seq, int nslots, int first_step, int n_steps, double* dt_seq,
                            int dt_seq_rows, float* u, float* v, float* p, float* V, void* workspace, size_t workspace_bytes, int B, int H,
                            int W, void* stream) {
  const ClockArgs none = {nullptr, nullptr, nullptr, nullptr, 0};
  return rollout_impl(ctx, net, members, xc, yc, ycc, xcoef, ycoef, dx_min, cn_max, per_member_dt, T_seq, nslots, first_step,
                      n_steps, dt_seq, dt_seq_rows, u, v, p, V, workspace, workspace_bytes, B, H, W, none, nullptr, nullptr,
                      nullptr, stream);
}

// the refusals of a clocked rollout, shared by pbmc_rollout_clocked and pbmc_rollout_queued
static int validate_clock(const pbmc_member_clock* clock, const double* dt_seq, const double* meanT_seq, const float* snap_ring,
                          const double* snap_meta, int snap_slots, int per_member_dt, int B) {
  if (!clock || !dt_seq || !meanT_seq || !snap_ring || !snap_meta) return PBMC_ERR_NULL_POINTER;
  if (snap_slots < 1) return PBMC_ERR_BAD_SHAPE;
  if (!per_member_dt && B > 1) return PBMC_ERR_UNSUPPORTED;  // a frozen member would still set the others' batch-global dt
  return PBMC_OK;
}

extern "C" int pbmc_rollout_clocked(pbmc_ctx* ctx, const pbmc_net* net, const pbmc_member* members, const float* xc,
                                    const float* yc, const float* ycc, const float* xcoef, const float* ycoef, double dx_min,
                                    double cn_max, int per_member_dt, float* T_seq, int nslots, int first_step, int n_steps,
                                    double* dt_seq, int dt_seq_rows, float* u, float* v, float* p, float* V, void* workspace,
                                    size_t workspace_bytes, int B, int H, int W, pbmc_member_clock* clock, double* meanT_seq,
                                    float* snap_ring, double* snap_meta, int snap_slots, void* stream) {
  RC(validate_clock(clock, dt_seq, meanT_seq, snap_ring, snap_meta, snap_slots, per_member_dt, B));
  const ClockArgs clk = {clock, meanT_seq, snap_ring, snap_meta, snap_slots};
  return rollout_impl(ctx, net, members, xc, yc, ycc, xcoef, ycoef, dx_min, cn_max, per_member_dt, T_seq, nslots, first_step,
                      n_steps, dt_seq, dt_seq_rows, u, v, p, V, workspace, workspace_bytes, B, H, W, clk, nullptr, nullptr,
                      nullptr, stream);
}

// the refusals of a member queue, shared by pbmc_rollout_queued, pbmc_rollout_diagnosed and pbmc_rollout_chained
static int validate_queue(const pbmc_member_queue* queue, int B) {
  if (!queue) return PBMC_ERR_NULL_POINTER;
  const pbmc_member_queue& q = *queue;
  if (!q.T0 || !q.params || !q.t0 || !q.t_end || !q.save_every || !q.n_step0 || !q.max_steps || !q.next || !q.slot_member ||
      !q.member_seq || !q.snap_member)
    return PBMC_ERR_NULL_POINTER;
  if (q.Q < 1) return PBMC_ERR_BAD_SHAPE;
  if (!aligned16(q.T0)) return PBMC_ERR_MISALIGNED;  // the refill copies T0 rows with 16-byte loads
  if ((size_t)B * sizeof(int) > 48 * 1024) return PBMC_ERR_UNSUPPORTED;  // the commit kernel's [B] stop flags in shared memory
  return PBMC_OK;
}

extern "C" int pbmc_rollout_queued(pbmc_ctx* ctx, const pbmc_net* net, pbmc_member* members, const float* xc, const float* yc,
                                   const float* ycc, const float* xcoef, const float* ycoef, double dx_min, double cn_max,
                                   int per_member_dt, float* T_seq, int nslots, int first_step, int n_steps, double* dt_seq,
                                   int dt_seq_rows, float* u, float* v, float* p, float* V, void* workspace,
                                   size_t workspace_bytes, int B, int H, int W, pbmc_member_clock* clock, double* meanT_seq,
                                   float* snap_ring, double* snap_meta, int snap_slots, const pbmc_member_queue* queue,
                                   void* stream) {
  RC(validate_clock(clock, dt_seq, meanT_seq, snap_ring, snap_meta, snap_slots, per_member_dt, B));
  RC(validate_queue(queue, B));
  const ClockArgs clk = {clock, meanT_seq, snap_ring, snap_meta, snap_slots};
  return rollout_impl(ctx, net, members, xc, yc, ycc, xcoef, ycoef, dx_min, cn_max, per_member_dt, T_seq, nslots, first_step,
                      n_steps, dt_seq, dt_seq_rows, u, v, p, V, workspace, workspace_bytes, B, H, W, clk, queue, nullptr,
                      nullptr, stream);
}

// the refusals of a diagnostics descriptor, shared by pbmc_rollout_diagnosed and pbmc_rollout_chained
static int validate_diag(const pbmc_diag_desc& d, int H, int W) {
  if (!d.flux_seq || !d.vrms_seq || !d.steady || !d.part) return PBMC_ERR_NULL_POINTER;
  if (d.window < 0 || d.window > PBMC_STEADY_MAX_WINDOW) return PBMC_ERR_BAD_SHAPE;
  if (d.window > 0 && (!d.hist || !d.hist_n)) return PBMC_ERR_NULL_POINTER;
  if (!(d.rtol >= 0.0) || !std::isfinite(d.rtol)) return PBMC_ERR_BAD_SHAPE;  // NaN fails the first test
  if (H < 3 || W < 3) return PBMC_ERR_BAD_SHAPE;  // vrms averages over the interior cells
  return PBMC_OK;
}

extern "C" int pbmc_rollout_diagnosed(pbmc_ctx* ctx, const pbmc_net* net, pbmc_member* members, const float* xc,
                                      const float* yc, const float* ycc, const float* xcoef, const float* ycoef, double dx_min,
                                      double cn_max, int per_member_dt, float* T_seq, int nslots, int first_step, int n_steps,
                                      double* dt_seq, int dt_seq_rows, float* u, float* v, float* p, float* V, void* workspace,
                                      size_t workspace_bytes, int B, int H, int W, pbmc_member_clock* clock, double* meanT_seq,
                                      float* snap_ring, double* snap_meta, int snap_slots, const pbmc_member_queue* queue,
                                      const pbmc_diag_desc* diag, void* stream) {
  RC(validate_clock(clock, dt_seq, meanT_seq, snap_ring, snap_meta, snap_slots, per_member_dt, B));
  if (queue) RC(validate_queue(queue, B));
  if (!diag) return PBMC_ERR_NULL_POINTER;
  RC(validate_diag(*diag, H, W));
  const ClockArgs clk = {clock, meanT_seq, snap_ring, snap_meta, snap_slots};
  return rollout_impl(ctx, net, members, xc, yc, ycc, xcoef, ycoef, dx_min, cn_max, per_member_dt, T_seq, nslots, first_step,
                      n_steps, dt_seq, dt_seq_rows, u, v, p, V, workspace, workspace_bytes, B, H, W, clk, queue, diag, nullptr,
                      stream);
}

extern "C" int pbmc_rollout_chained(pbmc_ctx* ctx, const pbmc_net* net, pbmc_member* members, const float* xc,
                                    const float* yc, const float* ycc, const float* xcoef, const float* ycoef, double dx_min,
                                    double cn_max, int per_member_dt, float* T_seq, int nslots, int first_step, int n_steps,
                                    double* dt_seq, int dt_seq_rows, float* u, float* v, float* p, float* V, void* workspace,
                                    size_t workspace_bytes, int B, int H, int W, pbmc_member_clock* clock, double* meanT_seq,
                                    float* snap_ring, double* snap_meta, int snap_slots, const pbmc_member_queue* queue,
                                    const pbmc_diag_desc* diag, const pbmc_member_chain* chain, void* stream) {
  RC(validate_clock(clock, dt_seq, meanT_seq, snap_ring, snap_meta, snap_slots, per_member_dt, B));
  RC(validate_queue(queue, B));
  if (diag) RC(validate_diag(*diag, H, W));
  if (!chain || !chain->heads || !chain->succ) return PBMC_ERR_NULL_POINTER;
  if (chain->K < 1 || chain->K > queue->Q) return PBMC_ERR_BAD_SHAPE;
  const ClockArgs clk = {clock, meanT_seq, snap_ring, snap_meta, snap_slots};
  return rollout_impl(ctx, net, members, xc, yc, ycc, xcoef, ycoef, dx_min, cn_max, per_member_dt, T_seq, nslots, first_step,
                      n_steps, dt_seq, dt_seq_rows, u, v, p, V, workspace, workspace_bytes, B, H, W, clk, queue, diag, chain,
                      stream);
}
