/*
 * pbmc.h -- C ABI of libpbmc.so: the B200 (sm_100a) kernels behind the surrogate
 * time-stepping hot path of agsiddhant/PBML_Mantle_Convection.
 *
 * The reference has NO native interface for this path (it is pure PyTorch; SURVEY.md
 * section 2 "Native components: none"), so every entry point below replaces a group of
 * ATen/cuDNN library calls made by the reference's Python.  Each declaration cites the
 * reference lines (relative to the reference repo root) whose arithmetic it implements.
 *
 * Conventions
 *   - plain pointers + sizes; no torch types.  All pointers are DEVICE pointers unless
 *     the name ends in _h.  The caller owns every buffer (outputs, workspace).
 *   - every function only ENQUEUES work on `stream` (a cudaStream_t passed as void*);
 *     no host synchronisation, no allocation => capturable in a CUDA graph.
 *   - return value: 0 = ok, negative = pbmc_status.  There is no CPU fallback.
 *   - activation layout ("blocked"): float [B][CB][H][W][4], CB = ceil(C/4), channel
 *     c lives at block c/4, lane c%4; unused lanes are zero.  Field layout ("plain"):
 *     float [B][H][W].
 */
#ifndef PBMC_H_
#define PBMC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PBMC_VERSION 3
#define PBMC_MAX_SRC 8
#define PBMC_MAX_LEVELS 8
#define PBMC_MAX_REPEATS 8

typedef enum {
  PBMC_OK = 0,
  PBMC_ERR_BAD_SHAPE = -1,
  PBMC_ERR_UNSUPPORTED = -2,
  PBMC_ERR_NULL_POINTER = -3,
  PBMC_ERR_MISALIGNED = -4,
  PBMC_ERR_WORKSPACE = -5,
  PBMC_ERR_CUDA = -6,
  PBMC_ERR_NOT_DEVICE_POINTER = -7
} pbmc_status;

enum { PBMC_PAD_ZEROS = 0, PBMC_PAD_REPLICATE = 1, PBMC_PAD_REFLECT = 2 };
enum { PBMC_XFORM_NONE = 0, PBMC_XFORM_GN_GELU = 1, PBMC_XFORM_GN = 2, PBMC_XFORM_GELU = 3 };
enum { PBMC_ACT_NONE = 0, PBMC_ACT_GELU = 1 };
/* Source layouts.  BLOCKED: float [B][nblk][H][W][4].  STAGED16: the tensor-core operand image of a 16-channel
 * tensor, ready to be copied into shared memory by the TMA engine with no thread touching it:
 *   __half [B][H][part = hi, lo][chunk = channels 0-7, 8-15][Wp][8],  Wp = pbmc_staged_width(W) = roundup(W,128) + 2,
 * position 0 / W+1 = the replicate-padded columns -1 / W, hi + lo = the fp32 value split into two fp16
 * (the split the row conv kernel's producer warps would compute).  Accepted by pbmc_conv_fwd for 3x3, replicate
 * padding, xform NONE, nblk = 4, on the ROW_F16X2 kernel (AUTO picks it). */
enum { PBMC_LAYOUT_BLOCKED = 0, PBMC_LAYOUT_STAGED16 = 1 };
enum { PBMC_HEAD_CURL = 0, PBMC_HEAD_MAE = 1 };
/* pbmc_net.flags: PER_LAYER = never use the persistent trunk kernel; UP_STAGED = the bicubic kernel writes the up-sampled
 * levels as conv[1]'s fp16 hi|lo operand image (PBMC_LAYOUT_STAGED16) and conv[1] stages them with TMA bulk copies
 * (bit-identical results; measured neutral-to-slower, so off by default); LEARNED = every conv is the learned 9-region
 * convolution (r_p = "learned", see pbmc_net) */
enum { PBMC_NET_TRUNK_PER_LAYER = 1, PBMC_NET_UP_STAGED = 2, PBMC_NET_TRUNK_BULK_LOADER = 4, PBMC_NET_LEARNED = 8 };
/* pbmc_trunk_desc.loader: THREADS (default) = every worker loads its own pixels with ld.global.cg; BULK = TMA bulk copies
 * (cp.async.bulk + mbarrier transaction bytes): all raw rows of a layer are requested up front by one warp, land in the
 * stage slot their operand image will occupy and are converted in place.  Same results; measured SLOWER on B200 (77.9 vs
 * 67.6 us per 4-layer launch at 512^2: the extra shared-memory loads and the per-row group barrier cost more than the
 * hidden global-load latency gains), so it is opt-in. */
enum { PBMC_TRUNK_LOADER_THREADS = 0, PBMC_TRUNK_LOADER_BULK = 1 };
/* conv implementation selector: FFMA = fp32 CUDA cores; UMMA_* = tcgen05 tensor cores:
 * 3XTF32 / F16X2 split every operand into hi + lo (tf32 resp. fp16) and issue 3 passes --
 * fp32-grade accuracy; BF16 = single pass with bf16 operands (looser, stated bound).
 * ROW_* = the row-streaming warp-specialised tcgen05 kernel (csrc/conv_row.cu; vertical taps folded
 * into the MMA's N dimension), F16X2 = fp16 hi+lo 3-pass (fp32-grade), BF16 = single bf16 pass.
 * MUX_* = the time-multiplexed row kernel (csrc/conv_mux.cu: the same GEMM, all warps stage rows, then all
 * warps run the epilogue) for single-source 3x3 convs with c_in, c_out <= 16; other shapes asked for with
 * MUX_* run the ROW_* kernel of the same precision.
 * AUTO = MUX_F16X2 where the shape is supported and the grid fits one wave, else ROW_F16X2, else UMMA_F16X2, else FFMA. */
enum { PBMC_CONV_AUTO = 0, PBMC_CONV_FFMA = 1, PBMC_CONV_UMMA_3XTF32 = 2, PBMC_CONV_UMMA_BF16 = 3, PBMC_CONV_UMMA_F16X2 = 4,
       PBMC_CONV_ROW_F16X2 = 5, PBMC_CONV_ROW_BF16 = 6, PBMC_CONV_MUX_F16X2 = 7, PBMC_CONV_MUX_BF16 = 8 };

const char* pbmc_error_string(int status);
int pbmc_version(void);
/* struct sizes, so a foreign-language binding can assert its mirror declarations */
size_t pbmc_sizeof(const char* struct_name);
/* last CUDA error text recorded by this library on the calling thread ("" if none) */
const char* pbmc_last_cuda_error(void);

/* ------------------------------------------------------------------ per-run parameters
 * One per ensemble member (device array of B).  Values are what the reference derives on
 * the host at advect_wi_gaia.py:443-460 and pytorch_networks_convae.py:343-350. */
typedef struct {
  float raq_nd, fkt_nd, fkp_nd; /* normalised inputs, advect_wi_gaia.py:446-450 */
  float ln_fkt, ln_fkp;         /* log(gamma), log(beta), pytorch_networks_convae.py:337 */
  float raq;                    /* internal heating term RaQ, :459 / :562 */
  float scaler;                 /* velocity de-normalisation, :343-350 */
  float reserved;
} pbmc_member;

/* ------------------------------------------------------------------ layout conversion
 * NCHW float <-> blocked.  Replaces nothing in the reference (it is NCHW throughout);
 * needed so the module-level API (NewFluidNet.forward(inputs[B,c_i,H,W])) is drop-in. */
int pbmc_pack_nchw(const float* src_nchw, float* dst_blocked, int B, int C, int H, int W, void* stream);
int pbmc_unpack_nchw(const float* src_blocked, float* dst_nchw, int B, int C, int H, int W, void* stream);

/* ------------------------------------------------------------------ A1: network input
 * TS.forward input build, pytorch_networks_convae.py:379-407 (eta_torch :86-102):
 *   V = clip(exp(ln_fkt*(0-T) + ln_fkp*(1-ycc)), 1e-8, 1)
 *   channels = [x/4, y/4, log10(V)/8, raq_nd, fkt_nd, fkp_nd, T] (+1 zero lane) -> blocked [B][2][H][W][4]
 * xc/yc/ycc are [H][W] fields shared by the batch.  V_out (plain [B][H][W]) may be NULL. */
int pbmc_build_input(const float* T, const float* xc, const float* yc, const float* ycc, const pbmc_member* members,
                     float* inp_blocked, float* V_out, int B, int H, int W, void* stream);

/* ------------------------------------------------------------------ A2/A3/A6: convolution
 * One conv "source" = a blocked tensor contributing nblk channel blocks, with the
 * producer's GroupNorm (+GELU) applied while the tile is loaded:
 *   FluidLayer.forward conv -> GroupNorm -> GELU, pytorch_networks_convae.py:790-799,
 *   GroupNorm(C/4 groups) :788 / :1279  (one group == one channel block),
 *   channel concat :1327/:1332 == several sources (never materialised). */
typedef struct {
  const float* ptr;    /* [B][nblk][H][W][4] */
  const double* stats; /* [B][nblk][2] = (sum, sum of squares) of the RAW tensor per (b, group); NULL if xform==NONE */
  const float* gamma;  /* [nblk*4] GroupNorm weight (NULL if xform==NONE) */
  const float* beta;   /* [nblk*4] GroupNorm bias */
  int nblk;
  int xform;           /* PBMC_XFORM_* */
  double inv_count;    /* 1 / (channels_per_group * H * W) */
  int layout;          /* PBMC_LAYOUT_*: BLOCKED (default) or STAGED16 (see pbmc_bicubic_up_staged) */
  int reserved;
} pbmc_src;

/* k x k, stride 1, 'same' conv (k in {3,5}) over the concatenation of `nsrc` sources.
 *   SymmetricConv2d.forward  symmetric_layers_torch.py:113-138 (mirrored filters are expanded once at pack time)
 *   nn.Conv2d heads          pytorch_networks_convae.py:1263-1309
 *   padding_mode             zeros / replicate / reflect, folded into the tile load
 * Epilogue: + bias, optional GELU (:1339-1340), raw output, and per-(b, block) sum / sum^2
 * accumulated into out_stats (double, must be zeroed by the caller) for the next GroupNorm,
 * or per-channel sums for the zero-mean at :1343 (out_chan_sum, [B][cout_blks*4] doubles).
 * Packed weights: float [ceil(cout/16)][cin_blks][k*k][4][16]  (see pbmc_pack helpers in Python). */
typedef struct {
  pbmc_src src[PBMC_MAX_SRC];
  int nsrc;
  int B, H, W;
  int cout;     /* real output channels */
  int ksize;    /* 3 or 5 */
  int pad_mode; /* PBMC_PAD_* */
  int epi_act;  /* PBMC_ACT_* */
  int impl;     /* PBMC_CONV_* */
  int max_ctas; /* 0 = fill the GPU; > 0: use at most this many CTAs (several convs sharing the GPU on different streams) */
  const float* wpk;
  const void* wpk_umma;  /* tensor-core operand image of the same weights (NULL => FFMA only) */
  const void* wpk_row;   /* operand image for the row-streaming tensor-core kernel (NULL => not available) */
  const float* bias;     /* [ceil(cout/4)*4], zero padded */
  float* out;            /* [B][ceil(cout/4)][H][W][4] */
  double* out_stats;     /* [B][ceil(cout/4)][2] or NULL */
  double* out_chan_sum;  /* [B][ceil(cout/4)*4] or NULL */
} pbmc_conv_desc;

int pbmc_conv_fwd(const pbmc_conv_desc* desc_h, void* stream);

/* ------------------------------------------------------------------ A4: learned 9-region boundary convolution
 * BoundaryLearnedConvolution2D.forward pytorch_networks_convae.py:1022-1065 (bc_x = bc_y = 1) in TWO launches:
 *   1. pbmc_conv_fwd with the INTERIOR filters (`conv`), bias = learnable_bias, any padding mode (zeros is cheapest),
 *      over the whole image: correct wherever the k x k window stays inside the image;
 *   2. pbmc_conv_edge9 overwrites the ring of width (k-1)/2 with the eight edge / corner regions -- per pixel ONE k x k
 *      window whose position and filter set follow from its row / column class, the reference's row swap included
 *      (the strip computed from the LAST input rows is output row 0, :1060) -- and repairs out_stats / out_chan_sum
 *      (subtracts what launch 1 accumulated for the ring pixels, adds the new values).
 * Same sources (concat order, fused producer transforms), same `out` / statistics buffers in both calls.
 *   wedge  float [8][cin_blks][k*k][16][4]: region (top_left, top_right, bottom_left, bottom_right, top, bottom, left,
 *          right -- the reference's names), input-channel block of the concatenation, tap dy*k+dx, c_out, c_in % 4;
 *          zero padded (ops.pack_edge9_weights).  c_out <= 16, every source <= 128 channels. */
typedef struct {
  pbmc_src src[PBMC_MAX_SRC];
  int nsrc;
  int B, H, W;
  int cout, ksize, epi_act, reserved;
  const float* wedge;
  const float* bias;      /* [16] learnable_bias, zero padded */
  float* out;             /* [B][ceil(cout/4)][H][W][4], written by pbmc_conv_fwd before this call */
  double* out_stats;      /* as passed to pbmc_conv_fwd, or NULL */
  double* out_chan_sum;   /* as passed to pbmc_conv_fwd, or NULL */
} pbmc_edge9_desc;
int pbmc_conv_edge9(const pbmc_edge9_desc* desc_h, void* stream);

/* blocked -> NCHW with the producer's GroupNorm(+GELU) applied: the tail of a stand-alone
 * FluidLayer.forward (pytorch_networks_convae.py:796-797). */
int pbmc_finalize_nchw(const pbmc_src* src_h, float* dst_nchw, int B, int C, int H, int W, void* stream);

/* ------------------------------------------------------------------ A5: pyramid
 * AvgPool2d(2,2) with floor (pytorch_networks_convae.py:1225, :1321-1322), source transform fused. */
int pbmc_avgpool2(const pbmc_src* src_h, float* dst, int B, int H, int W, void* stream);
/* nn.Upsample(size=(H,W), mode="bicubic"), align_corners=False, A=-0.75 (:1227-1229, :1326),
 * source transform (GroupNorm+GELU of the level's last FluidLayer) fused. */
int pbmc_bicubic_up(const pbmc_src* src_h, float* dst, int B, int Hs, int Ws, int H, int W, void* stream);
/* Same, written in PBMC_LAYOUT_STAGED16 (src nblk must be 4): the up-sampled levels are read only by conv[1]
 * (:1332-1335), whose operand loader is then a bulk copy.  dst: pbmc_staged_bytes(B, H, W) bytes. */
int pbmc_bicubic_up_staged(const pbmc_src* src_h, void* dst, int B, int Hs, int Ws, int H, int W, void* stream);
int pbmc_staged_width(int W);
size_t pbmc_staged_bytes(int B, int H, int W);

/* ------------------------------------------------------------------ A7: head
 * zero-mean (:1343), curl (:1357-1370), replicate pad + wall BCs (:1372-1386),
 * velocity un-scaling (TS.__unscale_var :341-352, :411-412), and max|u|,|v| over the
 * interior (ADNet :524-525,:556) in the same pass.
 *   y      blocked [B][1][H][W][4] raw conv[3] output;  chan_sum [B][4] doubles
 *   u,v,p  plain [B][H][W] (p may be NULL);  uvmax [B] float bits (must be zeroed) */
int pbmc_head(const float* y, const double* chan_sum, const pbmc_member* members, float a_bound, int head_kind,
              int p_pred, float* u, float* v, float* p, uint32_t* uvmax, int B, int H, int W, void* stream);

/* ------------------------------------------------------------------ A8/A9: advection-diffusion
 * ADNet.forward pytorch_networks_convae.py:522-568 + TS boundary rows/cols :468-471, one pass:
 * upwind advection (:547-548), non-uniform central diffusion (:550-552), RaQ source,
 * dt = min(CN/2 * dx_min / max|u,v|, dx_min^2/4) (:554-559) read from uvmax_in, and
 * max|u|,|v| of the interior written to uvmax_out (may alias nothing; zeroed by caller; may be NULL).
 *   xcoef [3][W], ycoef [3][H]: inverse spacings of the separable grid from pbmc_stencil_coefs
 *   (1/d_minus, 1/d_plus, 1/(0.5 d_plus + 0.5 d_minus); wall coordinates forced to 0/4 and 0/1, :532-545)
 *   uvmax_in: [B] float bits (member_stride=1) or a single batch-global value (member_stride=0, ADNet semantics :556)
 *   dt_fixed: if > 0 it is used instead of the CFL value (ADNet's dt argument)
 *   dt_out:   [B] doubles, may be NULL */
int pbmc_stencil_coefs(const double* coord, int n, double wall_lo, double wall_hi, float* coef, void* stream);
int pbmc_advect_diffuse(const float* T, const float* u, const float* v, const float* xcoef, const float* ycoef,
                        const pbmc_member* members, const uint32_t* uvmax_in, int member_stride, double dx_min,
                        double cn_max, double dt_fixed, float* T_out, uint32_t* uvmax_out, double* dt_out, int B, int H,
                        int W, void* stream);
/* Row-slab form for a grid decomposed over several GPUs (new: the reference is single-device, SURVEY.md 8e).
 * T, u, v, T_out are the LOCAL [H][W] arrays of one rank, ghost rows included: has_up / has_down say that local
 * row 0 / H-1 is a ghost row (a neighbour's row) instead of a wall; ghost rows are read, never written.
 * ycoef [3][H] must be the slice of the GLOBAL coefficients.  If peer_*_ghost_row is non-NULL the first / last
 * OWNED row of T_out is additionally stored there -- a pointer into the neighbour rank's T_out ghost row
 * (peer memory over NVLink): the halo exchange is fused into the update, no send/recv follows.  The caller
 * orders steps across ranks (the per-step dt all-reduce does).  Needs W % 4 == 0 and 16-byte aligned rows. */
int pbmc_advect_diffuse_slab(const float* T, const float* u, const float* v, const float* xcoef, const float* ycoef,
                             const pbmc_member* members, const uint32_t* uvmax_in, double dx_min, double cn_max,
                             double dt_fixed, float* T_out, uint32_t* uvmax_out, double* dt_out, int H, int W, int has_up,
                             int has_down, float* peer_up_ghost_row, float* peer_down_ghost_row, void* stream);
/* Flag-synchronised slab step: the halo exchange AND the global dt reduction happen inside the update kernel, so a time
 * step of a decomposed grid is ONE kernel launch per rank and no collective call (the reference is single-device; this
 * replaces what would be ncclAllReduce(max) + ncclSend/Recv per step, SURVEY.md 8b "halo_exchange / dt_allreduce").
 * Every rank owns one pbmc_slab_sync block in memory ALL ranks can write (CUDA IPC / symmetric memory over NVLink),
 * zero-initialised; peers_h is a HOST array of the `world` blocks' addresses as mapped into this device (own included).
 *   slot[par][r] = (step tag << 32) | float bits of rank r's max|u|,|v| over its owned interior rows
 *   steps_done / ctas_done / local_max: private to the owning rank's kernels
 * Protocol (step s = steps_done + 1): the kernel waits (ld.acquire.sys) until all `world` slots of parity s & 1 carry
 * tag s, takes their max -> dt (pytorch_networks_convae.py:554-559: ONE scalar for the whole grid); stores its
 * boundary rows into the neighbours' ghost rows; the CTA that finishes last publishes (s + 1, local max) into every
 * rank's slot of parity (s + 1) & 1 with st.release.sys and sets steps_done = s.  pbmc_slab_sync_publish makes the
 * first publication of a run (tag steps_done + 1) from u, v; call it again -- after a host-side barrier and with the
 * blocks re-zeroed -- whenever the velocity field changes.  If a peer stays silent for 10 s the kernel records it in
 * `failed` and goes on; the host must check `failed` when it synchronises.
 * Ranks must run on DIFFERENT devices (or be launched strictly one after the other on one stream, as the
 * single-GPU tests do): a kernel that waits for a peer's kernel must never share a GPU with it. */
#define PBMC_MAX_RANKS 16
typedef struct {
  unsigned long long slot[2][PBMC_MAX_RANKS];
  unsigned int steps_done, ctas_done, local_max;
  unsigned int failed; /* 0, or 0x80000000 | (bit r: rank r's publication did not arrive within 10 s); checked by the host */
} pbmc_slab_sync;
int pbmc_slab_sync_publish(const float* u, const float* v, int H, int W, pbmc_slab_sync* self,
                           pbmc_slab_sync* const* peers_h, int rank, int world, void* stream);
int pbmc_advect_diffuse_slab_sync(const float* T, const float* u, const float* v, const float* xcoef, const float* ycoef,
                                  const pbmc_member* members, double dx_min, double cn_max, float* T_out, double* dt_out,
                                  int H, int W, int has_up, int has_down, float* peer_up_ghost_row,
                                  float* peer_down_ghost_row, pbmc_slab_sync* self, pbmc_slab_sync* const* peers_h,
                                  int rank, int world, void* stream);
/* max|u|,|v| over the interior as a stand-alone reduction (only needed when nothing upstream produced it) */
int pbmc_uvmax(const float* u, const float* v, uint32_t* uvmax, int member_stride, int B, int H, int W, void* stream);
/* general form, exactly ADNet's inputs tensor: xc, yc as [H][W] fields (coord_batch_stride = 0) or
 * per-sample fields (= H*W), RaQ as an optional [B][H][W] field (NULL: members[b].raq), and
 * dx_min read from device memory (double) so the module-level ADNet.forward needs no host sync. */
int pbmc_advect_diffuse_fields(const float* T, const float* u, const float* v, const double* xc, const double* yc,
                               size_t coord_batch_stride, const float* raq_field, const pbmc_member* members,
                               const uint32_t* uvmax_in, int member_stride, const double* dx_min_dev, double cn_max,
                               const double* dt_fixed_dev, float* T_out, double* dt_out, int B, int H, int W,
                               void* stream);

/* ------------------------------------------------------------------ A10: driver clamp
 * advect_wi_gaia.py:624-629: wall rows, side columns, clip(T, 0, 2) */
int pbmc_clamp_T(float* T, int core_cool, int B, int H, int W, void* stream);

/* ------------------------------------------------------------------ A11: diagnostics
 * mean-T (advect_wi_gaia.py:547,647) and horizontal-mean profile
 * (.ipynb_checkpoints/load_advection_results-checkpoint.ipynb:322); doubles.
 *   prof [B][H] (row means), meanT [B] */
int pbmc_diagnostics(const float* T, double* prof, double* meanT, int B, int H, int W, void* stream);

/* ------------------------------------------------------------------ whole surrogate + rollout
 * NewFluidNet.forward pytorch_networks_convae.py:1315-1388 and TS.forward's loop :377-475,
 * enqueued as one DAG over a few internal streams (pyramid levels are independent). */
typedef struct {
  const float* wpk;
  const void* wpk_umma;
  const void* wpk_row;
  const float* bias;
  const float* gamma; /* GroupNorm affine applied to THIS layer's output by its consumers (NULL: none) */
  const float* beta;
  int cin_blks, cout, ksize, reserved;
} pbmc_layer;

typedef struct {
  int levels, repeats, c_i, c_h, c_o, ksize, pad_mode, head_kind, p_pred, conv_impl;
  float a_bound;
  int flags; /* PBMC_NET_*: 0 = defaults (the R layers of a level as one persistent launch where every level's grid can be
                resident at once -- pbmc_trunk_fwd -- else one launch per layer; up-sampled levels as blocked fp32) */
  pbmc_layer conv0;
  pbmc_layer trunk[PBMC_MAX_LEVELS * PBMC_MAX_REPEATS]; /* [level][repeat] */
  pbmc_layer conv1, conv2, conv3;
  /* flags & PBMC_NET_LEARNED only (NULL otherwise): the eight edge / corner filter sets of each layer in the wedge layout
   * of pbmc_conv_edge9 (ops.pack_edge9_weights).  The layer's wpk / wpk_umma / wpk_row then hold the INTERIOR filters and
   * its bias the learnable_bias. */
  const float* wedge_conv0;
  const float* wedge_trunk[PBMC_MAX_LEVELS * PBMC_MAX_REPEATS]; /* [level][repeat] */
  const float* wedge_conv1;
  const float* wedge_conv2;
  const float* wedge_conv3;
} pbmc_net;

/* ------------------------------------------------------------------ A3/A5: the R FluidLayers of one pyramid level, ONE launch
 * NewFluidNet.forward pytorch_networks_convae.py:1323-1324 (`for r in range(R): y1 = convs[l][r](y1)`), FluidLayer :790-799.
 * Persistent kernel (csrc/conv_trunk.cu): a CTA keeps its strip, TMEM and barriers for all R layers; GroupNorm's
 * whole-image reduction between two layers is a grid-wide arrive/poll counter.  16 hidden channels, 3x3.
 *   src0    the level's input (xform NONE, or GN_GELU of its producer)
 *   layers  HOST array [R]: wpk_row, bias and the GroupNorm affine (gamma, beta) of each layer's OUTPUT
 *   ping    layer r writes its raw output to ping[r & 1]  -> the level's result is ping[(R-1) & 1], to be read with
 *           GN_GELU(stats + (R-1)*B*8, layers[R-1].gamma/beta) by its consumers
 *   stats   [R][B][4][2] doubles, sync [B] unsigned: scratch, zeroed by the call unless pre_zeroed != 0
 *   max_ctas  CTA budget (0 = 148): the WHOLE grid must be resident at once, PBMC_ERR_UNSUPPORTED if it cannot be
 *           (the caller then runs the layers one by one with pbmc_conv_fwd) */
typedef struct {
  pbmc_src src0;
  const pbmc_layer* layers;
  float* ping[2];
  double* stats;
  unsigned int* sync;
  int R, B, H, W, pad_mode, impl, max_ctas, pre_zeroed;
  int loader;   /* PBMC_TRUNK_LOADER_*: how the raw input rows reach shared memory (fp16 hi+lo kernel; bf16 always THREADS) */
  int reserved;
} pbmc_trunk_desc;
int pbmc_trunk_fwd(const pbmc_trunk_desc* desc_h, void* stream);
/* 1 if pbmc_trunk_fwd would take this configuration (shape, budget), else 0 */
int pbmc_trunk_supported(const pbmc_trunk_desc* desc_h);

typedef struct pbmc_ctx pbmc_ctx; /* internal streams + events only; owns no tensor memory */
int pbmc_ctx_create(pbmc_ctx** out);
int pbmc_ctx_destroy(pbmc_ctx* ctx);

size_t pbmc_workspace_bytes(const pbmc_net* net_h, int B, int H, int W);
/* How a forward of this network at this size shares the 148 SMs between the pyramid levels (NewFluidNet.forward's trunk,
 * pytorch_networks_convae.py:1319-1327, runs the levels side by side): budgets[l] = CTAs of level l's conv kernels
 * (PBMC_MAX_LEVELS entries; 0 = no budget, the level's launches run in waves).  Returns 1 when the trunk runs as persistent
 * kernels (one launch per level: every level has a budget and the budgets fit the GPU), 0 when it runs one launch per layer,
 * < 0 on error.  Pure host computation: no GPU needed. */
int pbmc_trunk_cta_budgets(const pbmc_net* net_h, int B, int H, int W, int* budgets);

/* Learned-boundary networks (flags & PBMC_NET_LEARNED; r_p = "learned", every conv a BoundaryLearnedConvolution2D,
 * pytorch_networks_convae.py:1022-1065, bc_x = bc_y = 1): every layer of the DAG is two launches on the same stream -- the
 * interior filters through the conv kernels with zeros padding (pad_mode is not used), then the ring kernel of
 * pbmc_conv_edge9 with the same sources, output and statistics.  The trunk always runs one launch per layer (the persistent
 * kernel would consume each layer's GroupNorm statistics before the ring kernel repairs them) and the up-sampled levels stay
 * blocked fp32 (PBMC_NET_UP_STAGED is ignored).  Supported when c_h <= 16, c_o <= 4, every source <= 128 channels and every
 * pyramid level holds the reference's boundary strips (at least k rows and columns for k = 3, k + 1 for k = 5); otherwise
 * pbmc_workspace_bytes returns 0 and pbmc_surrogate_forward / pbmc_rollout / pbmc_trunk_cta_budgets PBMC_ERR_UNSUPPORTED. */
/* inp: blocked [B][ceil(c_i/4)][H][W][4] network input (A1's output, or a packed user tensor).
 * u,v,p plain [B][H][W] (mae head with p_pred: p too).  members may be NULL => scaler 1
 * (module-level NewFluidNet.forward does not un-scale).  uvmax may be NULL. */
int pbmc_surrogate_forward(pbmc_ctx* ctx, const pbmc_net* net_h, const float* inp, const pbmc_member* members, float* u,
                           float* v, float* p, uint32_t* uvmax, void* workspace, size_t workspace_bytes, int B, int H,
                           int W, void* stream);

/* n_steps of: build input -> surrogate -> un-scale -> advect/diffuse -> BCs.
 *   T_seq: [nslots][B][H][W]; step i reads slot (i-1)%nslots and writes slot i%nslots (i = first_step .. first_step+n_steps-1)
 *   dt_seq: [dt_seq_rows][B] doubles, entry i-1 written by step i (may be NULL); dt_seq_rows >= first_step + n_steps - 1
 *           is checked (PBMC_ERR_BAD_SHAPE), so a chunked caller cannot write past its history buffer
 *   per_member_dt: 1 = each member has its own CFL dt (independent rollouts); 0 = ADNet's batch-global dt (:556)
 *   u,v,p,V: plain [B][H][W] buffers holding the LAST step's fields (V may be NULL) */
int pbmc_rollout(pbmc_ctx* ctx, const pbmc_net* net_h, const pbmc_member* members, const float* xc, const float* yc,
                 const float* ycc, const float* xcoef, const float* ycoef, double dx_min, double cn_max, int per_member_dt, float* T_seq,
                 int nslots, int first_step, int n_steps, double* dt_seq, int dt_seq_rows, float* u, float* v, float* p, float* V,
                 void* workspace, size_t workspace_bytes, int B, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PBMC_H_ */
