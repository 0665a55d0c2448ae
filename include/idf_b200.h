/* idf_b200 -- C ABI of the B200-native InfoDiffusion denoising hot path.
 *
 * The reference (isjakewong/InfoDiffusion) has no FFI: its boundary is the Python nn.Module
 * call surface (SURVEY.md section 8b).  Every entry point below therefore names the reference
 * Python construct whose arithmetic it replaces (file:line in the reference checkout).  The
 * host-side mirror of the reference interface (infodiffusion_b200/{models,modules,sampling,utils}.py)
 * binds these symbols with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *  - plain pointers + sizes, no torch types; all pointers are DEVICE pointers unless stated.
 *  - every launcher is asynchronous on `stream`, allocates nothing, keeps no global state
 *    besides the plan objects the caller owns, and is CUDA-graph capturable.
 *  - return value: 0 on success, negative idf_status on error; idf_last_error() gives text.
 *  - reductions whose order depends on arrival (split-K weight gradients, bias / GroupNorm-affine gradients, split-K
 *    fp32 GEMM, MMD) have ORDERED variants: partials go to a caller-owned fp32 workspace and are combined in a fixed
 *    index order (slab, block, sample, warp), so training is bitwise reproducible run to run.  Partition sizes follow the
 *    SM count: results repeat on one GPU model, not across models.  Where a variant combines in the last-arriving CTA
 *    it takes a ticket from caller-zeroed uint32 counters and leaves them zero again (CUDA-graph replays need no reset).
 *  - activations live in the "pad-flat" NHWC layout: image n, pixel (y,x), channel c of an
 *    H x W x C map is element ((n*(H+1) + y)*(W+1) + x)*C + c; row y==H and column x==W of every
 *    image are zero padding shared with the neighbouring row/image, so a 3x3 tap is a constant
 *    row offset (dy*(W+1)+dx) and the zero border implements `padding=1`.  Kernels never write
 *    pad rows; buffers must be zero-initialised once by the caller.
 *  - 16-bit storage type is bfloat16 (IDF_BF16).
 */
#ifndef IDF_B200_H_
#define IDF_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* idf_stream_t; /* == cudaStream_t */

typedef enum {
  IDF_OK = 0,
  IDF_ERR_ARG = -1,      /* bad argument / unsupported shape           */
  IDF_ERR_CUDA = -2,     /* CUDA runtime/driver error                  */
  IDF_ERR_ARCH = -3,     /* device is not sm_100 (no fallback exists)  */
  IDF_ERR_NOMEM = -4
} idf_status;

int idf_version(void);
const char* idf_last_error(void);
/* Checks that the current device is sm_100, records its SM count and resolves the driver's tensor-map encoder. */
int idf_init(void);
/* Switches for tests, measurement and launch behaviour (unknown keys or values: IDF_ERR_ARG):
 *   "conv_force_mt" = 0 (auto) | 1 | 2 | 4   128-row tiles per CTA work unit of the conv kernel
 *   "conv_debug_skip_epilogue" = 0 | 1       plans created while set drain no output (main-loop ceiling)
 *   "pdl" = 0 | 1 (default)                   launch the conv / AdaGN kernels with programmatic dependent launch
 *   "conv_pair" = 0 | 1 (default)             conv plans with block_n >= 64 run as CTA pairs (tcgen05 cta_group::2)
 *   "xf_debug" = 0 | 1 | 2 | 5                measurement only: fused-AdaGN transform warps do nothing / skip the SiLU /
 *                                             5: no MMAs are issued (what the transform costs alone) */
int idf_set_option(const char* key, int32_t value);

/* ------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution on tcgen05 tensor cores (TMA-fed, TMEM accumulators).
 * Replaces nn.Conv2d 3x3/1x1 at modules.py:66,81,133-136,216,222,228,231,267,281,287,291,337,
 * 343,346 and models.py:246,283,431,467 (cuDNN in the reference), plus -- through the epilogue
 * modes -- the residual add modules.py:255,322,364, the attention residual modules.py:164 and
 * the sampler updates sampling.py:35-37,52-59,71-72.
 *
 * GEMM view: out[r, n] = sum_kb  A_kb[r + rowoff_kb, c0_kb : c0_kb+64] . Wp[n, 64*kb : 64*kb+64]
 * where A_kb is one of up to three pad-flat activation matrices (concat-K / fused 1x1 shortcut),
 * r runs over the pad-flat rows of the OUTPUT geometry and Wp is the packed bf16 weight matrix
 * [Cout_pad, 64*num_kb] (K contiguous).
 * ------------------------------------------------------------------------------------------ */
#define IDF_CONV_MAX_KB 160   /* 9 taps x 1024 input channels / 64 + a 1x1 shortcut over 1024 channels */
#define IDF_CONV_MAX_SRC 3

typedef enum {
  IDF_EPI_BF16 = 0,        /* out(bf16 pad-flat)[r, n] = acc + bias[n] (+ residual[r, n])            */
  IDF_EPI_F32_NCHW = 1,    /* out_f32 (NCHW [B,Cout,H,W]) = acc + bias                                */
  IDF_EPI_SAMPLER = 2      /* eps = acc + bias;  x = cx*x + ce*eps + cn*noise  (x, noise fp32 NCHW);
                              (cx,ce,cn) = coef[3*step], step = *step_ptr; eps also stored if out_f32 */
} idf_conv_epilogue;

typedef struct {
  /* A sources: pad-flat bf16 matrices [src_rows, src_ld] */
  int32_t n_src;
  const void* src[IDF_CONV_MAX_SRC];
  int64_t src_rows[IDF_CONV_MAX_SRC];
  int32_t src_ld[IDF_CONV_MAX_SRC];   /* channels per row (multiple of 64)                       */
  /* K-block table */
  int32_t num_kb;
  int32_t kb_src[IDF_CONV_MAX_KB];
  int32_t kb_c0[IDF_CONV_MAX_KB];     /* first channel of the 64-wide slice                      */
  int32_t kb_rowoff[IDF_CONV_MAX_KB]; /* signed row offset of the tap                            */
  /* B: packed weights [cout_pad, 64*num_kb] bf16, row-major */
  const void* weight;
  int32_t cout_pad;                   /* multiple of block_n                                     */
  int32_t block_n;                    /* 16, 64 or 128                                           */
  int32_t cout;                       /* real output channels                                    */
  const float* bias;                  /* [cout_pad] fp32                                         */
  /* output geometry */
  int32_t batch, H, W;                /* rows = batch*(H+1)*(W+1)                                */
  int32_t epilogue;                   /* idf_conv_epilogue                                       */
  void* out;                          /* bf16 pad-flat [rows, out_ld] (IDF_EPI_BF16)             */
  int32_t out_ld;
  const void* residual;               /* optional bf16 pad-flat [rows, res_ld]                   */
  int32_t res_ld;
  float* out_f32;                     /* NCHW fp32 (modes 1,2; may be NULL in mode 2)            */
  float* x_io;                        /* NCHW fp32, updated in place (mode 2)                    */
  const float* noise;                 /* NCHW fp32 (mode 2; may be NULL => cn ignored)           */
  const float* coef;                  /* [n_steps, 3] fp32 (mode 2)                              */
  const int32_t* step_ptr;            /* device scalar (mode 2)                                  */
  /* optional (IDF_EPI_BF16): GroupNorm partial sums of the stored (bf16-rounded) output, fp32
   * [2][ceil(rows/128)*4][cout][2] (capacity; the item form below fills a prefix).  Records cover UNITS of
   * idf_conv_plan_stats_unit(plan) rows:
   *   unit = 32   one record per 32-row window k = row/32 (windows never span 128-row tiles);
   *   unit = 128*MT (chosen when an image has at least that many pad-flat rows): 4 records per work item of MT
   *                 tiles, k = item*4 + q, q = lane quarter (rows 32q..32q+31 of each of the item's tiles).
   *   A[k][c] = (sum, sumsq) over the record's rows in the image the UNIT starts in,
   *   B[k][c] = the same over its rows in the following image (only written if the unit straddles).
   * Consumed by idf_adagn_silu_fwd / idf_adagn_coef (stats0 / stats1 with stats_unit0 / stats_unit1).   */
  float* stats_out;
  /* optional: AdaGN (+SiLU) of the CONSUMED activation fused into the A-operand path (inference): k-blocks with
   * kb_xf[k] >= 0 are read as bf16(act(A*x + B)), (A, B) = xf_coef[image][kb_xf[k] + channel - kb_c0[k]], act = SiLU
   * if xf_silu.  xf_coef: fp32 [batch][xf_ctot][2] written by idf_adagn_coef.  Pad rows stay zero.  A slice may be
   * read both transformed and raw (fused 1x1 shortcut).  xf_coef == NULL disables (kb_xf ignored).  Replaces the separate
   * GroupNorm/modulate/SiLU pass in front of every conv of modules.py:214-231, 265-291, 335-345, 132-136. */
  const float* xf_coef;
  int32_t xf_ctot;
  int32_t xf_silu;
  int32_t kb_xf[IDF_CONV_MAX_KB];
  /* optional (IDF_EPI_BF16): nearest-neighbour x2 upsampling folded into a 3x3 conv (UpSample, modules.py:89-92:
   * F.interpolate(scale 2, nearest) then Conv2d 3x3).  Output pixel (2y+py, 2x+px) only sees the 2x2 input
   * neighbourhood rows {y-1+py, y+py} x columns {x-1+px, x+px}, with the 3x3 weights that fall on the same input
   * pixel pre-summed: 4 taps instead of 9 and no upsampled tensor.  With up2 = 1 the GEMM runs over the INPUT grid
   * (batch, H, W = input geometry); the k-blocks are the 4 taps of parity (0, 0) (row offsets -(W+1)-1, -(W+1), -1, 0);
   * weight is [4*cout, 4*cin]: row block p = 2*py+px holds parity p's pre-summed taps; block_n == cout, cout_pad ==
   * 4*cout (column tile = parity, whose taps are shifted by py*(W+1)+px); `out` is the (2H) x (2W) pad-flat map
   * [batch*(2H+1)*(2W+1), out_ld]; stats_out records are 4*cout wide (one plane per parity, see idf_adagn_args
   * stats_planes / stats_rows).  residual must be NULL. */
  int32_t up2;
} idf_conv_desc;

typedef struct idf_conv_plan idf_conv_plan;
int idf_conv_plan_create(const idf_conv_desc* desc, idf_conv_plan** plan);
int idf_conv_plan_destroy(idf_conv_plan* plan);
int idf_conv_run(const idf_conv_plan* plan, idf_stream_t stream);
/* number of 128-row x block_n tiles a run processes (for roofline accounting) */
int64_t idf_conv_plan_tiles(const idf_conv_plan* plan);
/* rows per GroupNorm statistics unit of the records this plan writes to stats_out (32, or 128 * tiles per work item) */
int32_t idf_conv_plan_stats_unit(const idf_conv_plan* plan);

/* ------------------------------------------------------------------------------------------
 * Convolution weight gradient (autograd of nn.Conv2d w.r.t. weight), tcgen05, split-K with atomics (or ordered):
 *   dW[co, t, ci] += sum_r dY[r, co] * X[r + tap_off[t], ci]       dW fp32 [cout, n_taps, cin]
 * dY: bf16 pad-flat [rows, cout] (pad rows zero), X: bf16 [x_rows, cin] (cin multiple of 64).
 * The data gradient needs no kernel of its own: it is idf_conv_run over dY with transposed weights.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  const void* dy; int64_t rows; int32_t cout;
  const void* x; int64_t x_rows; int32_t cin;
  int32_t n_taps; int32_t tap_off[9];
  float* dw;
  /* optional: fp32 workspace of idf_wgrad_plan_partials_floats(plan) floats.  When set, every split-K slab stores its
   * partial dW and a second launch adds the slabs to dw in slab order (bitwise reproducible); NULL = atomics.  Plans
   * with one slab need none and add directly either way.  The pointer is captured by idf_wgrad_plan_create. */
  float* partials;
} idf_wgrad_desc;
typedef struct idf_wgrad_plan idf_wgrad_plan;
int idf_wgrad_plan_create(const idf_wgrad_desc* desc, idf_wgrad_plan** plan);
int64_t idf_wgrad_plan_partials_floats(const idf_wgrad_plan* plan);   /* 0 for single-slab plans */
int idf_wgrad_plan_destroy(idf_wgrad_plan* plan);
int idf_wgrad_run(const idf_wgrad_plan* plan, idf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Fused AdaGN: GroupNorm(32) statistics + affine + timestep scale/shift + latent-z scale/shift
 * + SiLU, one HBM read and one HBM write.  Replaces nn.GroupNorm + the modulation chain + nn.SiLU
 * at modules.py:214-215, 219-221, 225-227, 249-253, 265-266, 278-280, 284-286, 312-319, 335-336,
 * 340-341, the attention GroupNorm modules.py:132,147 and the torch.cat of models.py:321,505
 * (two sources are normalised as one concatenated map).
 *   y = silu?( ((gn(x)*gamma+beta) * (1+s_t) + b_t) * (1+s_z) + b_z )
 * mod_t / mod_z point at [.., 2*C] rows holding (scale | shift); the row used for sample n is
 *   mod + (step_ptr ? *step_ptr : 0) * step_stride + n * batch_stride        (either may be NULL)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  const void* src0; int32_t c0;       /* bf16 pad-flat [rows, c0]                                */
  const void* src1; int32_t c1;       /* optional second source (concat along C), c1 may be 0    */
  void* out;                          /* bf16 pad-flat [rows, c0+c1]                             */
  int32_t batch, H, W;
  const float* gamma; const float* beta;   /* [c0+c1]                                            */
  float eps;
  const float* mod_t; int64_t mod_t_step_stride; int64_t mod_t_batch_stride;
  const float* mod_z; int64_t mod_z_step_stride; int64_t mod_z_batch_stride;
  const int32_t* step_ptr;
  int32_t apply_silu;
  /* optional: per-tile partial sums written by the producing convolution (idf_conv_desc.stats_out).
   * When given for every source the kernel is a single streaming sweep (no statistics pass).     */
  const float* stats0; const float* stats1;
  /* training only: inverted dropout applied after SiLU (nn.Dropout at modules.py:221,227,280,286,342).
   * keep-mask = hash(*dropout_seed, dropout_layer, element index) >= p; 0 disables.               */
  float dropout_p; const uint64_t* dropout_seed; uint32_t dropout_layer;
  /* training only, optional: fp32 [batch, C, 4] = (A, B, group mean, group rstd) per sample and channel with
   * v = A*x + B, written by the forward (streaming variant) and read back by idf_adagn_silu_bwd. */
  float* save_coef;
  /* rows per statistics unit of stats0 / stats1 (idf_conv_plan_stats_unit of the producing plan); 0 = 32 */
  int32_t stats_unit0, stats_unit1;
  /* statistics written by an up2 conv plan: records are stats_planes * c columns wide (the planes are summed) and
   * indexed over the PRODUCER's grid of stats_rows pad-flat rows per image ((H/2+1)*(W/2+1)); 0 = 1 plane, this map's rows */
  int32_t stats_planes0, stats_planes1;
  int32_t stats_rows0, stats_rows1;
} idf_adagn_args;
int idf_adagn_silu_fwd(const idf_adagn_args* args, idf_stream_t stream);
/* Coefficients only: coef_out[n][c] = (A, B) with AdaGN(x)[n, c, :, :] = A*x + B (before the activation), from the
 * producers' window records (stats0 / stats1 required).  Feeds idf_conv_desc.xf_coef; out / src pointers of
 * `args` are not dereferenced. */
int idf_adagn_coef(const idf_adagn_args* args, float* coef_out, idf_stream_t stream);

/* Backward of idf_adagn_silu_fwd (streaming variant: stats0/stats1 required).
 *   dx0 / dx1 : gradient w.r.t. the sources (bf16 pad-flat; added to the buffer if acc0 / acc1)
 *   sums      : fp32 [batch, C, 2] = (sum_hw dv, sum_hw dv * xhat) with dv = dL/d(pre-activation) -- every
 *               parameter / modulation gradient of the op is a closed form of these (see models.py mirror)
 *   ws        : fp32 workspace, idf_adagn_bwd_ws_floats(batch, C) floats                            */
typedef struct {
  idf_adagn_args f;
  const void* dy;
  void* dx0; void* dx1;
  int32_t acc0, acc1;
  float* sums;
  float* ws;
  /* optional fused parameter gradients (closed forms of S1, S2; any pointer may be NULL):
   *   d_mod_t / d_mod_z : fp32 rows laid out like mod_t / mod_z of the forward args (same strides), receive
   *                       (d scale | d shift) of this op;  dgamma / dbeta : fp32 [C], accumulated (atomics) */
  float* d_mod_t; float* d_mod_z; float* dgamma; float* dbeta;
  /* optional, ordered dgamma / dbeta: fp32 [batch, C, 2] workspace and one caller-zeroed uint32 ticket; the per-sample
   * contributions are added in sample order instead of with atomics.  NULL = atomics. */
  float* dparam_ws; uint32_t* dparam_ticket;
} idf_adagn_bwd_args;
int64_t idf_adagn_bwd_ws_floats(int32_t batch, int32_t C);
int idf_adagn_silu_bwd(const idf_adagn_bwd_args* args, idf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Fused single-head self attention (QK^T -> softmax -> PV on tcgen05), S = H*W tokens, d = 128.
 * Replaces torch.bmm / F.softmax / permutes at modules.py:152-161.
 * qkv: bf16 pad-flat [rows, 3*d] (q | k | v), out: bf16 pad-flat [rows, d]; scale = d^-0.5.
 * ------------------------------------------------------------------------------------------ */
int idf_attn_fwd(const void* qkv, void* out, int32_t batch, int32_t H, int32_t W, int32_t d, float scale,
                 idf_stream_t stream);

/* Backward of idf_attn_fwd (autograd of modules.py:145-164): dqkv [rows, 3*d] (dq | dk | dv, interior rows only) from the
 * saved qkv and dout = dL/dO [rows, d].  Supported shapes:
 *   H*W in {64, 256} with d in {128, 256, 512}: two tcgen05 kernels per call (scores: P and dS rows -> workspace;
 *     gradients: dQ = dS K, dK = dS^T Q, dV = P^T dO); ws = idf_attn_bwd_ws_bytes(batch, H, W) bytes of device memory,
 *     1024-aligned (the same for every d);
 *   otherwise H*W <= 64 with H*W*d <= 8192: a small-map kernel (ws unused).
 * Other shapes return IDF_ERR_CUDA with a message naming these. */
int idf_attn_bwd(const void* qkv, const void* dout, void* dqkv, void* ws, int32_t batch, int32_t H, int32_t W, int32_t d,
                 float scale, idf_stream_t stream);
int64_t idf_attn_bwd_ws_bytes(int32_t batch, int32_t H, int32_t W);


/* ------------------------------------------------------------------------------------------
 * Small fp32 linear:  y[m, n] = sum_k act(x[m, k]) * w[n, k] + b[n]   (act = SiLU if silu_in)
 * Replaces nn.Linear at modules.py:24,26,211,271,275 and models.py:244,470-472 (cuBLAS addmm).
 * ------------------------------------------------------------------------------------------ */
int idf_linear_f32(const float* x, int64_t ldx, const float* w, const float* b, float* y, int64_t ldy, int32_t M,
                   int32_t N, int32_t K, int32_t silu_in, idf_stream_t stream);
/* General small fp32 GEMM, C[M,N] (+)= op(A)[M,K] . op(B)[K,N] with op(X) = X or X^T (row-major, leading dimensions):
 * the BACKWARD of those Linears under autograd (dX = dY.W, dW = dY^T.X, db = 1^T.dY) -- replaces cuBLAS gemm / addmm
 * in the autograd graph of modules.py:24-27, 211, 271-275 and models.py:147-163, 223-234, 470-472. */
int idf_gemm_f32(const float* A, int64_t lda, int32_t transA, const float* B, int64_t ldb, int32_t transB, float* C,
                 int64_t ldc, int32_t M, int32_t N, int32_t K, int32_t accumulate, idf_stream_t stream);
/* Same result with split-K partial tiles combined in split order (bitwise reproducible): ws holds
 * idf_gemm_f32_ws_floats(M, N, K) floats (0: no split, ws and tickets unused), tickets 64 caller-zeroed uint32. */
int idf_gemm_f32_ordered(const float* A, int64_t lda, int32_t transA, const float* B, int64_t ldb, int32_t transB, float* C,
                         int64_t ldc, int32_t M, int32_t N, int32_t K, int32_t accumulate, float* ws, uint32_t* tickets,
                         idf_stream_t stream);
int64_t idf_gemm_f32_ws_floats(int32_t M, int32_t N, int32_t K);

/* y[m, :] = table[idx[m], :]  (nn.Embedding lookup, modules.py:23,37) */
int idf_gather_rows_f32(const float* table, const int64_t* idx, float* y, int32_t M, int32_t N, idf_stream_t stream);
/* LatentUNet layer tail, MLPLNAct.forward (models.py:147-163) after the Linear: out[m, :] = SiLU(LayerNorm(y[m, :] *
 * (1 + cond[m, :]))), condition_bias = 1 (models.py:219).  cond may be NULL (no modulation) or one broadcast row
 * (cond_row_stride = 0); with step_ptr the row block starts at cond + *step_ptr * cond_step_stride (per-timestep
 * table inside a captured sampler graph); gamma/beta NULL = no affine; apply_silu = 0 for an activation-less
 * layer. fp32, N <= 8192. */
int idf_scale_layernorm_silu(const float* y, int64_t ldy, const float* cond, int64_t cond_row_stride,
                             int64_t cond_step_stride, const int32_t* step_ptr, const float* gamma, const float* beta,
                             float eps, float* out, int64_t ldo, int32_t M, int32_t N, int32_t apply_silu,
                             idf_stream_t stream);
/* Train-step tail: torch.nn.utils.clip_grad_norm_(params, max_norm) + torch.optim.AdamW.step() (run.py:199-200, 177)
 * over all parameter tensors in three launches.  Tables live in device memory: one pointer per tensor and one
 * (tensor, offset / 4096) pair per 4096-element chunk.  fp32 everywhere.  norm_out[0] = total gradient norm (what
 * clip_grad_norm_ returns), norm_out[1] = applied clip coefficient.  Gradients are scaled on the fly, not written
 * back.  max_norm <= 0 disables clipping.  bias_corrections[2*i + k-1] = 1 - betaK^step_i for tensor i (torch keeps
 * one step count per parameter; a parameter that skipped steps has its own). */
typedef struct {
  void* const* params; const void* const* grads; void* const* exp_avg; void* const* exp_avg_sq;
  const int64_t* numel; const int32_t* chunk_tensor; const int32_t* chunk_offset;
  int32_t n_chunks;
  const float* bias_corrections;   /* device, [n_tensors][2] */
  float lr, beta1, beta2, eps, weight_decay, max_norm;
  float* partial;      /* [n_chunks] scratch */
  float* norm_out;     /* [2] */
} idf_clip_adamw_args;
int idf_clip_adamw(const idf_clip_adamw_args* args, idf_stream_t stream);
/* eval_fid output stage (run.py:288-295 followed by torchvision.utils.save_image): x fp32 NCHW in [-1, 1] ->
 * uint8 NHWC, u = trunc(clamp(((clip(x,-1,1) + 1) / 2) * 255 + 0.5, 0, 255)), the bytes the reference's PNGs hold. */
int idf_to_uint8_hwc(const float* x, uint8_t* out, int32_t batch, int32_t C, int32_t H, int32_t W, idf_stream_t stream);
/* dst[m, n] = src[m, n] for an M x N fp32 block with row pitches lds / ldd: places x next to h for the skip
 * concatenation cat([h, x]) of LatentUNet (models.py:230-232). */
int idf_copy2d_f32(const float* src, int64_t lds, float* dst, int64_t ldd, int32_t M, int32_t N, idf_stream_t stream);
/* dst[i] (+)= src[idx[i]-1] (+ src[idx2[i]-1]);  index 0 = literal zero, idx2 may be NULL, n % 4 == 0.
 * Training only: one launch re-packs all fp32 parameters into the bf16 GEMM operand layouts that the
 * reference obtains implicitly from nn.Conv2d.weight (modules.py:66,81,133-136,216-231), another assembles
 * parameter-shaped gradients from the weight-gradient arena (what autograd does per parameter). */
int idf_gather_elems(const float* src, const int32_t* idx, const int32_t* idx2, void* dst, int64_t n, int32_t dst_bf16,
                     int32_t accumulate, idf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Layout / data-movement kernels
 * ------------------------------------------------------------------------------------------ */
/* x NCHW fp32 [B,C,H,W] (C<=7) -> 3x3 im2col patches bf16 pad-flat [rows, 64] (k = tap*C + c,
 * zero beyond 9*C): turns the head conv (models.py:246,304,431) into a K=64 1x1 GEMM. */
int idf_im2col_head(const float* x, void* out, int32_t batch, int32_t C, int32_t H, int32_t W, idf_stream_t stream);
/* nearest x2 upsample (F.interpolate, modules.py:90-91) in pad-flat layout: [B,H,W,C] -> [B,2H,2W,C] */
int idf_upsample2x(const void* in, void* out, int32_t batch, int32_t H, int32_t W, int32_t C, idf_stream_t stream);
/* space-to-depth split for the stride-2 conv (modules.py:66): in [B,H,W,C] -> out[4][B,H/2,W/2,C],
 * out[py*2+px][n,y,x] = in[n,2y+py,2x+px]. */
int idf_space_to_depth(const void* in, void* out, int32_t batch, int32_t H, int32_t W, int32_t C,
                       idf_stream_t stream);
/* pad-flat bf16 [B,H,W,C] <-> NCHW fp32 (debug / block-level tests / training boundary) */
int idf_nchw_to_padflat(const float* x, void* out, int32_t batch, int32_t C, int32_t H, int32_t W,
                        idf_stream_t stream);
int idf_padflat_to_nchw(const void* in, float* y, int32_t batch, int32_t C, int32_t H, int32_t W,
                        idf_stream_t stream);
/* same as idf_nchw_to_padflat but into rows of `ld` >= C channels (the extra channels are left untouched) */
int idf_nchw_to_padflat_ld(const float* x, void* out, int32_t batch, int32_t C, int32_t H, int32_t W, int32_t ld,
                           idf_stream_t stream);
/* backward of the layout ops (training): gradients are bf16 pad-flat; `accumulate` adds into the target */
int idf_upsample2x_bwd(const void* dout, void* din, int32_t batch, int32_t H, int32_t W, int32_t C, int32_t accumulate,
                       idf_stream_t stream);   /* H, W: INPUT (low) resolution */
int idf_depth_to_space(const void* dphases, void* din, int32_t batch, int32_t H, int32_t W, int32_t C, int32_t accumulate,
                       idf_stream_t stream);   /* H, W: full resolution; inverse of idf_space_to_depth */
/* out[c] += sum_r m[r, c]  (bias gradient of a conv: column sums of dY), fp32 atomics */
int idf_colsum_bf16(const void* m, float* out, int64_t rows, int32_t C, idf_stream_t stream);
/* the same sum with the block partials added in block order: ws = idf_colsum_ws_floats(rows, C) floats, tickets = one
 * caller-zeroed uint32 */
int idf_colsum_bf16_ordered(const void* m, float* out, int64_t rows, int32_t C, float* ws, uint32_t* tickets,
                            idf_stream_t stream);
int64_t idf_colsum_ws_floats(int64_t rows, int32_t C);

/* ------------------------------------------------------------------------------------------
 * Stand-alone sampler update (the unfused variant of IDF_EPI_SAMPLER):
 *   x = cx*x + ce*eps + cn*noise,  (cx,ce,cn) = coef[3*step].  sampling.py:35-37, 52-59, 71-72.
 * ------------------------------------------------------------------------------------------ */
int idf_sampler_update(float* x, const float* eps, const float* noise, const float* coef, const int32_t* step_ptr,
                       int64_t n, idf_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * MMD prior loss (utils.py:74-90), fused pairwise Gaussian-kernel reduction.
 *   loss = mean k(x,x) + mean k(y,y) - 2 mean k(x,y),  k(u,v) = exp(-|u-v|^2 / D^2)
 * x: prior samples [B,D], y: latents [B,D]; grad_y (optional) = d loss / d y.
 * ------------------------------------------------------------------------------------------ */
int idf_mmd_fwd_bwd(const float* x, const float* y, float* loss, float* grad_y, int32_t B, int32_t D,
                    idf_stream_t stream);
/* the same with grad_y summed per warp and the per-row loss partials summed in row order: ws = idf_mmd_ws_floats(B)
 * floats, tickets = one caller-zeroed uint32 */
int idf_mmd_fwd_bwd_ordered(const float* x, const float* y, float* loss, float* grad_y, int32_t B, int32_t D, float* ws,
                            uint32_t* tickets, idf_stream_t stream);
int64_t idf_mmd_ws_floats(int32_t B);

#ifdef __cplusplus
}
#endif
#endif /* IDF_B200_H_ */
