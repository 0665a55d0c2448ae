// extern "C" boundary of libidf_b200.so (declared in include/idf_b200.h).
// Plain pointers and sizes only; TMA tensor maps are built here so callers never see CUtensorMap.
#include <cudaTypedefs.h>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <new>
#include <vector>

#include "kernels.cuh"

using namespace idf;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int cuda_fail(cudaError_t e, const char* what) {
  return fail(IDF_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
int g_num_sms = 0;
int g_force_mt = 0;   // 0 = choose automatically
int g_skip_epilogue = 0;
int g_conv_pair = 1;  // conv kernels with N >= 64 run as CTA pairs (idf_set_option "conv_pair", 0 = single CTAs)

int ensure_init() {
  if (g_encode != nullptr) return IDF_OK;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceProperties");
  if (prop.major != 10)
    return fail(IDF_ERR_ARCH, "idf_b200 requires an sm_100 device (found sm_%d%d); there is no fallback path",
                prop.major, prop.minor);
  g_num_sms = prop.multiProcessorCount;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || fn == nullptr || qres != cudaDriverEntryPointSuccess)
    return fail(IDF_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
  return IDF_OK;
}

// 2-D bf16 row-major matrix [rows, ld] -> box {64 elements, box_rows}, 128B swizzle
int encode_2d(CUtensorMap* tm, const void* base, int64_t rows, int32_t ld, int32_t box_rows) {
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return fail(IDF_ERR_ARG, "TMA base not 16-byte aligned");
  if (ld % 64 != 0 && ld % 8 != 0) return fail(IDF_ERR_ARG, "row pitch must be a multiple of 16 bytes");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(ld), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {64, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estride[2] = {1, 1};
  CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estride,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(IDF_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return IDF_OK;
}

// 2-D bf16 row-major matrix [rows, ld] -> box {32 elements, 32 rows}, 64B swizzle: the epilogue's output tile
// (one epilogue warp's 32 rows x 32 columns), written with a TMA store
int encode_2d_out(CUtensorMap* tm, const void* base, int64_t rows, int32_t ld) {
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return fail(IDF_ERR_ARG, "TMA base not 16-byte aligned");
  if (ld % 8 != 0) return fail(IDF_ERR_ARG, "row pitch must be a multiple of 16 bytes");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(ld), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estride[2] = {1, 1};
  CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estride,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(IDF_ERR_CUDA, "cuTensorMapEncodeTiled (output) failed with CUresult %d", (int)r);
  return IDF_OK;
}

}  // namespace

struct idf_conv_plan {
  ConvKernelParams params;
  int block_n;
  int mt;      // 128-row tiles per CTA work unit
  int grid;
  bool xform;  // some halo group carries a fused AdaGN: launch the variant with transform warps
  bool pair;   // launched as clusters of two CTAs (tcgen05 cta_group::2)
  int stats_unit;  // rows per GroupNorm statistics unit of the records written to stats_out
  int64_t tiles;
};

extern "C" {

int idf_version(void) { return 100; }
const char* idf_last_error(void) { return g_err; }
int idf_init(void) { return ensure_init(); }

int idf_set_option(const char* key, int32_t value) {
  if (key != nullptr && std::strcmp(key, "conv_force_mt") == 0 && (value == 0 || value == 1 || value == 2 || value == 4)) {
    g_force_mt = value;
    return IDF_OK;
  }
  if (key != nullptr && std::strcmp(key, "conv_debug_skip_epilogue") == 0) {
    g_skip_epilogue = value ? 1 : 0;
    return IDF_OK;
  }
  if (key != nullptr && std::strcmp(key, "conv_pair") == 0 && (value == 0 || value == 1)) { g_conv_pair = value; return IDF_OK; }
  if (key != nullptr && std::strcmp(key, "pdl") == 0) { g_pdl = value ? 1 : 0; return IDF_OK; }
  if (key != nullptr && std::strcmp(key, "xf_debug") == 0 && value >= 0 && value <= 5) { g_xf_debug = value; return IDF_OK; }
  return fail(IDF_ERR_ARG, "unknown option or value");
}

int idf_conv_plan_create(const idf_conv_desc* d, idf_conv_plan** out_plan) {
  if (d == nullptr || out_plan == nullptr) return fail(IDF_ERR_ARG, "null argument");
  int rc = ensure_init();
  if (rc != IDF_OK) return rc;
  if (d->n_src < 1 || d->n_src > IDF_CONV_MAX_SRC) return fail(IDF_ERR_ARG, "n_src out of range");
  if (d->num_kb < 1 || d->num_kb > IDF_CONV_MAX_KB) return fail(IDF_ERR_ARG, "num_kb out of range (%d)", d->num_kb);
  if (d->block_n != 16 && d->block_n != 64 && d->block_n != 128) return fail(IDF_ERR_ARG, "block_n must be 16/64/128");
  if (d->cout_pad % d->block_n != 0) return fail(IDF_ERR_ARG, "cout_pad must be a multiple of block_n");
  if (d->batch < 1 || d->H < 1 || d->W < 1) return fail(IDF_ERR_ARG, "bad geometry");
  if (d->cout_pad > 1536) return fail(IDF_ERR_ARG, "cout_pad > 1536 not supported (bias staging)");
  if (static_cast<int64_t>(d->batch) * (d->H + 1) * (d->W + 1) >= (1 << 22))
    return fail(IDF_ERR_ARG, "more than 2^22 pad-flat rows per launch: split the batch");
  if (d->epilogue == IDF_EPI_BF16) {
    if (d->block_n < 64) return fail(IDF_ERR_ARG, "bf16 epilogue needs block_n >= 64");
    if (d->out == nullptr || d->out_ld % 8 != 0 || (d->up2 == 0 && d->cout != d->cout_pad))
      return fail(IDF_ERR_ARG, "bf16 epilogue: out/out_ld/cout invalid");
    if (d->up2 != 0 && (d->block_n != d->cout || d->cout_pad != 4 * d->cout || d->residual != nullptr || d->xf_coef != nullptr))
      return fail(IDF_ERR_ARG, "up2: needs block_n == cout, cout_pad == 4*cout, no residual, no fused AdaGN");
    if (d->residual != nullptr && d->res_ld % 8 != 0) return fail(IDF_ERR_ARG, "res_ld must be a multiple of 8");
  } else if (d->up2 != 0) {
    return fail(IDF_ERR_ARG, "up2 needs the bf16 epilogue");
  } else if (d->epilogue == IDF_EPI_F32_NCHW || d->epilogue == IDF_EPI_SAMPLER) {
    if (d->block_n != 16 || d->cout > 16) return fail(IDF_ERR_ARG, "fp32/sampler epilogue needs block_n == 16");
    if (d->epilogue == IDF_EPI_F32_NCHW && d->out_f32 == nullptr) return fail(IDF_ERR_ARG, "out_f32 is null");
    if (d->epilogue == IDF_EPI_SAMPLER && (d->x_io == nullptr || d->coef == nullptr))
      return fail(IDF_ERR_ARG, "sampler epilogue needs x_io and coef");
  } else {
    return fail(IDF_ERR_ARG, "unknown epilogue %d", d->epilogue);
  }
  idf_conv_plan* pl = new (std::nothrow) idf_conv_plan;
  if (pl == nullptr) return fail(IDF_ERR_NOMEM, "out of host memory");
  std::memset(pl, 0, sizeof(*pl));
  ConvKernelParams& p = pl->params;
  for (int i = 0; i < d->n_src; ++i) {
    if (d->src[i] == nullptr || d->src_ld[i] % 64 != 0) {
      delete pl;
      return fail(IDF_ERR_ARG, "source %d: null or channel count not a multiple of 64", i);
    }
  }
  // ---- K-block table -> groups: per (source, 64-channel slice), taps whose row offsets lie within a
  //      few hundred rows of each other share one halo load (3x3 taps; the phases of a stride-2 conv
  //      are far apart and form separate groups).
  struct Tap { int src, c0, off, kb, xf; };
  const bool use_xf = d->xf_coef != nullptr;
  if (use_xf && (d->xf_ctot <= 0 || d->xf_ctot % 8 != 0)) { delete pl; return fail(IDF_ERR_ARG, "xf_ctot must be a positive multiple of 8"); }
  std::vector<Tap> taps;
  for (int k = 0; k < d->num_kb; ++k) {
    if (d->kb_src[k] < 0 || d->kb_src[k] >= d->n_src || d->kb_c0[k] < 0 || d->kb_c0[k] % 64 != 0 ||
        d->kb_c0[k] + kBK > d->src_ld[d->kb_src[k]]) {
      delete pl;
      return fail(IDF_ERR_ARG, "k-block %d out of range", k);
    }
    const int xf = use_xf ? d->kb_xf[k] : -1;
    if (xf >= 0 && (xf % 8 != 0 || xf + kBK > d->xf_ctot)) { delete pl; return fail(IDF_ERR_ARG, "k-block %d: kb_xf out of range", k); }
    taps.push_back({d->kb_src[k], d->kb_c0[k], d->kb_rowoff[k], k, xf < 0 ? -1 : xf});
  }
  std::stable_sort(taps.begin(), taps.end(), [](const Tap& a, const Tap& b) {
    if (a.src != b.src) return a.src < b.src;
    if (a.c0 != b.c0) return a.c0 < b.c0;
    if (a.xf != b.xf) return a.xf > b.xf;      // transformed and raw reads of one slice are separate halo loads
    return a.off < b.off;
  });
  p.n_src = d->n_src;
  p.n_groups = 0;
  p.n_taps = 0;
  int group_hi[kMaxGroups] = {0};
  for (size_t i = 0; i < taps.size(); ++i) {
    const Tap& t = taps[i];
    int g = p.n_groups - 1;
    const bool same = g >= 0 && p.g_src[g] == t.src && p.g_c0[g] == t.c0 && p.g_xf[g] == t.xf && (t.off - p.g_lo[g]) <= 248;
    if (!same) {
      if (p.n_groups == kMaxGroups) { delete pl; return fail(IDF_ERR_ARG, "too many halo groups"); }
      g = p.n_groups++;
      p.g_src[g] = t.src; p.g_c0[g] = t.c0; p.g_lo[g] = t.off; p.g_ntaps[g] = 0; p.g_xf[g] = t.xf;
    }
    p.t_rel[p.n_taps] = t.off - p.g_lo[g];
    p.t_kb[p.n_taps] = t.kb;
    p.n_taps++;
    p.g_ntaps[g]++;
    group_hi[g] = t.off;
  }
  if (d->up2 != 0)      // the parity column tiles shift the taps by up to one row and one pixel
    for (int g = 0; g < p.n_groups; ++g) group_hi[g] += (d->W + 1) + 1;
  int extra_max = 0;
  for (int i = 0; i < d->n_src; ++i) p.extra_rows[i] = 0;
  for (int g = 0; g < p.n_groups; ++g) {
    const int ex = (group_hi[g] - p.g_lo[g] + 7) / 8 * 8;
    if (ex > p.extra_rows[p.g_src[g]]) p.extra_rows[p.g_src[g]] = ex;
    if (ex > extra_max) extra_max = ex;
  }
  // ---- geometry and tile shape
  p.Hp = d->H + 1;
  p.Wp = d->W + 1;
  p.H = d->H;
  p.W = d->W;
  p.rows = static_cast<int64_t>(d->batch) * p.Hp * p.Wp;
  const int64_t m_tiles = (p.rows + kBM - 1) / kBM;
  p.n_tiles = d->cout_pad / d->block_n;
  // MT 128-row tiles per CTA work unit: the largest (best weight-tile reuse: MT = 1 streams 16 KB of
  // weights per 256 MMA cycles and is L2-bound) that still fills the machine with <= 15 % quantisation
  // loss in the number of rounds over the SMs.
  // CTA pairs (cta_group::2, see conv_igemm.cu): a worker is two CTAs and its work unit 2*MT tiles.
  const bool pair = g_conv_pair != 0 && d->block_n >= 64 && g_num_sms % 2 == 0;
  const int pw = pair ? 2 : 1;
  const int workers = g_num_sms / pw;
  // MT 128-row tiles per work item: larger items reuse every streamed weight tile MT times and have relatively less
  // halo, but quantise the work more coarsely.  Cost model: rounds over the workers x (MT tiles + 0.4 of a tile for the
  // per-item pipeline fill and weight stream), e.g. 162 tiles on 74 pairs: MT = 2 -> 41 items, one round of 2.4, beats
  // MT = 1 -> 81 items, two rounds of 1.4.  Ties go to the larger MT.
  const int mt_max = (d->block_n == 128) ? 2 : 4;
  int mt = 1;
  double best = 1e30;
  for (int cand = 1; cand <= mt_max; cand <<= 1) {
    if (d->block_n == 16 && cand == 2) continue;   // instantiated: 16x{1,4}
    const int stage = ((cand * kBM + extra_max) * 128 + 1023) / 1024 * 1024;
    if (conv_config_smem(d->block_n, cand, stage, pair, use_xf) > 227 * 1024) continue;
    const int64_t units = (m_tiles + cand * pw - 1) / (cand * pw) * p.n_tiles;
    const int64_t rounds = (units + workers - 1) / workers;
    const double cost = static_cast<double>(rounds) * (cand + 0.4);
    if (cost <= best) { best = cost; mt = cand; }
  }
  if (g_force_mt != 0) {
    mt = g_force_mt;
    if (mt > mt_max || (d->block_n == 16 && mt == 2)) { delete pl; return fail(IDF_ERR_ARG, "forced MT not available"); }
  }
  p.a_stage_bytes = ((mt * kBM + extra_max) * 128 + 1023) / 1024 * 1024;
  if (conv_config_smem(d->block_n, mt, p.a_stage_bytes, pair, use_xf) > 227 * 1024) {
    delete pl;
    return fail(IDF_ERR_ARG, "halo does not fit in shared memory (extra rows %d)", extra_max);
  }
  p.m_super = static_cast<int32_t>((m_tiles + mt * pw - 1) / (mt * pw));
  p.m_tiles = static_cast<int32_t>(m_tiles);
  p.debug_skip_epilogue = g_skip_epilogue;
  p.stats = (d->epilogue == IDF_EPI_BF16) ? d->stats_out : nullptr;
  p.up2 = d->up2 != 0 ? 1 : 0;
  p.stats_ld = d->up2 != 0 ? d->cout_pad : d->out_ld;
  p.stats_b_off = static_cast<int64_t>(m_tiles) * 4 * p.stats_ld * 2;
  // item-level records when a work item spans at most two images
  p.stats_item = (p.stats != nullptr && d->block_n >= 64 &&
                  static_cast<int64_t>(p.Hp) * p.Wp >= static_cast<int64_t>(mt) * kBM) ? 1 : 0;
  pl->stats_unit = p.stats_item ? mt * kBM : 32;
  if (p.stats != nullptr && d->out_ld != d->cout) { delete pl; return fail(IDF_ERR_ARG, "stats_out needs out_ld == cout"); }
  if (p.stats != nullptr && !window_records_exact(d->H, d->W)) {
    delete pl;
    return fail(IDF_ERR_ARG, "stats_out: 32-row GroupNorm records cannot keep the images of a %dx%d grid apart "
                "(needs (H+1)*(W+1) >= 32 or 31 - (H+1)*(W+1) <= W+2)", d->H, d->W);
  }
  for (int i = 0; i < d->n_src; ++i) {
    rc = encode_2d(&p.tmA[i], d->src[i], d->src_rows[i], d->src_ld[i], kBM);
    if (rc != IDF_OK) { delete pl; return rc; }
    if (p.extra_rows[i] > 0) {
      if (p.extra_rows[i] > 256) { delete pl; return fail(IDF_ERR_ARG, "tap spread too large for one TMA box"); }
      rc = encode_2d(&p.tmAx[i], d->src[i], d->src_rows[i], d->src_ld[i], p.extra_rows[i]);
      if (rc != IDF_OK) { delete pl; return rc; }
    }
  }
  rc = encode_2d(&p.tmB, d->weight, d->cout_pad, d->num_kb * kBK, d->block_n / pw);
  if (rc != IDF_OK) { delete pl; return rc; }
  if (d->epilogue == IDF_EPI_BF16 && d->up2 == 0) {
    rc = encode_2d_out(&p.tmOut, d->out, p.rows, d->out_ld);
    if (rc != IDF_OK) { delete pl; return rc; }
  }
  p.cout = d->cout;
  p.epilogue = d->epilogue;
  p.bias = d->bias;
  p.out = static_cast<bf16*>(d->out);
  p.out_ld = d->out_ld;
  p.residual = static_cast<const bf16*>(d->residual);
  p.res_ld = d->res_ld;
  p.out_f32 = d->out_f32;
  p.x_io = d->x_io;
  p.noise = d->noise;
  p.coef = d->coef;
  p.step_ptr = d->step_ptr;
  p.xf_coef = reinterpret_cast<const float2*>(d->xf_coef);
  p.xf_ctot = d->xf_ctot;
  p.xf_silu = d->xf_silu;
  p.xf_debug = g_xf_debug;
  pl->xform = false;
  for (int g = 0; g < p.n_groups; ++g) pl->xform = pl->xform || p.g_xf[g] >= 0;
  if (p.bias == nullptr) { delete pl; return fail(IDF_ERR_ARG, "bias is null"); }
  pl->block_n = d->block_n;
  pl->mt = mt;
  pl->pair = pair;
  pl->tiles = m_tiles * p.n_tiles;
  const long long units = static_cast<long long>(p.m_super) * p.n_tiles;
  pl->grid = pw * static_cast<int>(units < workers ? units : workers);
  *out_plan = pl;
  return IDF_OK;
}

int idf_conv_plan_destroy(idf_conv_plan* plan) {
  delete plan;
  return IDF_OK;
}

int64_t idf_conv_plan_tiles(const idf_conv_plan* plan) {
  return plan ? plan->tiles : 0;
}

int32_t idf_conv_plan_stats_unit(const idf_conv_plan* plan) {
  return plan ? plan->stats_unit : 0;
}

int idf_conv_run(const idf_conv_plan* plan, idf_stream_t stream) {
  if (plan == nullptr) return fail(IDF_ERR_ARG, "null plan");
  cudaError_t e = launch_conv_igemm(plan->params, plan->block_n, plan->mt, plan->xform, plan->pair, plan->grid, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "conv_igemm launch");
  return IDF_OK;
}

struct idf_wgrad_plan {
  WgradKernelParams params;
  int grid;
  int slabs;
};

int idf_wgrad_plan_create(const idf_wgrad_desc* d, idf_wgrad_plan** out_plan) {
  if (d == nullptr || out_plan == nullptr) return fail(IDF_ERR_ARG, "null argument");
  int rc = ensure_init();
  if (rc != IDF_OK) return rc;
  if (d->dy == nullptr || d->x == nullptr || d->dw == nullptr) return fail(IDF_ERR_ARG, "null tensor");
  if (d->cin % 64 != 0 || d->cout % 8 != 0 || d->n_taps < 1 || d->n_taps > 9) return fail(IDF_ERR_ARG, "bad wgrad shape");
  idf_wgrad_plan* pl = new (std::nothrow) idf_wgrad_plan;
  if (pl == nullptr) return fail(IDF_ERR_NOMEM, "out of host memory");
  std::memset(pl, 0, sizeof(*pl));
  WgradKernelParams& p = pl->params;
  // tap clusters: taps whose offsets lie within 8 rows share one X halo (the kx = 0,1,2 taps of a kernel row)
  std::vector<std::pair<int, int>> taps;   // (offset, tap id)
  for (int t = 0; t < d->n_taps; ++t) taps.push_back({d->tap_off[t], t});
  std::sort(taps.begin(), taps.end());
  struct Cl { int base; int n; int rel[3]; int id[3]; };
  std::vector<Cl> cls;
  for (auto& t : taps) {
    if (!cls.empty() && cls.back().n < 3 && t.first - cls.back().base < 8) {
      Cl& c = cls.back();
      c.rel[c.n] = t.first - c.base; c.id[c.n] = t.second; c.n++;
    } else {
      Cl c{}; c.base = t.first; c.n = 1; c.rel[0] = 0; c.id[0] = t.second;
      cls.push_back(c);
    }
  }
  const int ci_step = d->cin >= 128 ? 128 : 64;
  p.n_cl = static_cast<int32_t>(cls.size());
  for (int c = 0; c < p.n_cl; ++c) {
    p.c_ntap[c] = cls[c].n; p.c_base[c] = cls[c].base;
    for (int k = 0; k < cls[c].n; ++k) { p.c_rel[c * 3 + k] = cls[c].rel[k]; p.c_tap[c * 3 + k] = cls[c].id[k]; }
  }
  p.ci_step = ci_step;
  p.n_ci = (d->cin + ci_step - 1) / ci_step;
  p.n_units = (d->cout + 127) / 128 * p.n_ci * p.n_cl;     // the kernel derives (co tile, ci chunk, cluster) from the index
  p.n_kb = static_cast<int32_t>((d->rows + 127) / 128);
  int slabs = (g_num_sms + p.n_units - 1) / p.n_units;   // one wave of CTAs: split-K only as far as needed
  if (slabs > p.n_kb) slabs = p.n_kb;
  if (slabs < 1) slabs = 1;
  p.kb_per_slab = (p.n_kb + slabs - 1) / slabs;
  slabs = (p.n_kb + p.kb_per_slab - 1) / p.kb_per_slab;
  p.cout = d->cout; p.cin = d->cin; p.ntaps = d->n_taps; p.dw = d->dw; p.partials = d->partials;
  rc = encode_2d(&p.tmDY, d->dy, d->rows, d->cout, 128);
  if (rc == IDF_OK) rc = encode_2d(&p.tmX, d->x, d->x_rows, d->cin, 136);
  if (rc != IDF_OK) { delete pl; return rc; }
  pl->grid = p.n_units * slabs;
  pl->slabs = slabs;
  *out_plan = pl;
  return IDF_OK;
}

int64_t idf_wgrad_plan_partials_floats(const idf_wgrad_plan* plan) {
  if (plan == nullptr || plan->slabs < 2) return 0;
  return static_cast<int64_t>(plan->slabs) * plan->params.cout * plan->params.ntaps * plan->params.cin;
}

int idf_wgrad_plan_destroy(idf_wgrad_plan* plan) {
  delete plan;
  return IDF_OK;
}

int idf_wgrad_run(const idf_wgrad_plan* plan, idf_stream_t stream) {
  if (plan == nullptr) return fail(IDF_ERR_ARG, "null plan");
  cudaError_t e = launch_wgrad(plan->params, plan->grid, plan->slabs, g_num_sms, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "wgrad launch");
  return IDF_OK;
}

// The producers' 32-row window records of an AdaGN's sources (over this map, or over the half-resolution input grid of
// an up2 producer) must keep the images apart; otherwise the statistics have to come from the AdaGN kernel itself.
static int check_records(const idf_adagn_args* a) {
  const float* st[2] = {a->stats0, a->stats1};
  const int planes[2] = {a->stats_planes0, a->stats_planes1};
  for (int i = 0; i < 2; ++i) {
    const int H = planes[i] > 1 ? a->H / 2 : a->H, W = planes[i] > 1 ? a->W / 2 : a->W;
    if (st[i] != nullptr && !window_records_exact(H, W))
      return fail(IDF_ERR_ARG, "stats%d: 32-row GroupNorm records cannot keep the images of a %dx%d grid apart "
                  "(needs (H+1)*(W+1) >= 32 or 31 - (H+1)*(W+1) <= W+2); pass no statistics", i, H, W);
  }
  return IDF_OK;
}

int idf_adagn_coef(const idf_adagn_args* a, float* coef_out, idf_stream_t stream) {
  if (a == nullptr || coef_out == nullptr) return fail(IDF_ERR_ARG, "null argument");
  const int rc = check_records(a);
  if (rc != IDF_OK) return rc;
  cudaError_t e = launch_adagn_coef(*a, coef_out, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "adagn_coef launch (needs stats0/stats1, C <= 1024, C % 32 == 0)");
  return IDF_OK;
}

int idf_adagn_silu_fwd(const idf_adagn_args* a, idf_stream_t stream) {
  if (a == nullptr || a->src0 == nullptr || a->out == nullptr) return fail(IDF_ERR_ARG, "null argument");
  const int rc = check_records(a);
  if (rc != IDF_OK) return rc;
  cudaError_t e = launch_adagn(*a, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "adagn launch");
  return IDF_OK;
}

int64_t idf_adagn_bwd_ws_floats(int32_t batch, int32_t C) { return adagn_bwd_ws_floats(batch, C); }

int idf_adagn_silu_bwd(const idf_adagn_bwd_args* b, idf_stream_t stream) {
  if (b == nullptr) return fail(IDF_ERR_ARG, "null argument");
  if (b->f.save_coef == nullptr) {           // the statistics come from the records
    const idf_adagn_args& f = b->f;
    if (f.stats_unit0 > 32 || f.stats_unit1 > 32 || f.stats_planes0 > 1 || f.stats_planes1 > 1)
      return fail(IDF_ERR_ARG, "adagn backward: without save_coef the statistics must be 32-row window records of this map "
                  "(stats_unit 32, no up2 planes)");
    const int rc = check_records(&f);
    if (rc != IDF_OK) return rc;
  }
  cudaError_t e = launch_adagn_bwd(*b, g_num_sms, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "adagn backward launch (needs stats0/stats1, dy, dx, sums, ws; C <= 1024, C % 32 == 0)");
  return IDF_OK;
}

int idf_attn_fwd(const void* qkv, void* out, int32_t batch, int32_t H, int32_t W, int32_t d, float scale,
                 idf_stream_t stream) {
  if (qkv == nullptr || out == nullptr) return fail(IDF_ERR_ARG, "null argument");
  int rc = ensure_init();
  if (rc != IDF_OK) return rc;
  cudaError_t e;
  const int S_tok = H * W;
  if (d != 128 || (S_tok != 64 && S_tok != 256)) {
    if (S_tok <= 64 && S_tok * d <= 8192)      // small maps (e.g. 4x4): plain-FMA kernel, one CTA per sample
      e = launch_attn_small(static_cast<const bf16*>(qkv), static_cast<bf16*>(out), batch, H, W, d, scale,
                            reinterpret_cast<cudaStream_t>(stream));
    else                                       // wide heads (vanilla Diff model, d = 256 / 512): CUDA-core kernel
      e = launch_attn_generic(static_cast<const bf16*>(qkv), static_cast<bf16*>(out), batch, H, W, d, scale,
                              reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess)
      return cuda_fail(e, "attention launch (supported: d = 128 with H*W in {64, 256}; H*W <= 64 with H*W*d <= 8192; "
                          "or d % 8 == 0, d <= 1024, H*W <= 1024)");
    return IDF_OK;
  }
  CUtensorMap tm;   // TMA boxes per image row
  rc = encode_2d(&tm, qkv, static_cast<int64_t>(batch) * (H + 1) * (W + 1), 3 * d, W);
  if (rc != IDF_OK) return rc;
  e = launch_attn_v2(tm, static_cast<bf16*>(out), batch, H, W, d, scale, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "attention launch (supported: d=128, H*W in {64,256})");
  return IDF_OK;
}

int idf_attn_bwd(const void* qkv, const void* dout, void* dqkv, void* ws, int32_t batch, int32_t H, int32_t W, int32_t d,
                 float scale, idf_stream_t stream) {
  if (qkv == nullptr || dout == nullptr || dqkv == nullptr) return fail(IDF_ERR_ARG, "null argument");
  int rc = ensure_init();
  if (rc != IDF_OK) return rc;
  cudaError_t e;
  const int S_tok = H * W;
  if ((d != 128 && d != 256 && d != 512) || (S_tok != 64 && S_tok != 256)) {
    e = launch_attn_small_bwd(static_cast<const bf16*>(qkv), static_cast<const bf16*>(dout), static_cast<bf16*>(dqkv), batch,
                              H, W, d, scale, reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess)
      return cuda_fail(e, "attention backward launch (supported: d in {128,256,512} with H*W in {64,256}; "
                          "or H*W <= 64 with H*W*d <= 8192)");
    return IDF_OK;
  }
  if (ws == nullptr) return fail(IDF_ERR_ARG, "attention backward needs a workspace of idf_attn_bwd_ws_bytes()");
  const int64_t rows = static_cast<int64_t>(batch) * (H + 1) * (W + 1);
  const int64_t srows = static_cast<int64_t>(batch) * S_tok;
  bf16* P = static_cast<bf16*>(ws);
  bf16* dS = P + srows * S_tok;
  CUtensorMap tmQKV, tmDO, tmPr, tmDSr, tmDSc;
  rc = encode_2d(&tmQKV, qkv, rows, 3 * d, W);
  if (rc == IDF_OK) rc = encode_2d(&tmDO, dout, rows, d, W);
  if (rc == IDF_OK) rc = encode_2d(&tmPr, P, srows, S_tok, S_tok);
  if (rc == IDF_OK) rc = encode_2d(&tmDSr, dS, srows, S_tok, 128);
  if (rc == IDF_OK) rc = encode_2d(&tmDSc, dS, srows, S_tok, S_tok);
  if (rc != IDF_OK) return rc;
  e = launch_attn_bwd(tmQKV, tmDO, tmPr, tmDSr, tmDSc, P, dS, static_cast<bf16*>(dqkv), batch, H, W, d, scale,
                      reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "attention backward launch");
  return IDF_OK;
}

int64_t idf_attn_bwd_ws_bytes(int32_t batch, int32_t H, int32_t W) {
  return 2ll * batch * H * W * H * W * 2ll + 1024;
}

int idf_linear_f32(const float* x, int64_t ldx, const float* w, const float* b, float* y, int64_t ldy, int32_t M,
                   int32_t N, int32_t K, int32_t silu_in, idf_stream_t stream) {
  if (M <= 0 || N <= 0 || K <= 0) return fail(IDF_ERR_ARG, "bad linear shape");
  cudaError_t e = launch_linear_f32(x, ldx, w, b, y, ldy, M, N, K, silu_in, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "linear launch");
  return IDF_OK;
}

int idf_gemm_f32(const float* A, int64_t lda, int32_t transA, const float* B, int64_t ldb, int32_t transB, float* Cm,
                 int64_t ldc, int32_t M, int32_t N, int32_t K, int32_t accumulate, idf_stream_t stream) {
  if (A == nullptr || B == nullptr || Cm == nullptr || M <= 0 || N <= 0 || K <= 0) return fail(IDF_ERR_ARG, "bad gemm arguments");
  cudaError_t e = launch_gemm_f32(A, lda, transA, B, ldb, transB, Cm, ldc, M, N, K, accumulate, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "gemm_f32 launch");
  return IDF_OK;
}

int idf_gemm_f32_ordered(const float* A, int64_t lda, int32_t transA, const float* B, int64_t ldb, int32_t transB, float* Cm,
                         int64_t ldc, int32_t M, int32_t N, int32_t K, int32_t accumulate, float* ws, uint32_t* tickets,
                         idf_stream_t stream) {
  if (A == nullptr || B == nullptr || Cm == nullptr || M <= 0 || N <= 0 || K <= 0) return fail(IDF_ERR_ARG, "bad gemm arguments");
  cudaError_t e = launch_gemm_f32_ordered(A, lda, transA, B, ldb, transB, Cm, ldc, M, N, K, accumulate, ws, tickets,
                                          reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "gemm_f32 (ordered) launch (split-K shapes need ws and tickets)");
  return IDF_OK;
}

int64_t idf_gemm_f32_ws_floats(int32_t M, int32_t N, int32_t K) {
  return (M <= 0 || N <= 0 || K <= 0) ? 0 : gemm_f32_ws_floats(M, N, K);
}

int idf_gather_rows_f32(const float* table, const int64_t* idx, float* y, int32_t M, int32_t N, idf_stream_t stream) {
  cudaError_t e = launch_gather_rows(table, idx, y, M, N, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "gather launch");
  return IDF_OK;
}

int idf_clip_adamw(const idf_clip_adamw_args* a, idf_stream_t stream) {
  if (a == nullptr) return fail(IDF_ERR_ARG, "clip_adamw: null argument");
  if (a->n_chunks < 0 || (a->n_chunks > 0 && (!a->params || !a->grads || !a->exp_avg || !a->exp_avg_sq || !a->numel ||
                                              !a->chunk_tensor || !a->chunk_offset || !a->partial || !a->norm_out)))
    return fail(IDF_ERR_ARG, "clip_adamw: bad tables");
  if (a->n_chunks > 0 && a->bias_corrections == nullptr) return fail(IDF_ERR_ARG, "clip_adamw: bias_corrections table missing");
  ClipAdamWParams p;
  p.params = a->params; p.grads = a->grads; p.exp_avg = a->exp_avg; p.exp_avg_sq = a->exp_avg_sq;
  p.numel = reinterpret_cast<const long long*>(a->numel); p.chunk_tensor = a->chunk_tensor; p.chunk_offset = a->chunk_offset;
  p.n_chunks = a->n_chunks;
  p.lr = a->lr; p.beta1 = a->beta1; p.beta2 = a->beta2; p.eps = a->eps; p.weight_decay = a->weight_decay;
  p.bias_corrections = a->bias_corrections; p.max_norm = a->max_norm;
  p.partial = a->partial; p.norm_out = a->norm_out;
  cudaError_t e = launch_clip_adamw(p, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "clip_adamw launch");
  return IDF_OK;
}

int idf_to_uint8_hwc(const float* x, uint8_t* out, int32_t batch, int32_t C, int32_t H, int32_t W, idf_stream_t stream) {
  if (x == nullptr || out == nullptr) return fail(IDF_ERR_ARG, "to_uint8_hwc: null argument");
  cudaError_t e = launch_to_uint8_hwc(x, out, batch, C, H, W, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "to_uint8_hwc launch");
  return IDF_OK;
}

int idf_copy2d_f32(const float* src, int64_t lds, float* dst, int64_t ldd, int32_t M, int32_t N, idf_stream_t stream) {
  if (src == nullptr || dst == nullptr) return fail(IDF_ERR_ARG, "copy2d: null argument");
  cudaError_t e = launch_copy2d_f32(src, lds, dst, ldd, M, N, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "copy2d launch");
  return IDF_OK;
}

int idf_scale_layernorm_silu(const float* y, int64_t ldy, const float* cond, int64_t cond_row_stride,
                             int64_t cond_step_stride, const int32_t* step_ptr, const float* gamma, const float* beta,
                             float eps, float* out, int64_t ldo, int32_t M, int32_t N, int32_t apply_silu,
                             idf_stream_t stream) {
  if (y == nullptr || out == nullptr || (gamma == nullptr) != (beta == nullptr)) return fail(IDF_ERR_ARG, "scale_layernorm_silu: bad pointers");
  cudaError_t e = launch_scale_ln_silu(y, ldy, cond, cond_row_stride, cond_step_stride, step_ptr, gamma, beta, eps, out, ldo,
                                       M, N, apply_silu, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "scale_layernorm_silu launch (N <= 8192)");
  return IDF_OK;
}

int idf_gather_elems(const float* src, const int32_t* idx, const int32_t* idx2, void* dst, int64_t n, int32_t dst_bf16,
                     int32_t accumulate, idf_stream_t stream) {
  if (n < 0 || (n & 3) != 0) return fail(IDF_ERR_ARG, "gather_elems: n must be a non-negative multiple of 4");
  if (dst_bf16 && accumulate) return fail(IDF_ERR_ARG, "gather_elems: accumulation needs an fp32 destination");
  if ((reinterpret_cast<uintptr_t>(idx) | reinterpret_cast<uintptr_t>(idx2) | reinterpret_cast<uintptr_t>(dst)) & 15)
    return fail(IDF_ERR_ARG, "gather_elems: idx / dst must be 16-byte aligned");
  cudaError_t e = launch_gather_elems(src, idx, idx2, dst, n, dst_bf16 != 0, accumulate != 0, g_num_sms,
                                      reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "gather_elems launch");
  return IDF_OK;
}

int idf_im2col_head(const float* x, void* out, int32_t batch, int32_t C, int32_t H, int32_t W, idf_stream_t stream) {
  cudaError_t e = launch_im2col_head(x, static_cast<bf16*>(out), batch, C, H, W, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "im2col_head launch (needs 9*C <= 64)");
  return IDF_OK;
}

int idf_upsample2x(const void* in, void* out, int32_t batch, int32_t H, int32_t W, int32_t C, idf_stream_t stream) {
  cudaError_t e = launch_upsample2x(static_cast<const bf16*>(in), static_cast<bf16*>(out), batch, H, W, C,
                                    reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "upsample2x launch");
  return IDF_OK;
}

int idf_space_to_depth(const void* in, void* out, int32_t batch, int32_t H, int32_t W, int32_t C,
                       idf_stream_t stream) {
  cudaError_t e = launch_space_to_depth(static_cast<const bf16*>(in), static_cast<bf16*>(out), batch, H, W, C,
                                        reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "space_to_depth launch");
  return IDF_OK;
}

int idf_nchw_to_padflat(const float* x, void* out, int32_t batch, int32_t C, int32_t H, int32_t W,
                        idf_stream_t stream) {
  cudaError_t e = launch_nchw_to_padflat(x, static_cast<bf16*>(out), batch, C, H, W, C, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "nchw_to_padflat launch");
  return IDF_OK;
}

int idf_nchw_to_padflat_ld(const float* x, void* out, int32_t batch, int32_t C, int32_t H, int32_t W, int32_t ld,
                           idf_stream_t stream) {
  if (ld < C) return fail(IDF_ERR_ARG, "ld < C");
  cudaError_t e = launch_nchw_to_padflat(x, static_cast<bf16*>(out), batch, C, H, W, ld, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "nchw_to_padflat launch");
  return IDF_OK;
}

int idf_upsample2x_bwd(const void* dout, void* din, int32_t batch, int32_t H, int32_t W, int32_t C, int32_t accumulate,
                       idf_stream_t stream) {
  cudaError_t e = launch_upsample2x_bwd(static_cast<const bf16*>(dout), static_cast<bf16*>(din), batch, H, W, C, accumulate,
                                        reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "upsample2x_bwd launch");
  return IDF_OK;
}

int idf_depth_to_space(const void* dphases, void* din, int32_t batch, int32_t H, int32_t W, int32_t C, int32_t accumulate,
                       idf_stream_t stream) {
  cudaError_t e = launch_depth_to_space(static_cast<const bf16*>(dphases), static_cast<bf16*>(din), batch, H, W, C,
                                        accumulate, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "depth_to_space launch");
  return IDF_OK;
}

int idf_colsum_bf16(const void* m, float* out, int64_t rows, int32_t C, idf_stream_t stream) {
  cudaError_t e = launch_colsum(static_cast<const bf16*>(m), out, rows, C, g_num_sms, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "colsum launch");
  return IDF_OK;
}

int idf_colsum_bf16_ordered(const void* m, float* out, int64_t rows, int32_t C, float* ws, uint32_t* tickets,
                            idf_stream_t stream) {
  int rc = ensure_init();
  if (rc != IDF_OK) return rc;
  cudaError_t e = launch_colsum_ordered(static_cast<const bf16*>(m), out, rows, C, g_num_sms, ws, tickets,
                                        reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "colsum (ordered) launch");
  return IDF_OK;
}

int64_t idf_colsum_ws_floats(int64_t rows, int32_t C) {
  if (ensure_init() != IDF_OK) return 0;
  return colsum_ws_floats(rows, C, g_num_sms);
}

int idf_padflat_to_nchw(const void* in, float* y, int32_t batch, int32_t C, int32_t H, int32_t W,
                        idf_stream_t stream) {
  cudaError_t e = launch_padflat_to_nchw(static_cast<const bf16*>(in), y, batch, C, H, W, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "padflat_to_nchw launch");
  return IDF_OK;
}

int idf_sampler_update(float* x, const float* eps, const float* noise, const float* coef, const int32_t* step_ptr,
                       int64_t n, idf_stream_t stream) {
  if (x == nullptr || eps == nullptr || coef == nullptr) return fail(IDF_ERR_ARG, "null argument");
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(eps) | reinterpret_cast<uintptr_t>(noise)) & 15)
    return fail(IDF_ERR_ARG, "sampler_update needs 16-byte aligned tensors");
  cudaError_t e = launch_sampler_update(x, eps, noise, coef, step_ptr, n, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "sampler_update launch");
  return IDF_OK;
}

int idf_reparameterize_f32(const float* mu, const float* log_var, const float* noise, float* out, int64_t n,
                           idf_stream_t stream) {
  if (mu == nullptr || log_var == nullptr || noise == nullptr || out == nullptr || n < 0)
    return fail(IDF_ERR_ARG, "bad reparameterize arguments");
  cudaError_t e = launch_reparameterize(mu, log_var, noise, out, n, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "reparameterize launch");
  return IDF_OK;
}

int idf_mmd_fwd_bwd(const float* x, const float* y, float* loss, float* grad_y, int32_t B, int32_t D,
                    idf_stream_t stream) {
  if (x == nullptr || y == nullptr || loss == nullptr || B <= 0 || D <= 0 || D > 4096)
    return fail(IDF_ERR_ARG, "bad mmd arguments");
  cudaError_t e = launch_mmd(x, y, loss, grad_y, B, D, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "mmd launch");
  return IDF_OK;
}

int idf_mmd_fwd_bwd_ordered(const float* x, const float* y, float* loss, float* grad_y, int32_t B, int32_t D, float* ws,
                            uint32_t* tickets, idf_stream_t stream) {
  if (x == nullptr || y == nullptr || loss == nullptr || ws == nullptr || tickets == nullptr || B <= 0 || D <= 0 || D > 4096)
    return fail(IDF_ERR_ARG, "bad mmd arguments");
  cudaError_t e = launch_mmd_ordered(x, y, loss, grad_y, B, D, ws, tickets, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "mmd (ordered) launch");
  return IDF_OK;
}

int64_t idf_mmd_ws_floats(int32_t B) { return B > 0 ? B : 0; }

}  // extern "C"
