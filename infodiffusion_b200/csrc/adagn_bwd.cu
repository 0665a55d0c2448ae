// Backward of the fused AdaGN op (GroupNorm + affine + timestep / latent-z scale-shift + SiLU + dropout).
//
// Forward per element:  xhat = (x - mean_g) * rstd_g,  v = A_c x + B_c  with A_c = rstd_g * g_c,
// g_c = gamma_c (1+s_t)(1+s_z),  y = keep/(1-p) * silu(v).
// With dv = dy * keep/(1-p) * silu'(v):
//     S1[n,c] = sum_hw dv            S2[n,c] = sum_hw dv * xhat
//     dx = A_c dv - rstd_g / cnt * ( G1_g + xhat * G2_g ),   G1_g = sum_{c in g} g_c S1,  G2_g = sum g_c S2
// and every parameter / modulation gradient of the op is a closed form of (S1, S2) (done by the host
// side on [B, C] tensors).  Two sweeps: `stats` accumulates per-slice (S1, S2) partials, `apply` folds them
// in a fixed order (deterministic) and writes dx (optionally accumulating into an existing gradient).  The fused
// dgamma / dbeta sums over the batch are atomics, or (ordered variant, dparam_ws given) per-sample rows that the last
// sample's CTA adds in sample order.
// The forward statistics come from the producing conv's window records, as in the forward kernel.
#include "kernels.cuh"

namespace idf {

constexpr int kBT = 256;       // threads
constexpr int kBMaxC = 256;       // every InfoDiff layer
constexpr int kBMaxCWide = 1024;  // the vanilla Diff UNet (ch_mult [1,2,4,8]): 512 channels, concatenations of 768 / 1024
constexpr int kBSlices = 16;   // max row slices per sample (the launcher uses fewer for large batches / small maps)

struct AdaGNBwdParams {
  const bf16* src0; const bf16* src1;
  int c0, c1, C, Hp, Wp, H, W, R;
  const float* gamma; const float* beta; float eps;
  const float* mod_t; long long mod_t_step_stride, mod_t_batch_stride;
  const float* mod_z; long long mod_z_step_stride, mod_z_batch_stride;
  const int* step_ptr;
  int apply_silu;
  const float* stats0; const float* stats1; long long stats_b_windows;
  unsigned drop_thr16; float drop_scale; const unsigned long long* drop_seed; unsigned drop_layer;
  const bf16* dy;
  bf16* dx0; bf16* dx1; int acc0, acc1;
  const float* save_coef;
  float* sums; float* ws;
  float* d_mod_t; float* d_mod_z; float* dgamma; float* dbeta;
  int slice_rows;
  int n_slices;
  float* dparam_ws; unsigned* dparam_ticket;   // ordered dgamma / dbeta: per-sample rows summed in sample order
};

constexpr int kUn = 2;            // rows in flight per thread (more would cost occupancy: 4 CTAs/SM at <= 64 registers)
// resident CTAs per SM the register budget is sized for: 3 at <= 256 channels (80 registers, a few bytes of spills), 2 for
// the wide instantiation, which then needs no spills (its layers are the few 8x8 / 16x16 maps of the vanilla UNet)
template <int kMaxC> constexpr int kBwdMinCtas = kMaxC > kBMaxC ? 2 : 3;

// Above kBT channels the prologue sweeps the channels once (nsub == 1), so the wide instantiation keeps one row of
// `sub` and its shared state stays static (stats kernel: 24 KB here + 17 KB of s_part at 1024 channels).
template <int kMaxC>
struct BwdShared {
  float2 sub[kMaxC > kBT ? 1 : 4][kMaxC];
  float tot[2 * kMaxC];
  float mean[32], rstd[32];
  float2 ab[kMaxC];
};

// Forward statistics + folded coefficients for sample n (same arithmetic, same order as adagn_apply_kernel).
template <int kMaxC>
__device__ void bwd_prologue(const AdaGNBwdParams& p, int n, BwdShared<kMaxC>& sh) {
  const int t = threadIdx.x, C = p.C, R = p.R;
  if (p.save_coef != nullptr) {               // coefficients saved by the forward kernel
    const int cpg = C / 32;
    for (int ch = t; ch < C; ch += kBT) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(p.save_coef) + static_cast<long long>(n) * C + ch);
      sh.ab[ch] = make_float2(v.x, v.y);
      if (ch % cpg == 0) { sh.mean[ch / cpg] = v.z; sh.rstd[ch / cpg] = v.w; }
    }
    __syncthreads();
    return;
  }
  const int w_first = (n * R) / 32, w_last = ((n + 1) * R - 1) / 32;
  const bool first_straddles = (w_first * 32) < n * R;
  const int nsub = (kBT / C) > 0 ? (kBT / C) : 1;
  for (int idx = t; idx < C * nsub; idx += kBT) {
    const int ch = idx % C, sub = idx / C;
    const bool first = ch < p.c0;
    const int cs = first ? p.c0 : p.c1;
    const float2* stA = reinterpret_cast<const float2*>(first ? p.stats0 : p.stats1) + (first ? ch : ch - p.c0);
    const float2* stB = stA + p.stats_b_windows * cs;
    auto part = [&](int w) -> float2 {
      const float2* st = (w == w_first && first_straddles) ? stB : stA;
      return __ldg(st + static_cast<long long>(w) * cs);
    };
    float sx = 0.f, sq = 0.f;
    int w = w_first + sub;
    for (; w + 7 * nsub <= w_last; w += 8 * nsub) {
      const float2 v0 = part(w), v1 = part(w + nsub), v2 = part(w + 2 * nsub), v3 = part(w + 3 * nsub);
      const float2 v4 = part(w + 4 * nsub), v5 = part(w + 5 * nsub), v6 = part(w + 6 * nsub), v7 = part(w + 7 * nsub);
      sx += ((v0.x + v1.x) + (v2.x + v3.x)) + ((v4.x + v5.x) + (v6.x + v7.x));
      sq += ((v0.y + v1.y) + (v2.y + v3.y)) + ((v4.y + v5.y) + (v6.y + v7.y));
    }
    for (; w <= w_last; w += nsub) { const float2 v = part(w); sx += v.x; sq += v.y; }
    sh.sub[sub][ch] = make_float2(sx, sq);
  }
  __syncthreads();
  for (int ch = t; ch < C; ch += kBT) {
    float sx = 0.f, sq = 0.f;
    for (int sub = 0; sub < nsub; ++sub) { sx += sh.sub[sub][ch].x; sq += sh.sub[sub][ch].y; }
    sh.tot[ch] = sx; sh.tot[C + ch] = sq;
  }
  __syncthreads();
  const int cpg = C / 32;
  if (t < 32) {
    float gs = 0.f, gq = 0.f;
    for (int j = 0; j < cpg; ++j) { gs += sh.tot[t * cpg + j]; gq += sh.tot[C + t * cpg + j]; }
    const float inv_cnt = 1.0f / (static_cast<float>(cpg) * p.H * p.W);
    const float mean = gs * inv_cnt;
    const float var = fmaxf(gq * inv_cnt - mean * mean, 0.f);
    sh.mean[t] = mean; sh.rstd[t] = rsqrtf(var + p.eps);
  }
  __syncthreads();
  const int step = p.step_ptr ? *p.step_ptr : 0;
  for (int ch = t; ch < C; ch += kBT) {
    const int g = ch / cpg;
    float A = sh.rstd[g] * p.gamma[ch];
    float B = p.beta[ch] - sh.mean[g] * A;
    if (p.mod_t != nullptr) {
      const float* m = p.mod_t + step * p.mod_t_step_stride + n * p.mod_t_batch_stride;
      const float sc = 1.0f + m[ch], shf = m[C + ch];
      A *= sc; B = B * sc + shf;
    }
    if (p.mod_z != nullptr) {
      const float* m = p.mod_z + step * p.mod_z_step_stride + n * p.mod_z_batch_stride;
      const float sc = 1.0f + m[ch], shf = m[C + ch];
      A *= sc; B = B * sc + shf;
    }
    sh.ab[ch] = make_float2(A, B);
  }
  __syncthreads();
}

// dv for the 8 channels of one granule
__device__ __forceinline__ void granule_dv(const AdaGNBwdParams& p, const uint4& ux, const uint4& ud, const float (&A)[8],
                                           const float (&B)[8], uint64_t seed, uint64_t granule, float (&x)[8],
                                           float (&dv)[8]) {
  const float2 a0 = unpack_bf16x2(ux.x), a1 = unpack_bf16x2(ux.y), a2 = unpack_bf16x2(ux.z), a3 = unpack_bf16x2(ux.w);
  const float2 d0 = unpack_bf16x2(ud.x), d1 = unpack_bf16x2(ud.y), d2 = unpack_bf16x2(ud.z), d3 = unpack_bf16x2(ud.w);
  const float xs[8] = {a0.x, a0.y, a1.x, a1.y, a2.x, a2.y, a3.x, a3.y};
  const float ds[8] = {d0.x, d0.y, d1.x, d1.y, d2.x, d2.y, d3.x, d3.y};
  uint32_t keep = 0xffu;
  if (p.drop_thr16 != 0) keep = dropout_keep8(seed, p.drop_layer, granule, p.drop_thr16);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    x[j] = xs[j];
    float g = ((keep >> j) & 1u) ? ds[j] * p.drop_scale : 0.f;
    if (p.apply_silu) {
      const float v = fmaf(xs[j], A[j], B[j]);
      const float sg = 1.0f / (1.0f + __expf(-v));
      g *= sg * (1.0f + v * (1.0f - sg));
    }
    dv[j] = g;
  }
}

template <int kMaxC>
__global__ void __launch_bounds__(kBT, kBwdMinCtas<kMaxC>) adagn_bwd_stats_kernel(const AdaGNBwdParams p) {
  __shared__ BwdShared<kMaxC> sh;
  __shared__ float s_part[kBT][17];
  const int n = blockIdx.y, t = threadIdx.x, C = p.C, R = p.R;
  griddep_launch();
  griddep_wait();                 // programmatic dependent launch: all inputs come from earlier kernels
  bwd_prologue(p, n, sh);
  const int VPR = C >> 3, rpp = kBT / VPR;    // 768 channels: 2 rows per pass, threads 192..255 idle
  const bool active = t < rpp * VPR;
  const int vl = t % VPR, rsub = t / VPR, v0 = p.c0 >> 3, cpg = C / 32;
  float A[8], B[8], s1[8], s2[8];          // s2 accumulates sum dv*x; the (x - mean)*rstd form is applied at the end
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int ch = (active ? vl : 0) * 8 + j;
    A[j] = sh.ab[ch].x; B[j] = sh.ab[ch].y;
    s1[j] = 0.f; s2[j] = 0.f;
  }
  const bool from0 = vl < v0;
  const bf16* src = from0 ? (p.src0 + vl * 8) : (p.src1 + (vl - v0) * 8);
  const int pitch = from0 ? p.c0 : p.c1;
  const long long row_base = static_cast<long long>(n) * R;
  const int r_begin = blockIdx.x * p.slice_rows, r_end = min(R, r_begin + p.slice_rows);
  const float inv_wp = 1.0f / static_cast<float>(p.Wp);
  const uint64_t seed = (p.drop_thr16 != 0 && p.drop_seed != nullptr) ? *p.drop_seed : 0ull;
  if (active) {
    // kUn rows per trip, all loads issued before the arithmetic (memory-level parallelism)
    for (int rb = r_begin + rsub; rb < r_end; rb += kUn * rpp) {
      uint4 ux[kUn], ud[kUn];
      bool ok[kUn];
#pragma unroll
      for (int u = 0; u < kUn; ++u) {
        const int r = rb + u * rpp;
        const int y = __float2int_rd((static_cast<float>(r) + 0.5f) * inv_wp);
        const int xw = r - y * p.Wp;
        ok[u] = r < r_end && xw < p.W && y < p.H;
        if (ok[u]) {
          ux[u] = __ldg(reinterpret_cast<const uint4*>(src + (row_base + r) * pitch));
          ud[u] = __ldg(reinterpret_cast<const uint4*>(p.dy + (row_base + r) * C + vl * 8));
        }
      }
#pragma unroll
      for (int u = 0; u < kUn; ++u) {
        if (!ok[u]) continue;
        const int r = rb + u * rpp;
        float x[8], dv[8];
        granule_dv(p, ux[u], ud[u], A, B, seed, static_cast<uint64_t>(row_base + r) * VPR + vl, x, dv);
#pragma unroll
        for (int j = 0; j < 8; ++j) { s1[j] += dv[j]; s2[j] = fmaf(dv[j], x[j], s2[j]); }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) { s_part[t][j] = s1[j]; s_part[t][8 + j] = s2[j]; }
  __syncthreads();
  for (int i = t; i < 2 * C; i += kBT) {
    const int which = i / C, ch = i - which * C, cvl = ch >> 3, j = ch & 7;
    float acc = 0.f;
    for (int rs = 0; rs < rpp; ++rs) acc += s_part[rs * VPR + cvl][which * 8 + j];
    if (which == 1) {                       // sum dv*xhat = rstd * (sum dv*x - mean * sum dv)
      float a1 = 0.f;
      for (int rs = 0; rs < rpp; ++rs) a1 += s_part[rs * VPR + cvl][j];
      acc = (acc - sh.mean[ch / cpg] * a1) * sh.rstd[ch / cpg];
    }
    p.ws[((static_cast<long long>(n) * kBSlices + blockIdx.x) * C + ch) * 2 + which] = acc;
  }
}

template <int kMaxC, bool kOrdered>
__global__ void __launch_bounds__(kBT, kBwdMinCtas<kMaxC>) adagn_bwd_apply_kernel(const AdaGNBwdParams p) {
  __shared__ BwdShared<kMaxC> sh;
  __shared__ float s_S[2 * kMaxC];
  __shared__ float s_G[64];
  const int n = blockIdx.y, t = threadIdx.x, C = p.C, R = p.R;
  griddep_launch();
  griddep_wait();
  bwd_prologue(p, n, sh);
  const int cpg = C / 32;
  for (int i = t; i < 2 * C; i += kBT) {
    const int which = i / C, ch = i - which * C;
    float acc = 0.f;
    const float* wsp = p.ws + (static_cast<long long>(n) * kBSlices * C + ch) * 2 + which;
    for (int s0 = 0; s0 < p.n_slices; s0 += 4) {        // four independent loads per trip, fixed summation order
      float q[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) q[j] = (s0 + j < p.n_slices) ? wsp[static_cast<long long>(s0 + j) * C * 2] : 0.f;
      acc += (q[0] + q[1]) + (q[2] + q[3]);
    }
    s_S[i] = acc;
    if (blockIdx.x == 0) p.sums[(static_cast<long long>(n) * C + ch) * 2 + which] = acc;
  }
  __syncthreads();
  if (blockIdx.x == 0) {
    // closed-form gradients of gamma / beta / modulation rows from (S1, S2):
    //   v = ((xhat g + b)(1+s_t) + b_t)(1+s_z) + b_z,  q = g S2 + b S1,  T = 1+s_t,  Z = 1+s_z
    const int step = p.step_ptr ? *p.step_ptr : 0;
    const long long off_t = step * p.mod_t_step_stride + n * p.mod_t_batch_stride;
    const long long off_z = step * p.mod_z_step_stride + n * p.mod_z_batch_stride;
    for (int ch = t; ch < C; ch += kBT) {
      const float S1 = s_S[ch], S2 = s_S[C + ch];
      const float g = p.gamma[ch], b = p.beta[ch];
      const float q = g * S2 + b * S1;
      float T = 1.f, Z = 1.f, bt = 0.f;
      if (p.mod_t != nullptr) { T = 1.f + p.mod_t[off_t + ch]; bt = p.mod_t[off_t + C + ch]; }
      if (p.mod_z != nullptr) Z = 1.f + p.mod_z[off_z + ch];
      if (p.d_mod_t != nullptr) { p.d_mod_t[off_t + ch] = Z * q; p.d_mod_t[off_t + C + ch] = Z * S1; }
      if (p.d_mod_z != nullptr) { p.d_mod_z[off_z + ch] = T * q + bt * S1; p.d_mod_z[off_z + C + ch] = S1; }
      if constexpr (kOrdered) {
        p.dparam_ws[(static_cast<long long>(n) * C + ch) * 2] = T * Z * S2;
        p.dparam_ws[(static_cast<long long>(n) * C + ch) * 2 + 1] = T * Z * S1;
      } else {
        if (p.dgamma != nullptr) atomicAdd(p.dgamma + ch, T * Z * S2);
        if (p.dbeta != nullptr) atomicAdd(p.dbeta + ch, T * Z * S1);
      }
    }
    if constexpr (kOrdered) {               // the last of the batch's slice-0 CTAs adds the rows in sample order
      __shared__ bool last;
      __threadfence();
      __syncthreads();
      if (t == 0) last = atomicAdd(p.dparam_ticket, 1u) == gridDim.y - 1;
      __syncthreads();
      if (last) {
        __threadfence();
        for (int ch = t; ch < C; ch += kBT) {
          float sg = 0.f, sb = 0.f;
          for (unsigned b = 0; b < gridDim.y; ++b) {
            const float2 v = __ldcg(reinterpret_cast<const float2*>(p.dparam_ws) + static_cast<long long>(b) * C + ch);
            sg += v.x; sb += v.y;
          }
          if (p.dgamma != nullptr) p.dgamma[ch] += sg;
          if (p.dbeta != nullptr) p.dbeta[ch] += sb;
        }
        if (t == 0) *p.dparam_ticket = 0u;
      }
    }
  }
  if (t < 32) {
    float g1 = 0.f, g2 = 0.f;
    for (int j = 0; j < cpg; ++j) {
      const int ch = t * cpg + j;
      const float gc = sh.ab[ch].x / sh.rstd[t];          // effective gamma g_c = A_c / rstd_g
      g1 = fmaf(gc, s_S[ch], g1);
      g2 = fmaf(gc, s_S[C + ch], g2);
    }
    const float k = sh.rstd[t] / (static_cast<float>(cpg) * p.H * p.W);
    s_G[t] = g1 * k;
    s_G[32 + t] = g2 * k;
  }
  __syncthreads();
  const int VPR = C >> 3, rpp = kBT / VPR;
  if (t >= rpp * VPR) return;
  const int vl = t % VPR, rsub = t / VPR, v0 = p.c0 >> 3;
  float A[8], B[8], K0[8], K1[8];           // dx = A*dv - (G1 + (x - mean)*rstd*G2) = A*dv - x*K1 + K0
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int ch = vl * 8 + j, g = ch / cpg;
    A[j] = sh.ab[ch].x; B[j] = sh.ab[ch].y;
    K1[j] = sh.rstd[g] * s_G[32 + g];
    K0[j] = sh.mean[g] * K1[j] - s_G[g];
  }
  const bool from0 = vl < v0;
  const bf16* src = from0 ? (p.src0 + vl * 8) : (p.src1 + (vl - v0) * 8);
  bf16* dst = from0 ? (p.dx0 + vl * 8) : (p.dx1 + (vl - v0) * 8);
  const int acc = from0 ? p.acc0 : p.acc1;
  const int pitch = from0 ? p.c0 : p.c1;
  const long long row_base = static_cast<long long>(n) * R;
  const int r_begin = blockIdx.x * p.slice_rows, r_end = min(R, r_begin + p.slice_rows);
  const float inv_wp = 1.0f / static_cast<float>(p.Wp);
  const uint64_t seed = (p.drop_thr16 != 0 && p.drop_seed != nullptr) ? *p.drop_seed : 0ull;
  for (int rb = r_begin + rsub; rb < r_end; rb += kUn * rpp) {
    uint4 ux[kUn], ud[kUn], uo[kUn];
    bool ok[kUn];
#pragma unroll
    for (int u = 0; u < kUn; ++u) {
      const int r = rb + u * rpp;
      const int y = __float2int_rd((static_cast<float>(r) + 0.5f) * inv_wp);
      const int xw = r - y * p.Wp;
      ok[u] = r < r_end && xw < p.W && y < p.H;              // pad rows keep a zero gradient
      if (ok[u]) {
        ux[u] = __ldg(reinterpret_cast<const uint4*>(src + (row_base + r) * pitch));
        ud[u] = __ldg(reinterpret_cast<const uint4*>(p.dy + (row_base + r) * C + vl * 8));
        if (acc) uo[u] = *reinterpret_cast<const uint4*>(dst + (row_base + r) * pitch);
      }
    }
#pragma unroll
    for (int u = 0; u < kUn; ++u) {
      if (!ok[u]) continue;
      const int r = rb + u * rpp;
      float x[8], dv[8], o[8];
      granule_dv(p, ux[u], ud[u], A, B, seed, static_cast<uint64_t>(row_base + r) * VPR + vl, x, dv);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = fmaf(A[j], dv[j], fmaf(-x[j], K1[j], K0[j]));
      if (acc) {
        const uint4 e = uo[u];
        const float2 e0 = unpack_bf16x2(e.x), e1 = unpack_bf16x2(e.y), e2 = unpack_bf16x2(e.z), e3 = unpack_bf16x2(e.w);
        o[0] += e0.x; o[1] += e0.y; o[2] += e1.x; o[3] += e1.y; o[4] += e2.x; o[5] += e2.y; o[6] += e3.x; o[7] += e3.y;
      }
      uint4 w;
      w.x = pack_bf16x2(o[0], o[1]); w.y = pack_bf16x2(o[2], o[3]); w.z = pack_bf16x2(o[4], o[5]); w.w = pack_bf16x2(o[6], o[7]);
      *reinterpret_cast<uint4*>(dst + (row_base + r) * pitch) = w;
    }
  }
}

int64_t adagn_bwd_ws_floats(int batch, int C) { return static_cast<int64_t>(batch) * kBSlices * C * 2; }

cudaError_t launch_adagn_bwd(const idf_adagn_bwd_args& b, int num_sms, cudaStream_t stream) {
  const idf_adagn_args& a = b.f;
  AdaGNBwdParams p;
  p.src0 = static_cast<const bf16*>(a.src0); p.src1 = static_cast<const bf16*>(a.src1);
  p.c0 = a.c0; p.c1 = a.src1 ? a.c1 : 0; p.C = p.c0 + p.c1;
  p.H = a.H; p.W = a.W; p.Hp = a.H + 1; p.Wp = a.W + 1; p.R = p.Hp * p.Wp;
  p.gamma = a.gamma; p.beta = a.beta; p.eps = a.eps;
  p.mod_t = a.mod_t; p.mod_t_step_stride = a.mod_t_step_stride; p.mod_t_batch_stride = a.mod_t_batch_stride;
  p.mod_z = a.mod_z; p.mod_z_step_stride = a.mod_z_step_stride; p.mod_z_batch_stride = a.mod_z_batch_stride;
  p.step_ptr = a.step_ptr; p.apply_silu = a.apply_silu;
  p.stats0 = a.stats0; p.stats1 = a.stats1;
  p.stats_b_windows = (static_cast<long long>(a.batch) * p.R + kBM - 1) / kBM * 4;
  p.drop_thr16 = 0; p.drop_scale = 1.f;
  p.drop_seed = reinterpret_cast<const unsigned long long*>(a.dropout_seed); p.drop_layer = a.dropout_layer;
  if (a.dropout_p > 0.f) {
    p.drop_thr16 = static_cast<unsigned>(a.dropout_p * 65536.f + 0.5f);
    p.drop_scale = 65536.f / (65536.f - static_cast<float>(p.drop_thr16));
  }
  p.dy = static_cast<const bf16*>(b.dy);
  p.dx0 = static_cast<bf16*>(b.dx0); p.dx1 = static_cast<bf16*>(b.dx1); p.acc0 = b.acc0; p.acc1 = b.acc1;
  p.sums = b.sums; p.ws = b.ws; p.save_coef = a.save_coef;
  p.d_mod_t = b.d_mod_t; p.d_mod_z = b.d_mod_z; p.dgamma = b.dgamma; p.dbeta = b.dbeta;
  p.dparam_ws = b.dparam_ws; p.dparam_ticket = b.dparam_ticket;
  const bool ordered = p.dparam_ws != nullptr && (p.dgamma != nullptr || p.dbeta != nullptr);
  if (p.dparam_ws != nullptr && p.dparam_ticket == nullptr) return cudaErrorInvalidValue;
  if (p.C > kBMaxCWide || p.C % 32 != 0 || p.c0 % 8 != 0 || p.c1 % 8 != 0 || a.batch <= 0) return cudaErrorInvalidValue;
  if (p.stats0 == nullptr || (p.c1 != 0 && (p.stats1 == nullptr || p.dx1 == nullptr)) || p.dx0 == nullptr ||
      p.dy == nullptr || p.sums == nullptr || p.ws == nullptr)
    return cudaErrorInvalidValue;
  // one wave of CTAs (3 resident per SM), but at least 64 rows per slice
  int ns = (3 * num_sms) / a.batch;
  if (ns > kBSlices) ns = kBSlices;
  if (ns > (p.R + 63) / 64) ns = (p.R + 63) / 64;
  if (ns < 1) ns = 1;
  p.slice_rows = (p.R + ns - 1) / ns;
  p.n_slices = (p.R + p.slice_rows - 1) / p.slice_rows;
  const dim3 grid(p.n_slices, a.batch, 1);
  const bool wide = p.C > kBMaxC;
  cudaError_t e = launch_kernel(wide ? adagn_bwd_stats_kernel<kBMaxCWide> : adagn_bwd_stats_kernel<kBMaxC>, grid, dim3(kBT),
                                0, stream, g_pdl != 0, 0, p);
  if (e != cudaSuccess) return e;
  if (ordered)
    return launch_kernel(wide ? adagn_bwd_apply_kernel<kBMaxCWide, true> : adagn_bwd_apply_kernel<kBMaxC, true>, grid,
                         dim3(kBT), 0, stream, g_pdl != 0, 0, p);
  return launch_kernel(wide ? adagn_bwd_apply_kernel<kBMaxCWide, false> : adagn_bwd_apply_kernel<kBMaxC, false>, grid,
                       dim3(kBT), 0, stream, g_pdl != 0, 0, p);
}

}  // namespace idf
