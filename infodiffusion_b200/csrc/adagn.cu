// Fused AdaGN: GroupNorm(32) statistics + affine + timestep / latent-z scale-shift + SiLU (+ concat).
//
// v2 (smem-resident): one thread-block CLUSTER per sample (1..8 CTAs).  Each CTA pulls its contiguous
// slice of the sample's pad-flat rows into shared memory with ONE bulk-async copy per source
// (cp.async.bulk, completion on an mbarrier: no load instructions, the whole slice is in flight
// immediately), accumulates per-channel sum / sum-of-squares from shared memory, the cluster combines
// the partials through distributed shared memory (fixed order: deterministic), every CTA folds
// mean/rstd, gamma/beta and both modulations into one (A, B) pair per channel, and a second sweep over
// the slice -- still in shared memory -- applies y = silu(A*x + B) and streams bf16 to HBM with 16-byte
// coalesced stores.  HBM traffic is exactly one read + one write of the tensor.
//
// v1 re-read the slice from L2 for the second sweep and spent ~50 instructions + two integer divisions
// per 16 bytes; ncu showed it issue-bound (sm throughput 55 %, 28 % of HBM peak).
//
// Two sources (c1 > 0) are treated as one map concatenated along C, which is how the reference's
// torch.cat([h, skip]) followed by GroupNorm behaves (models.py:321 -> modules.py:265).
#include <cooperative_groups.h>

#include "kernels.cuh"

namespace cg = cooperative_groups;

namespace idf {

// ring stages per CTA and CTAs per launch of the streaming kernel.  Measured on B200 (DESIGN.md section 4.1): two
// stages (five CTAs per SM) beat three or five -- the sweep is bound by resident warps, not by bytes in flight.
constexpr int kAdaRing = 2;
constexpr int kAdaCtas = 400;

constexpr int kAdaThreads = 256;
constexpr int kMaxC = 256;
constexpr int kUnroll = 4;

struct AdaGNParams {
  const bf16* src0;
  const bf16* src1;
  bf16* out;
  int c0, c1, C;
  int Hp, Wp, H, W;
  int rows_per_img;
  int batch;
  int chunk_rows;      // rows per CTA (last CTA of the cluster may have fewer)
  const float* gamma;
  const float* beta;
  float eps;
  const float* mod_t;
  long long mod_t_step_stride, mod_t_batch_stride;
  const float* mod_z;
  long long mod_z_step_stride, mod_z_batch_stride;
  const int* step_ptr;
  int apply_silu;
  const float* stats0;   // per-tile partial sums from the producing conv (streaming variant)
  const float* stats1;
  int slice_rows;        // rows per CTA of the streaming variant
  long long stats_b_windows;   // capacity in records of the A part (offset of the B records, in records)
  int unit0, unit1;            // rows per statistics unit of stats0 / stats1: 32 (1 record per unit) or 128*MT (4 records)
  int planes0, planes1;        // record rows are planes * c columns wide (up2 producers: 4 parity planes, summed here)
  int rsrc0, rsrc1;            // pad-flat rows per image of the PRODUCER's grid (up2: the half-resolution grid)
  long long bwin0, bwin1;      // records before the B part of stats0 / stats1
  int block_rows;              // rows per ring stage of the streaming variant
  int ring;                    // ring stages in use
  unsigned drop_thr16;         // dropout: drop iff 16 random bits < thr16 (0 = off)
  float drop_scale;            // 1 / (1 - p)
  const unsigned long long* drop_seed;
  unsigned drop_layer;
  float* save_coef;            // training: [batch, C, 4] = (A, B, mean, rstd)
};

// 1-D bulk async copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__global__ void __launch_bounds__(kAdaThreads) adagn_kernel(const AdaGNParams p) {
  cg::cluster_group cluster = cg::this_cluster();
  const int CL = static_cast<int>(cluster.num_blocks());
  const int crank = static_cast<int>(cluster.block_rank());
  const int n = blockIdx.y;

  extern __shared__ __align__(128) uint8_t slice_raw[];
  __shared__ float s_part[kAdaThreads][17];   // per-thread partials: 8 sums + 8 sums of squares (+1 pad)
  __shared__ float s_cta[2 * kMaxC];          // this CTA's per-channel (sum | sumsq), read by cluster peers
  __shared__ float s_tot[2 * kMaxC];
  __shared__ float s_mean[32], s_rstd[32];
  __shared__ float2 s_ab[kMaxC];
  __shared__ __align__(8) uint64_t s_bar;

  const int C = p.C;
  const int VPR = C >> 3;                       // 16-byte vectors per (concatenated) row
  const int rpp = kAdaThreads / VPR;            // rows per pass
  const int t = threadIdx.x;
  const bool active = t < rpp * VPR;
  const int vl = t % VPR;
  const int rsub = t / VPR;
  const int v0 = p.c0 >> 3;

  const int rows = p.rows_per_img;
  const int r_begin = min(rows, crank * p.chunk_rows);
  const int r_end = min(rows, r_begin + p.chunk_rows);
  const int nrows = r_end - r_begin;
  const long long row_base = static_cast<long long>(n) * rows + r_begin;

  uint8_t* slice0 = slice_raw;
  uint8_t* slice1 = slice_raw + static_cast<size_t>(p.chunk_rows) * p.c0 * 2;

  // ---------------------------------------------------------------- bulk load of the slice
  if (t == 0) {
    mbar_init(&s_bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (t == 0) {
    const uint32_t b0 = static_cast<uint32_t>(nrows) * p.c0 * 2;
    const uint32_t b1 = static_cast<uint32_t>(nrows) * p.c1 * 2;
    mbar_arrive_expect_tx(&s_bar, b0 + b1);
    if (b0) bulk_load(slice0, p.src0 + row_base * p.c0, b0, &s_bar);
    if (b1) bulk_load(slice1, p.src1 + row_base * p.c1, b1, &s_bar);
  }
  // this thread's 16-byte column of the concatenated row, inside the smem slice
  const uint8_t* my_base = (vl < v0) ? (slice0 + vl * 16) : (slice1 + (vl - v0) * 16);
  const int my_pitch = (vl < v0) ? p.c0 * 2 : p.c1 * 2;
  mbar_wait(&s_bar, 0);

  // ---------------------------------------------------------------- sweep 1: statistics (pad rows are zeros)
  float s[8], ss[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { s[j] = 0.f; ss[j] = 0.f; }
  if (active) {
    for (int r = rsub; r < nrows; r += kUnroll * rpp) {
      uint4 u[kUnroll];
#pragma unroll
      for (int k = 0; k < kUnroll; ++k) {
        const int rr = r + k * rpp;
        u[k] = (rr < nrows) ? *reinterpret_cast<const uint4*>(my_base + static_cast<size_t>(rr) * my_pitch)
                            : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int k = 0; k < kUnroll; ++k) {
        const float2 a0 = unpack_bf16x2(u[k].x), a1 = unpack_bf16x2(u[k].y), a2 = unpack_bf16x2(u[k].z),
                     a3 = unpack_bf16x2(u[k].w);
        const float f[8] = {a0.x, a0.y, a1.x, a1.y, a2.x, a2.y, a3.x, a3.y};
#pragma unroll
        for (int j = 0; j < 8; ++j) { s[j] += f[j]; ss[j] = fmaf(f[j], f[j], ss[j]); }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) { s_part[t][j] = s[j]; s_part[t][8 + j] = ss[j]; }
  __syncthreads();
  // per-channel totals of this CTA: channel ch = cvl*8 + j lives in threads (rs*VPR + cvl), rs = 0..rpp-1
  for (int i = t; i < 2 * C; i += kAdaThreads) {
    const int which = i / C;                    // 0: sum, 1: sumsq
    const int ch = i - which * C;
    const int cvl = ch >> 3, j = ch & 7;
    float acc = 0.f;
    for (int rs = 0; rs < rpp; ++rs) acc += s_part[rs * VPR + cvl][which * 8 + j];
    s_cta[i] = acc;
  }
  cluster.sync();
  // ---------------------------------------------------------------- cluster reduction (DSMEM, fixed order)
  for (int i = t; i < 2 * C; i += kAdaThreads) {
    float acc = 0.f;
    for (int rk = 0; rk < CL; ++rk) {
      const float* remote = cluster.map_shared_rank(s_cta, rk);
      acc += remote[i];
    }
    s_tot[i] = acc;
  }
  cluster.barrier_arrive();                     // peers may exit once everyone has read; waited at the end
  __syncthreads();
  const int cpg = C / 32;
  if (t < 32) {
    float gs = 0.f, gq = 0.f;
    for (int j = 0; j < cpg; ++j) { gs += s_tot[t * cpg + j]; gq += s_tot[C + t * cpg + j]; }
    const float inv_cnt = 1.0f / (static_cast<float>(cpg) * p.H * p.W);
    const float mean = gs * inv_cnt;
    const float var = fmaxf(gq * inv_cnt - mean * mean, 0.f);
    s_mean[t] = mean;
    s_rstd[t] = rsqrtf(var + p.eps);
  }
  __syncthreads();
  const int step = p.step_ptr ? *p.step_ptr : 0;
  for (int ch = t; ch < C; ch += kAdaThreads) {
    const int g = ch / cpg;
    const float rstd = s_rstd[g], mean = s_mean[g];
    float A = rstd * p.gamma[ch];
    float B = p.beta[ch] - mean * A;
    if (p.mod_t != nullptr) {
      const float* m = p.mod_t + step * p.mod_t_step_stride + n * p.mod_t_batch_stride;
      const float sc = 1.0f + m[ch], sh = m[C + ch];
      A *= sc;
      B = B * sc + sh;
    }
    if (p.mod_z != nullptr) {
      const float* m = p.mod_z + step * p.mod_z_step_stride + n * p.mod_z_batch_stride;
      const float sc = 1.0f + m[ch], sh = m[C + ch];
      A *= sc;
      B = B * sc + sh;
    }
    s_ab[ch] = make_float2(A, B);
  }
  __syncthreads();
  // ---------------------------------------------------------------- sweep 2: normalise + activate + store
  if (active) {
    float A[8], B[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { const float2 ab = s_ab[vl * 8 + j]; A[j] = ab.x; B[j] = ab.y; }
    const bool do_silu = p.apply_silu != 0;
    // (y, x) of this thread's first row, advanced incrementally (no per-row division)
    int gy = (r_begin + rsub) / p.Wp;
    int gx = (r_begin + rsub) - gy * p.Wp;
    bf16* out_col = p.out + row_base * C + vl * 8;
    for (int r = rsub; r < nrows; r += rpp) {
      const bool interior = (gx < p.W) && (gy < p.H);       // never write pad rows
      if (interior) {
        const uint4 u = *reinterpret_cast<const uint4*>(my_base + static_cast<size_t>(r) * my_pitch);
        const float2 a0 = unpack_bf16x2(u.x), a1 = unpack_bf16x2(u.y), a2 = unpack_bf16x2(u.z), a3 = unpack_bf16x2(u.w);
        float f[8] = {a0.x, a0.y, a1.x, a1.y, a2.x, a2.y, a3.x, a3.y};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float v = fmaf(f[j], A[j], B[j]);
          f[j] = do_silu ? __fdividef(v, 1.0f + __expf(-v)) : v;
        }
        uint4 o;
        o.x = pack_bf16x2(f[0], f[1]);
        o.y = pack_bf16x2(f[2], f[3]);
        o.z = pack_bf16x2(f[4], f[5]);
        o.w = pack_bf16x2(f[6], f[7]);
        *reinterpret_cast<uint4*>(out_col + static_cast<size_t>(r) * C) = o;
      }
      gx += rpp;
      while (gx >= p.Wp) { gx -= p.Wp; ++gy; }
    }
  }
  cluster.barrier_wait();
}

// ---------------------------------------------------------------------------------------------------
// Streaming variant: the GroupNorm statistics arrive as per-tile partial sums written by the epilogue
// of the convolution that produced the tensor (conv_igemm.cu), so this kernel is a single sweep:
// fold partials -> (A, B) per channel, then y = silu(A*x + B) with 16-byte loads / stores, 4 in flight.
// No clusters, no barriers in the hot loop, one HBM read + one HBM write.
// ---------------------------------------------------------------------------------------------------
constexpr int kRingMax = 8;         // bulk-copy stages per CTA: p.ring of them are used (16 KB each)
constexpr int kRingStageBytes = 16384;

// Per-channel coefficients of image n: GroupNorm statistics from the producers' 32-row window records, folded with
// gamma / beta and the two modulations into y = A*x + B.  All kAdaThreads threads of the block take part.
// MAXC = 256 serves every layer of the InfoDiff networks; the 1024 instantiation exists for the vanilla Diff model
// (ch_mult [1,2,4,8]: GroupNorm over 512 + 512 concatenated channels) and costs 18 KB more shared memory per CTA.
constexpr int kMaxCWide = 1024;
template <int NT, int MAXC = kMaxC>
struct CoefShared {
  float2 sub[(NT > MAXC) ? NT : MAXC];   // [sub-sequence][channel], max(1, NT / C) sub-sequences of windows per channel
  float tot[2 * MAXC];
  float mean[32], rstd[32];
  float2 ab[MAXC];
};
template <int NT, int MAXC>
__device__ __forceinline__ void fold_coefficients(const AdaGNParams& p, int n, CoefShared<NT, MAXC>& sh, bool save) {
  constexpr int kAdaThreads = NT;       // all NT threads of the block take part
  const int t = threadIdx.x;
  const int C = p.C;
  const int R = p.rows_per_img;
  float2* s_sub = sh.sub;
  float (&s_tot)[2 * MAXC] = sh.tot;
  float (&s_mean)[32] = sh.mean;
  float (&s_rstd)[32] = sh.rstd;
  float2 (&s_ab)[MAXC] = sh.ab;
  // per-channel totals over the statistics records that intersect image n (units of 32 rows with one record each, or
  // of a producer work item with four; see idf_conv_desc.stats_out).  All 256 threads take part: thread -> (channel,
  // sub-sequence of records), loads issued eight at a time; the order of every addition is a function of
  // (n, geometry) only, so the result is deterministic.
  // the affine / modulation values of this thread's (first) channel do not depend on the statistics: request them
  // first, so that their global-memory latency (step counter -> modulation row: two dependent loads) hides behind the
  // record loads instead of following the three block barriers below
  const int step = p.step_ptr ? *p.step_ptr : 0;
  float pg = 0.f, pb = 0.f, pts = 0.f, pth = 0.f, pzs = 0.f, pzh = 0.f;
  if (t < C) {
    pg = __ldg(p.gamma + t); pb = __ldg(p.beta + t);
    if (p.mod_t != nullptr) {
      const float* m = p.mod_t + step * p.mod_t_step_stride + n * p.mod_t_batch_stride;
      pts = __ldg(m + t); pth = __ldg(m + C + t);
    }
    if (p.mod_z != nullptr) {
      const float* m = p.mod_z + step * p.mod_z_step_stride + n * p.mod_z_batch_stride;
      pzs = __ldg(m + t); pzh = __ldg(m + C + t);
    }
  }
  const int nsub = (kAdaThreads / C) > 0 ? (kAdaThreads / C) : 1;     // 4, 2, 1, 1 for C = 64, 128, 192, 256
  for (int idx = t; idx < C * nsub; idx += kAdaThreads) {
    const int ch = idx % C, sub = idx / C;
    const bool first = ch < p.c0;
    const int cs = first ? p.c0 : p.c1;
    const int U = first ? p.unit0 : p.unit1;
    const int P = first ? p.planes0 : p.planes1;
    const int Rs = first ? p.rsrc0 : p.rsrc1;               // rows per image on the producer's grid
    const int S = U > 32 ? 4 : 1;                           // records per unit
    const int u_first = (n * Rs) / U;
    const int u_last = ((n + 1) * Rs - 1) / U;
    const bool first_straddles = (u_first * U) < n * Rs;    // unit starts in image n-1: take its B records
    const int w_first = u_first * S, w_last = u_last * S + S - 1;
    const int w_bend = w_first + S;                         // records below belong to the first unit
    const long long rw = static_cast<long long>(P) * cs;    // record row width
    const float2* stA = reinterpret_cast<const float2*>(first ? p.stats0 : p.stats1) + (first ? ch : ch - p.c0);
    const float2* stB = stA + (first ? p.bwin0 : p.bwin1) * rw;
    // record of the first unit (B when it starts in image n-1) and of the last window; the records between lie inside
    // image n (A).  32-row windows follow window_record_of: at R < 32 either end may also hold no rows of image n (-1).
    int rec_first = first_straddles ? 1 : 0, rec_last = 0;
    if (S == 1) {
      const int last_row = p.batch * Rs - 1;
      rec_first = window_record_of(w_first, n, Rs, last_row);
      rec_last = window_record_of(w_last, n, Rs, last_row);
    }
    auto part = [&](int w) -> float2 {
      const int rec = w < w_bend ? rec_first : (w == w_last ? rec_last : 0);
      if (rec < 0) return make_float2(0.f, 0.f);
      const float2* st = (rec ? stB : stA) + static_cast<long long>(w) * rw;
      float2 v = __ldg(st);
      for (int pl = 1; pl < P; ++pl) {                      // parity planes of an up2 producer (fixed order)
        const float2 o = __ldg(st + static_cast<long long>(pl) * cs);
        v.x += o.x; v.y += o.y;
      }
      return v;
    };
    float sx = 0.f, sq = 0.f;
    int w = w_first + sub;
    for (; w + 7 * nsub <= w_last; w += 8 * nsub) {
      const float2 v0 = part(w), v1 = part(w + nsub), v2 = part(w + 2 * nsub), v3 = part(w + 3 * nsub);
      const float2 v4 = part(w + 4 * nsub), v5 = part(w + 5 * nsub), v6 = part(w + 6 * nsub), v7 = part(w + 7 * nsub);
      sx += ((v0.x + v1.x) + (v2.x + v3.x)) + ((v4.x + v5.x) + (v6.x + v7.x));
      sq += ((v0.y + v1.y) + (v2.y + v3.y)) + ((v4.y + v5.y) + (v6.y + v7.y));
    }
    for (; w <= w_last; w += nsub) {
      const float2 v = part(w);
      sx += v.x;
      sq += v.y;
    }
    s_sub[sub * C + ch] = make_float2(sx, sq);
  }
  __syncthreads();
  for (int ch = t; ch < C; ch += kAdaThreads) {
    float sx = 0.f, sq = 0.f;
    for (int sub = 0; sub < nsub; ++sub) { sx += s_sub[sub * C + ch].x; sq += s_sub[sub * C + ch].y; }
    s_tot[ch] = sx;
    s_tot[C + ch] = sq;
  }
  __syncthreads();
  const int cpg = C / 32;
  if (t < 32) {
    float gs = 0.f, gq = 0.f;
    for (int j = 0; j < cpg; ++j) { gs += s_tot[t * cpg + j]; gq += s_tot[C + t * cpg + j]; }
    const float inv_cnt = 1.0f / (static_cast<float>(cpg) * p.H * p.W);
    const float mean = gs * inv_cnt;
    const float var = fmaxf(gq * inv_cnt - mean * mean, 0.f);
    s_mean[t] = mean;
    s_rstd[t] = rsqrtf(var + p.eps);
  }
  __syncthreads();
  for (int ch = t; ch < C; ch += kAdaThreads) {
    const int g = ch / cpg;
    const bool pre = ch == t;                       // first channel of the thread: values prefetched above
    float A = s_rstd[g] * (pre ? pg : p.gamma[ch]);
    float B = (pre ? pb : p.beta[ch]) - s_mean[g] * A;
    if (p.mod_t != nullptr) {
      const float* m = p.mod_t + step * p.mod_t_step_stride + n * p.mod_t_batch_stride;
      const float sc = 1.0f + (pre ? pts : m[ch]), sh = pre ? pth : m[C + ch];
      A *= sc;
      B = B * sc + sh;
    }
    if (p.mod_z != nullptr) {
      const float* m = p.mod_z + step * p.mod_z_step_stride + n * p.mod_z_batch_stride;
      const float sc = 1.0f + (pre ? pzs : m[ch]), sh = pre ? pzh : m[C + ch];
      A *= sc;
      B = B * sc + sh;
    }
    s_ab[ch] = make_float2(A, B);
    if (p.save_coef != nullptr && save)
      reinterpret_cast<float4*>(p.save_coef)[static_cast<long long>(n) * C + ch] = make_float4(A, B, s_mean[g], s_rstd[g]);
  }
  __syncthreads();

}

// coefficients only (consumer convolution applies them to its A operand): one block per image, same thread count --
// hence the same summation order, bit for bit -- as the apply kernels' prologue
constexpr int kCoefThreads = kAdaThreads;
template <int MAXC>
__global__ void __launch_bounds__(kCoefThreads) adagn_coef_kernel(const AdaGNParams p, float2* __restrict__ coef_out) {
  __shared__ CoefShared<kCoefThreads, MAXC> sh;
  const int n = blockIdx.x;
  griddep_launch();
  griddep_wait();
  fold_coefficients<kCoefThreads, MAXC>(p, n, sh, true);
  for (int ch = threadIdx.x; ch < p.C; ch += kCoefThreads) coef_out[static_cast<long long>(n) * p.C + ch] = sh.ab[ch];
}

template <int MAXC>
__global__ void __launch_bounds__(kAdaThreads) adagn_apply_kernel(const AdaGNParams p) {
  extern __shared__ __align__(128) uint8_t ring_raw[];
  __shared__ __align__(8) uint64_t s_full[kRingMax];
  const int kRing = p.ring;
  __shared__ CoefShared<kAdaThreads, MAXC> sh;
  const int n = blockIdx.y;
  const int t = threadIdx.x;
  const int C = p.C;
  const int R = p.rows_per_img;

  // ---- start streaming the slice right away: the ring fills while the coefficients are computed
  const long long row_base = static_cast<long long>(n) * R;
  const int r_begin = blockIdx.x * p.slice_rows;
  const int r_end = min(R, r_begin + p.slice_rows);
  const int RB = p.block_rows;                                  // rows per stage
  const int nblk = (r_end - r_begin + RB - 1) / RB;
  const uint32_t stage_bytes = static_cast<uint32_t>(RB) * C * 2;
  auto issue = [&](int blk) {                                   // thread 0 only
    const int st = blk % kRing;
    const int r0 = r_begin + blk * RB;
    const int nr = min(RB, r_end - r0);
    const uint32_t b0 = static_cast<uint32_t>(nr) * p.c0 * 2, b1 = static_cast<uint32_t>(nr) * p.c1 * 2;
    mbar_arrive_expect_tx(&s_full[st], b0 + b1);
    bulk_load(ring_raw + st * stage_bytes, p.src0 + (row_base + r0) * p.c0, b0, &s_full[st]);
    if (b1) bulk_load(ring_raw + st * stage_bytes + RB * p.c0 * 2, p.src1 + (row_base + r0) * p.c1, b1, &s_full[st]);
  };
  griddep_launch();
  if (t == 0) {
    for (int i = 0; i < kRing; ++i) mbar_init(&s_full[i], 1);
    fence_mbar_init();
  }
  griddep_wait();                 // the sources, their statistics and the modulation rows come from earlier kernels
  if (t == 0) {
    for (int b = 0; b < kRing && b < nblk; ++b) issue(b);
  }

  fold_coefficients<kAdaThreads, MAXC>(p, n, sh, blockIdx.x == 0);
  const float2 (&s_ab)[MAXC] = sh.ab;

  // ---------------------------------------------------------------- streaming sweep
  // The slice is pulled through a ring of kRing shared-memory stages by bulk-async copies (one per
  // source per stage, issued by thread 0, completion on an mbarrier), so ~48-64 KB per CTA are in
  // flight regardless of register pressure; threads read 16-byte vectors from the stage, apply
  // y = silu(A*x + B) and store straight to global memory (coalesced 16-byte stores).
  const int VPR = C >> 3;
  const int rpp = kAdaThreads / VPR;
  const bool active = t < rpp * VPR;
  const int vl = t % VPR;
  const int rsub = t / VPR;
  const int v0 = p.c0 >> 3;
  const bool do_silu = p.apply_silu != 0;
  const float cs = do_silu ? 0.5f : 1.0f;       // SiLU(v) = h + h*tanh(h) with h = v/2: the 1/2 is folded into (A, B)
  float A[8], B[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { const float2 ab = s_ab[(active ? vl : 0) * 8 + j]; A[j] = ab.x * cs; B[j] = ab.y * cs; }
  const bool from0 = vl < v0;
  const uint32_t ring = smem_u32(ring_raw);
  const uint32_t my_off = (from0 ? static_cast<uint32_t>(vl * 16) : static_cast<uint32_t>(RB * p.c0 * 2 + (vl - v0) * 16)) +
                          static_cast<uint32_t>(rsub) * (from0 ? p.c0 * 2 : p.c1 * 2);
  const uint32_t it_pitch = static_cast<uint32_t>(rpp) * (from0 ? p.c0 * 2 : p.c1 * 2);   // smem bytes between my rows
  const long long out_it = static_cast<long long>(rpp) * C;                                // elements between my rows
  const float inv_wp = 1.0f / static_cast<float>(p.Wp);
  const uint64_t drop_seed = (p.drop_thr16 != 0 && p.drop_seed != nullptr) ? *p.drop_seed : 0ull;
  for (int blk = 0; blk < nblk; ++blk) {
    const int st = blk % kRing;
    mbar_wait(&s_full[st], (blk / kRing) & 1u);
    const int r0 = r_begin + blk * RB;
    const int nr = min(RB, r_end - r0);
    if (active) {
      const uint32_t base = ring + st * stage_bytes + my_off;
      bf16* const optr = p.out + (row_base + r0 + rsub) * C + vl * 8;
      // a stage holds exactly 4 * rpp rows: four rows per thread.  All four loads are issued first and the arithmetic
      // is branch-free (only the store is predicated), so the four rows overlap inside one warp.
      uint4 u[4];
      bool ok[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int lr = rsub + k * rpp;
        const int rr = r0 + lr;
        const int y = __float2int_rd((static_cast<float>(rr) + 0.5f) * inv_wp);
        const int x = rr - y * p.Wp;
        ok[k] = lr < nr && x < p.W && y < p.H;                  // beyond the slice / pad rows: never written
        u[k] = lds128(base + k * it_pitch);                     // always inside the stage
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 a0 = unpack_bf16x2(u[k].x), a1 = unpack_bf16x2(u[k].y), a2 = unpack_bf16x2(u[k].z), a3 = unpack_bf16x2(u[k].w);
        float f[8] = {a0.x, a0.y, a1.x, a1.y, a2.x, a2.y, a3.x, a3.y};
        if (do_silu) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float h = fmaf(f[j], A[j], B[j]);
            float th;
            asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(h));
            f[j] = fmaf(h, th, h);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] = fmaf(f[j], A[j], B[j]);
        }
        if (p.drop_thr16 != 0) {
          const uint32_t keep = dropout_keep8(drop_seed, p.drop_layer,
                                              static_cast<uint64_t>(row_base + r0 + rsub + k * rpp) * VPR + vl, p.drop_thr16);
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] = ((keep >> j) & 1u) ? f[j] * p.drop_scale : 0.f;
        }
        uint4 o;
        o.x = pack_bf16x2(f[0], f[1]);
        o.y = pack_bf16x2(f[2], f[3]);
        o.z = pack_bf16x2(f[4], f[5]);
        o.w = pack_bf16x2(f[6], f[7]);
        if (ok[k]) *reinterpret_cast<uint4*>(optr + k * out_it) = o;
      }
    }
    __syncthreads();                                            // everyone is done reading this stage
    if (t == 0 && blk + kRing < nblk) issue(blk + kRing);
  }
}

// c1: channels of the second source.  The coefficient kernel counts them whenever their statistics are given (the
// consumer conv reads the second source itself); the apply kernels only when there is a second source to read.
static cudaError_t fill_params(const idf_adagn_args& a, int c1, AdaGNParams& p) {
  p.src0 = static_cast<const bf16*>(a.src0);
  p.src1 = static_cast<const bf16*>(a.src1);
  p.out = static_cast<bf16*>(a.out);
  p.c0 = a.c0;
  p.c1 = c1;
  p.C = p.c0 + p.c1;
  p.H = a.H; p.W = a.W; p.Hp = a.H + 1; p.Wp = a.W + 1;
  p.rows_per_img = p.Hp * p.Wp;
  p.batch = a.batch;
  p.gamma = a.gamma; p.beta = a.beta; p.eps = a.eps;
  p.mod_t = a.mod_t; p.mod_t_step_stride = a.mod_t_step_stride; p.mod_t_batch_stride = a.mod_t_batch_stride;
  p.mod_z = a.mod_z; p.mod_z_step_stride = a.mod_z_step_stride; p.mod_z_batch_stride = a.mod_z_batch_stride;
  p.step_ptr = a.step_ptr;
  p.apply_silu = a.apply_silu;
  if (p.C > kMaxCWide || p.C % 32 != 0 || p.c0 % 8 != 0 || p.c1 % 8 != 0 || a.batch <= 0) return cudaErrorInvalidValue;
  p.stats0 = a.stats0;
  p.stats1 = a.stats1;
  p.slice_rows = 0;
  p.drop_thr16 = 0; p.drop_scale = 1.f; p.drop_seed = reinterpret_cast<const unsigned long long*>(a.dropout_seed);
  p.drop_layer = a.dropout_layer;
  p.save_coef = a.save_coef;
  p.stats_b_windows = (static_cast<long long>(a.batch) * p.rows_per_img + kBM - 1) / kBM * 4;
  p.unit0 = a.stats_unit0 > 0 ? a.stats_unit0 : 32;
  p.unit1 = a.stats_unit1 > 0 ? a.stats_unit1 : 32;
  p.planes0 = a.stats_planes0 > 0 ? a.stats_planes0 : 1;
  p.planes1 = a.stats_planes1 > 0 ? a.stats_planes1 : 1;
  p.rsrc0 = a.stats_rows0 > 0 ? a.stats_rows0 : p.rows_per_img;
  p.rsrc1 = a.stats_rows1 > 0 ? a.stats_rows1 : p.rows_per_img;
  p.bwin0 = (static_cast<long long>(a.batch) * p.rsrc0 + kBM - 1) / kBM * 4;
  p.bwin1 = (static_cast<long long>(a.batch) * p.rsrc1 + kBM - 1) / kBM * 4;
  if ((p.unit0 > 32 && p.unit0 > p.rsrc0) || (p.unit1 > 32 && p.unit1 > p.rsrc1)) return cudaErrorInvalidValue;   // a unit spans <= 2 images
  return cudaSuccess;
}

cudaError_t launch_adagn_coef(const idf_adagn_args& a, float* coef_out, cudaStream_t stream) {
  AdaGNParams p;
  cudaError_t e = fill_params(a, (a.src1 || a.stats1) ? a.c1 : 0, p);
  if (e != cudaSuccess) return e;
  if (p.stats0 == nullptr || (p.c1 != 0 && p.stats1 == nullptr) || a.dropout_p > 0.f) return cudaErrorInvalidValue;
  p.save_coef = nullptr;
  return launch_kernel(p.C <= kMaxC ? adagn_coef_kernel<kMaxC> : adagn_coef_kernel<kMaxCWide>, dim3(a.batch),
                       dim3(kCoefThreads), 0, stream, g_pdl != 0, 0, p, reinterpret_cast<float2*>(coef_out));
}

cudaError_t launch_adagn(const idf_adagn_args& a, cudaStream_t stream) {
  AdaGNParams p;
  cudaError_t e = fill_params(a, a.src1 ? a.c1 : 0, p);
  if (e != cudaSuccess) return e;
  if (a.dropout_p > 0.f) {
    if (a.stats0 == nullptr) return cudaErrorInvalidValue;     // dropout lives in the streaming variant only
    p.drop_thr16 = static_cast<unsigned>(a.dropout_p * 65536.f + 0.5f);
    p.drop_scale = 65536.f / (65536.f - static_cast<float>(p.drop_thr16));
  }
  if (p.stats0 != nullptr && (p.c1 == 0 || p.stats1 != nullptr)) {
    // streaming variant: bytes in flight come from the per-CTA ring, not from occupancy, so a few hundred
    // CTAs suffice; large slices amortise the per-CTA coefficient prologue
    const long long bytes_s = static_cast<long long>(p.rows_per_img) * p.C * 2;
    const int max_slices = static_cast<int>((bytes_s + 32767) / 32768);
    int slices = (kAdaCtas + a.batch - 1) / a.batch;
    if (slices > max_slices) slices = max_slices;
    if (slices < 1) slices = 1;
    p.slice_rows = (p.rows_per_img + slices - 1) / slices;
    slices = (p.rows_per_img + p.slice_rows - 1) / p.slice_rows;
    p.block_rows = 4 * (kAdaThreads / (p.C / 8));            // four rows per thread and stage (<= 16 KB)
    p.ring = kAdaRing;
    const size_t ring_bytes = static_cast<size_t>(p.ring) * p.block_rows * p.C * 2;
    static bool attr_set = false;
    if (!attr_set) {
      e = cudaFuncSetAttribute(adagn_apply_kernel<kMaxC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               kRingMax * kRingStageBytes);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(adagn_apply_kernel<kMaxCWide>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 kRingMax * kRingStageBytes);
      if (e != cudaSuccess) return e;
      attr_set = true;
    }
    return launch_kernel(p.C > kMaxC ? adagn_apply_kernel<kMaxCWide> : adagn_apply_kernel<kMaxC>,
                         dim3(slices, a.batch, 1), dim3(kAdaThreads), ring_bytes, stream, g_pdl != 0, 0, p);
  }

  if (p.C > kMaxC) return cudaErrorInvalidValue;       // the two-sweep fallback (no producer statistics) serves <= 256 channels
  // cluster size: slices of <= ~72 KB (3 CTAs per SM) when possible, at most 8 CTAs (portable limit)
  const long long bytes = static_cast<long long>(p.rows_per_img) * p.C * 2;
  int CL = 1;
  while (CL < 8 && bytes > static_cast<long long>(CL) * 72 * 1024) CL <<= 1;
  p.chunk_rows = (p.rows_per_img + CL - 1) / CL;
  const size_t smem = static_cast<size_t>(p.chunk_rows) * p.C * 2;
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  static size_t attr_smem = 0;
  if (smem > attr_smem) {
    e = cudaFuncSetAttribute(adagn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    attr_smem = smem;
  }
  return launch_kernel(adagn_kernel, dim3(CL, a.batch, 1), dim3(kAdaThreads), smem, stream, false, CL, p);
}

}  // namespace idf
