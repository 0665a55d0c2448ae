// Backward of the fused single-head self attention (reference modules.py:145-164 under autograd), on tcgen05.
//
//   S = Q K^T * scale,  P = softmax(S),  O = P V
//   dV = P^T dO        dP = dO V^T       dS = P o (dP - rowsum(P o dP)) * scale
//   dQ = dS K          dK = dS^T Q
//
// Two kernels per attention block, grid (ceil(S/128), batch), 128 threads, everything recomputed from the saved
// q | k | v matrix (nothing but qkv and O's gradient is kept from the forward):
//   1. attn_bwd_scores_kernel : per 128-query tile, S = Q K^T and dP = dO V^T (two tcgen05 GEMMs, 2 x S TMEM columns),
//      then one thread per query row straight out of TMEM: softmax statistics, D = sum_j P dP, and the bf16 rows of
//      P and dS (scale folded in) go to a [batch*S, S] workspace (L2-resident: 2 x 128 KB per image at S = 256).
//   2. attn_bwd_grads_kernel  : per 128-token tile h, three GEMMs with the accumulators side by side in TMEM:
//        dQ_h = dS[h, :] K       A = rows of dS (K-major),              B = K as MN-major operand (N = d contiguous)
//        dK_h = dS[:, h]^T Q     A = columns of dS (MN-major: the TMA box [S queries x 64 keys] IS the transposed
//        dV_h = P[:, h]^T dO         operand, like the activations in wgrad.cu), B = Q / dO MN-major
//      and one thread per token writes the bf16 row (dq | dk | dv) of the pad-flat gradient matrix.
// Splitting at the [S, S] matrices keeps every CTA's operands in shared memory (<= 192 KB) without cross-CTA
// reductions: dK / dV sum over ALL queries, which a query-tile CTA cannot do alone.
//
// Wider heads (D = 256, 512: the vanilla Diff UNet's 16x16 and 8x8 levels) reuse the D = 128 machinery:
//   * scores: S and dP reduce over d, so the kernel walks d in 128-wide chunks through the same shared-memory buffers
//     and accumulates into the same two TMEM accumulators; the next chunk's Q | K load overlaps the dP MMAs of this one;
//   * grads: grid (ceil(S/128), batch, D/128), CTA z owns the 128-wide column slice z of dQ, dK and dV (the B operands
//     K / Q / dO are read at that slice), so each CTA is the D = 128 kernel at a column offset.
// The P / dS workspace does not depend on D.
#include "kernels.cuh"

namespace idf {

namespace {
constexpr int kT = 128;     // threads
constexpr int kDh = 128;    // head width

__device__ __forceinline__ uint32_t sw128(int r, int g) {
  return static_cast<uint32_t>((r >> 3) * 1024 + (r & 7) * 128 + ((g ^ (r & 7)) << 4));
}
__device__ __forceinline__ uint64_t desc_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3fffu);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3fffu) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
}  // namespace

// ---------------------------------------------------------------------------------------------------
// kernel 1: P and dS rows of one 128-query tile
// ---------------------------------------------------------------------------------------------------
template <int S, int D>
__global__ void __launch_bounds__(kT, 1)
attn_bwd_scores_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO,
                       bf16* __restrict__ Pbuf, bf16* __restrict__ dSbuf, int Hp, int Wp, int W, float scale) {
  constexpr uint32_t QT = 2 * 128 * 128;          // a 128-row tile, two 64-wide d-chunks
  constexpr uint32_t KV_CHUNK = S * 128;          // one 64-wide d-chunk of K or V: [S x 128 B]
  constexpr int NCH = D / kDh;                    // 128-wide d chunks, one after the other through the same buffers
  constexpr int NBAR = NCH > 1 ? 5 : 3;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smQ = smem;
  uint8_t* smDO = smQ + QT;
  uint8_t* smK = smDO + QT;
  uint8_t* smV = smK + 2 * KV_CHUNK;
  // 0: Q, K landed  1: dO, V landed  2: S, dP ready  (D > 128) 3: a chunk's S MMAs have read smQ / smK, 4: its dP MMAs smDO / smV
  uint64_t* bars = reinterpret_cast<uint64_t*>(smV + 2 * KV_CHUNK);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + NBAR);

  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int n = blockIdx.y;
  const int q0 = blockIdx.x * 128;
  const int img_row0 = n * Hp * Wp;
  const int H = S / W;
  const int q_rows = (S - q0 < 128) ? (S - q0) : 128;
  const int qy0 = q0 / W, q_imgrows = q_rows / W;

  if (t == 0) {
    for (int i = 0; i < NBAR; ++i) mbar_init(bars + i, 1);
    fence_mbar_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  if (q_rows < 128) {       // S = 64: rows beyond the image are never loaded; give the MMA defined data
    for (int i = t; i < (128 - q_rows) * 16; i += kT) {
      const int r = q_rows + (i >> 4), g = i & 15;
      const uint32_t off = (g >> 3) * (128 * 128) + sw128(r, g & 7);
      sts128(smem_u32(smQ) + off, make_uint4(0, 0, 0, 0));
      sts128(smem_u32(smDO) + off, make_uint4(0, 0, 0, 0));
    }
    fence_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = lds32(smem_u32(tmem_slot));
  const uint32_t tmem_S = tmem_base, tmem_dP = tmem_base + 256;

  if (t == 0) {
    const uint32_t box = static_cast<uint32_t>(W) * 128u;
    constexpr uint32_t idesc = umma_idesc_f16(128, S, kFmtBF16);
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
      const int dc = ch * kDh;                    // first column of this d chunk
      if (ch > 0) mbar_wait(bars + 3, (ch - 1) & 1);
      mbar_arrive_expect_tx(bars + 0, box * 2u * static_cast<uint32_t>(q_imgrows + H));
      for (int c = 0; c < 2; ++c)
        for (int y = 0; y < q_imgrows; ++y)
          tma_load_2d(smQ + c * (128 * 128) + y * box, &tmQKV, bars + 0, dc + c * 64, img_row0 + (qy0 + y) * Wp);
      for (int c = 0; c < 2; ++c)
        for (int y = 0; y < H; ++y)
          tma_load_2d(smK + c * KV_CHUNK + y * box, &tmQKV, bars + 0, D + dc + c * 64, img_row0 + y * Wp);
      if (ch > 0) mbar_wait(bars + 4, (ch - 1) & 1);
      mbar_arrive_expect_tx(bars + 1, box * 2u * static_cast<uint32_t>(q_imgrows + H));
      for (int c = 0; c < 2; ++c)
        for (int y = 0; y < q_imgrows; ++y)
          tma_load_2d(smDO + c * (128 * 128) + y * box, &tmDO, bars + 1, dc + c * 64, img_row0 + (qy0 + y) * Wp);
      for (int c = 0; c < 2; ++c)
        for (int y = 0; y < H; ++y)
          tma_load_2d(smV + c * KV_CHUNK + y * box, &tmQKV, bars + 1, 2 * D + dc + c * 64, img_row0 + y * Wp);
      mbar_wait(bars + 0, ch & 1);
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < 2; ++c) {               // S = Q K^T
        const uint64_t da = umma_desc_k_sw128(smem_u32(smQ + c * (128 * 128)));
        const uint64_t db = umma_desc_k_sw128(smem_u32(smK + c * KV_CHUNK));
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16(tmem_S, da + 2 * k, db + 2 * k, idesc, (ch | c | k) != 0 ? 1u : 0u);
      }
      if (ch + 1 < NCH) umma_commit(bars + 3);
      mbar_wait(bars + 1, ch & 1);
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < 2; ++c) {               // dP = dO V^T
        const uint64_t da = umma_desc_k_sw128(smem_u32(smDO + c * (128 * 128)));
        const uint64_t db = umma_desc_k_sw128(smem_u32(smV + c * KV_CHUNK));
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16(tmem_dP, da + 2 * k, db + 2 * k, idesc, (ch | c | k) != 0 ? 1u : 0u);
      }
      if (ch + 1 < NCH) umma_commit(bars + 4);
    }
    umma_commit(bars + 2);
  }
  mbar_wait(bars + 2, 0);
  tc_fence_after();

  // ---- one thread per query row (== TMEM lane)
  const int row = warp * 32 + lane;
  const uint32_t lane_addr = static_cast<uint32_t>(warp * 32) << 16;
  const float sl2 = scale * 1.4426950408889634f;
  float mx = -INFINITY;
#pragma unroll 1
  for (int c = 0; c < S / 32; ++c) {
    uint32_t v[32];
    tmem_ld_32x32(tmem_S + lane_addr + c * 32, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(v[j]));
  }
  const float mxs = mx * sl2;
  float sum = 0.f, acc = 0.f;                     // l = sum_j e_j,  acc = sum_j e_j dP_j
#pragma unroll 1
  for (int c = 0; c < S / 32; ++c) {
    uint32_t v[32], w[32];
    tmem_ld_32x32(tmem_S + lane_addr + c * 32, v);
    tmem_ld_32x32(tmem_dP + lane_addr + c * 32, w);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float e = exp2f(fmaf(__uint_as_float(v[j]), sl2, -mxs));
      sum += e;
      acc = fmaf(e, __uint_as_float(w[j]), acc);
    }
  }
  const float inv = 1.0f / sum;
  const float Dr = acc * inv;                     // D_i = sum_j P_ij dP_ij
  const bool valid = q0 + row < S;
  const long long orow = (static_cast<long long>(n) * S + q0 + row) * S;
#pragma unroll 1
  for (int c = 0; c < S / 32; ++c) {
    uint32_t v[32], w[32];
    tmem_ld_32x32(tmem_S + lane_addr + c * 32, v);
    tmem_ld_32x32(tmem_dP + lane_addr + c * 32, w);
    tmem_ld_wait();
    if (valid) {
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float pp[8], ds[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          pp[j] = exp2f(fmaf(__uint_as_float(v[g * 8 + j]), sl2, -mxs)) * inv;
          ds[j] = pp[j] * (__uint_as_float(w[g * 8 + j]) - Dr) * scale;
        }
        uint4 o, q;
        o.x = pack_bf16x2(pp[0], pp[1]); o.y = pack_bf16x2(pp[2], pp[3]);
        o.z = pack_bf16x2(pp[4], pp[5]); o.w = pack_bf16x2(pp[6], pp[7]);
        q.x = pack_bf16x2(ds[0], ds[1]); q.y = pack_bf16x2(ds[2], ds[3]);
        q.z = pack_bf16x2(ds[4], ds[5]); q.w = pack_bf16x2(ds[6], ds[7]);
        *reinterpret_cast<uint4*>(Pbuf + orow + c * 32 + g * 8) = o;
        *reinterpret_cast<uint4*>(dSbuf + orow + c * 32 + g * 8) = q;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------------
// kernel 2: dQ, dK, dV rows of one 128-token tile
// ---------------------------------------------------------------------------------------------------
template <int S, int D>
__global__ void __launch_bounds__(kT, 1)
attn_bwd_grads_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO,
                      const __grid_constant__ CUtensorMap tmPr, const __grid_constant__ CUtensorMap tmDSr,
                      const __grid_constant__ CUtensorMap tmDSc, bf16* __restrict__ dqkv, int Hp, int Wp, int W) {
  // tmPr / tmDSc: [batch*S, S] with box {64, S rows}   (columns of P / dS: MN-major A operand, K = queries)
  // tmDSr       : [batch*S, S] with box {64, 128 rows} (rows of dS: K-major A operand, K = keys)
  constexpr int KCH = S / 64;
  constexpr uint32_t ATOM = S * 128;              // [S rows x 64 elements]
  constexpr uint32_t A_BYTES = (KCH * 128 * 128 > 2 * ATOM) ? KCH * 128 * 128 : 2 * ATOM;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smA = smem;                            // phase 1: dS rows, KCH x [128 x 128 B]; phases 2, 3: two [S x 128 B] atoms
  uint8_t* smB = smem + A_BYTES;                  // K / Q / dO: two 64-wide d atoms [S x 128 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smB + 2 * ATOM);      // 0..2: operands of phase i landed, 3..5: MMAs of phase i done
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6);

  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int n = blockIdx.y;
  const int h0 = blockIdx.x * 128;                // first token of this tile
  const int img_row0 = n * Hp * Wp;
  const int H = S / W;
  const int dc = (D == kDh) ? 0 : blockIdx.z * kDh;   // this CTA's 128-wide column slice of dQ, dK, dV

  if (t == 0) {
    for (int i = 0; i < 6; ++i) mbar_init(bars + i, 1);
    fence_mbar_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = lds32(smem_u32(tmem_slot));

  if (t == 0) {
    const uint32_t box = static_cast<uint32_t>(W) * 128u;
    auto load_tokens = [&](const CUtensorMap* tm, int col0, uint64_t* bar) {     // all S tokens of the image, 2 d-atoms
      for (int c = 0; c < 2; ++c)
        for (int y = 0; y < H; ++y) tma_load_2d(smB + c * ATOM + y * box, tm, bar, col0 + c * 64, img_row0 + y * Wp);
    };
    // ---- phase 1: dQ_h = dS[h, :] K
    mbar_arrive_expect_tx(bars + 0, KCH * 128u * 128u + 2u * ATOM);
    for (int kc = 0; kc < KCH; ++kc) tma_load_2d(smA + kc * (128 * 128), &tmDSr, bars + 0, kc * 64, n * S + h0);
    load_tokens(&tmQKV, D + dc, bars + 0);
    mbar_wait(bars + 0, 0);
    tc_fence_after();
    {
      constexpr uint32_t idesc = umma_idesc_f16(128, kDh, kFmtBF16) | (1u << 16);      // B MN-major
#pragma unroll
      for (int kc = 0; kc < KCH; ++kc) {
        const uint64_t da = umma_desc_k_sw128(smem_u32(smA + kc * (128 * 128)));
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint64_t db = desc_mn(smem_u32(smB + (kc * 64 + k * 16) * 128), ATOM);
          umma_f16(tmem_base, da + 2 * k, db, idesc, (kc | k) != 0 ? 1u : 0u);
        }
      }
      umma_commit(bars + 3);
    }
    // ---- phases 2, 3: dK_h = dS[:, h]^T Q,  dV_h = P[:, h]^T dO   (both operands MN-major, K = the S queries)
    for (int ph = 0; ph < 2; ++ph) {
      mbar_wait(bars + 3 + ph, 0);                // the previous phase's MMAs have finished reading smA / smB
      mbar_arrive_expect_tx(bars + 1 + ph, 4u * ATOM);
      for (int j = 0; j < 2; ++j)                 // columns beyond S (S = 64) are zero-filled by the TMA
        tma_load_2d(smA + j * ATOM, ph == 0 ? &tmDSc : &tmPr, bars + 1 + ph, h0 + 64 * j, n * S);
      if (ph == 0) load_tokens(&tmQKV, dc, bars + 1 + ph);
      else         load_tokens(&tmDO, dc, bars + 1 + ph);
      mbar_wait(bars + 1 + ph, 0);
      tc_fence_after();
      constexpr uint32_t idesc = umma_idesc_f16(128, kDh, kFmtBF16) | (1u << 15) | (1u << 16);
#pragma unroll
      for (int k = 0; k < S / 16; ++k) {
        const uint64_t da = desc_mn(smem_u32(smA + k * 2048), ATOM);
        const uint64_t db = desc_mn(smem_u32(smB + k * 2048), ATOM);
        umma_f16(tmem_base + 128u * (1 + ph), da, db, idesc, k != 0 ? 1u : 0u);
      }
      umma_commit(bars + 4 + ph);
    }
  }
  mbar_wait(bars + 5, 0);                         // commits complete in order: all three accumulators are final
  tc_fence_after();

  const int row = warp * 32 + lane;
  const uint32_t lane_addr = static_cast<uint32_t>(warp * 32) << 16;
  const int tok = h0 + row;
  const bool valid = tok < S;
  bf16* orow = dqkv + (valid ? (static_cast<long long>(img_row0) + (tok / W) * Wp + (tok % W)) : 0) * (3 * D);
#pragma unroll 1
  for (int c = 0; c < 3 * kDh / 32; ++c) {        // TMEM columns [0, 384) = dq | dk | dv slices, at q / k / v + dc in dqkv
    const int col = (D == kDh) ? c * 32 : (c >> 2) * D + dc + (c & 3) * 32;
    uint32_t v[32];
    tmem_ld_32x32(tmem_base + lane_addr + c * 32, v);
    tmem_ld_wait();
    if (valid) {
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint4 o;
        o.x = pack_bf16x2(__uint_as_float(v[g * 8 + 0]), __uint_as_float(v[g * 8 + 1]));
        o.y = pack_bf16x2(__uint_as_float(v[g * 8 + 2]), __uint_as_float(v[g * 8 + 3]));
        o.z = pack_bf16x2(__uint_as_float(v[g * 8 + 4]), __uint_as_float(v[g * 8 + 5]));
        o.w = pack_bf16x2(__uint_as_float(v[g * 8 + 6]), __uint_as_float(v[g * 8 + 7]));
        *reinterpret_cast<uint4*>(orow + col + g * 8) = o;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int S, int D>
static cudaError_t launch_bwd_s(const CUtensorMap& tmQKV, const CUtensorMap& tmDO, const CUtensorMap& tmPr,
                                const CUtensorMap& tmDSr, const CUtensorMap& tmDSc, bf16* P, bf16* dS, bf16* dqkv,
                                int batch, int H, int W, float scale, cudaStream_t stream) {
  constexpr uint32_t SM1 = 2 * (2 * 128 * 128) + 4 * S * 128 + 64 + 1024;
  constexpr int KCH = S / 64;
  constexpr uint32_t ATOM = S * 128;
  constexpr uint32_t A_BYTES = (KCH * 128 * 128 > 2 * ATOM) ? KCH * 128 * 128 : 2 * ATOM;
  constexpr uint32_t SM2 = A_BYTES + 2 * ATOM + 64 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(attn_bwd_scores_kernel<S, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(SM1));
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_bwd_grads_kernel<S, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(SM2));
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  dim3 grid((S + 127) / 128, batch, 1);
  attn_bwd_scores_kernel<S, D><<<grid, kT, SM1, stream>>>(tmQKV, tmDO, P, dS, H + 1, W + 1, W, scale);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  grid.z = D / kDh;
  attn_bwd_grads_kernel<S, D><<<grid, kT, SM2, stream>>>(tmQKV, tmDO, tmPr, tmDSr, tmDSc, dqkv, H + 1, W + 1, W);
  return cudaGetLastError();
}

template <int S>
static cudaError_t launch_bwd_d(const CUtensorMap& tmQKV, const CUtensorMap& tmDO, const CUtensorMap& tmPr,
                                const CUtensorMap& tmDSr, const CUtensorMap& tmDSc, bf16* P, bf16* dS, bf16* dqkv,
                                int batch, int H, int W, int d, float scale, cudaStream_t stream) {
  if (d == 128) return launch_bwd_s<S, 128>(tmQKV, tmDO, tmPr, tmDSr, tmDSc, P, dS, dqkv, batch, H, W, scale, stream);
  if (d == 256) return launch_bwd_s<S, 256>(tmQKV, tmDO, tmPr, tmDSr, tmDSc, P, dS, dqkv, batch, H, W, scale, stream);
  if (d == 512) return launch_bwd_s<S, 512>(tmQKV, tmDO, tmPr, tmDSr, tmDSc, P, dS, dqkv, batch, H, W, scale, stream);
  return cudaErrorInvalidValue;
}

cudaError_t launch_attn_bwd(const CUtensorMap& tmQKV, const CUtensorMap& tmDO, const CUtensorMap& tmPr,
                            const CUtensorMap& tmDSr, const CUtensorMap& tmDSc, bf16* P, bf16* dS, bf16* dqkv, int batch,
                            int H, int W, int d, float scale, cudaStream_t stream) {
  const int S = H * W;
  if (S == 256) return launch_bwd_d<256>(tmQKV, tmDO, tmPr, tmDSr, tmDSc, P, dS, dqkv, batch, H, W, d, scale, stream);
  if (S == 64) return launch_bwd_d<64>(tmQKV, tmDO, tmPr, tmDSr, tmDSc, P, dS, dqkv, batch, H, W, d, scale, stream);
  return cudaErrorInvalidValue;
}

// ---------------------------------------------------------------------------------------------------
// Small maps (S = H*W <= 64 with S*d <= 8192, e.g. the 4x4 middle block of a 32x32 model): one CTA per sample, fp32
// shared memory, plain FMAs -- the counterpart of attn_small_kernel.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) attn_small_bwd_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ dout,
                                                             bf16* __restrict__ dqkv, int H, int W, int d, float scale) {
  extern __shared__ float sm[];
  const int S = H * W, n = blockIdx.x, t = threadIdx.x;
  float* q = sm;
  float* k = q + S * d;
  float* v = k + S * d;
  float* go = v + S * d;
  float* p = go + S * d;                                  // [S][S]
  float* ds = p + S * S;                                  // [S][S]
  const long long img_row0 = static_cast<long long>(n) * (H + 1) * (W + 1);
  auto prow = [&](int tok) -> long long { return img_row0 + (tok / W) * (W + 1) + (tok % W); };
  for (int i = t; i < S * 3 * d; i += 128) {
    const int tok = i / (3 * d), c = i - tok * 3 * d;
    const float val = __bfloat162float(qkv[prow(tok) * 3 * d + c]);
    (c < d ? q : (c < 2 * d ? k : v))[tok * d + (c % d)] = val;
  }
  for (int i = t; i < S * d; i += 128) go[i] = __bfloat162float(dout[prow(i / d) * d + (i % d)]);
  __syncthreads();
  for (int i = t; i < S * S; i += 128) {
    const int a = i / S, b = i - a * S;
    float s = 0.f, g = 0.f;
    for (int c = 0; c < d; ++c) { s = fmaf(q[a * d + c], k[b * d + c], s); g = fmaf(go[a * d + c], v[b * d + c], g); }
    p[i] = s * scale;
    ds[i] = g;                                            // dP for now
  }
  __syncthreads();
  for (int a = t; a < S; a += 128) {
    float m = -INFINITY;
    for (int b = 0; b < S; ++b) m = fmaxf(m, p[a * S + b]);
    float sum = 0.f;
    for (int b = 0; b < S; ++b) { const float e = __expf(p[a * S + b] - m); p[a * S + b] = e; sum += e; }
    const float inv = 1.0f / sum;
    float D = 0.f;
    for (int b = 0; b < S; ++b) { p[a * S + b] *= inv; D = fmaf(p[a * S + b], ds[a * S + b], D); }
    for (int b = 0; b < S; ++b) ds[a * S + b] = p[a * S + b] * (ds[a * S + b] - D) * scale;
  }
  __syncthreads();
  for (int i = t; i < S * d; i += 128) {
    const int a = i / d, c = i - a * d;
    float dq = 0.f, dk = 0.f, dv = 0.f;
    for (int b = 0; b < S; ++b) {
      dq = fmaf(ds[a * S + b], k[b * d + c], dq);
      dk = fmaf(ds[b * S + a], q[b * d + c], dk);
      dv = fmaf(p[b * S + a], go[b * d + c], dv);
    }
    bf16* o = dqkv + prow(a) * 3 * d;
    o[c] = __float2bfloat16(dq);
    o[d + c] = __float2bfloat16(dk);
    o[2 * d + c] = __float2bfloat16(dv);
  }
}

cudaError_t launch_attn_small_bwd(const bf16* qkv, const bf16* dout, bf16* dqkv, int batch, int H, int W, int d, float scale,
                                  cudaStream_t stream) {
  const int S = H * W;
  if (S > 64 || S * d > 8192 || S <= 0) return cudaErrorInvalidValue;
  const size_t smem = (4 * static_cast<size_t>(S) * d + 2 * static_cast<size_t>(S) * S) * sizeof(float);
  static size_t attr = 0;
  if (smem > attr) {
    cudaError_t e = cudaFuncSetAttribute(attn_small_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    attr = smem;
  }
  attn_small_bwd_kernel<<<batch, 128, smem, stream>>>(qkv, dout, dqkv, H, W, d, scale);
  return cudaGetLastError();
}

}  // namespace idf
