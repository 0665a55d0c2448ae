// Fused single-head self-attention for the UNet's 16x16 (S=256) and 8x8 (S=64) levels, d = 128.
//
// One CTA = one sample x one tile of 128 query tokens.  The whole problem for a sample fits on chip:
//   S = Q K^T   : tcgen05.mma  M=128, N=S,   K=128   -> TMEM columns [0, S)       (fp32)
//   P = softmax : one thread per query row, straight out of TMEM (exp2, fp32), bf16 P -> shared memory
//   O = P V     : tcgen05.mma  M=128, N=128, K=S     -> TMEM columns [256, 384)   (fp32)
// Tokens of one image row are W consecutive rows of the pad-flat [rows, 3d] qkv matrix, so Q, K and V
// arrive as [W x 64] TMA boxes (one per image row and 64-wide d-chunk) straight into the K-major
// 128B-swizzled layout -- no gather instructions.  V is not transposed: it is the MN-major B operand
// of O = P V (N = d contiguous).
// Scores never leave the SM (the reference materialises [B,S,S] fp32 in HBM, modules.py:154-156).
#include "kernels.cuh"

namespace idf {

constexpr int kAttnThreads = 128;
constexpr int kD = 128;

// byte offset of 16-byte granule g (0..7) of row r inside a [rows x 64 elem] K-major SW128 tile
__device__ __forceinline__ uint32_t sw128_off(int r, int g) {
  return static_cast<uint32_t>((r >> 3) * 1024 + (r & 7) * 128 + ((g ^ (r & 7)) << 4));
}

// MN-major SW128 operand descriptor of V: LBO = distance between the two 64-wide d-chunks, SBO = 1024 B
// (8 keys); the K loop of O = P V advances 16 keys = 2048 B per MMA.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3fffu);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3fffu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3fffu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

template <int S>
__global__ void __launch_bounds__(kAttnThreads, 1)
attn_tma_kernel(const __grid_constant__ CUtensorMap tm, bf16* __restrict__ out, int Hp, int Wp, int W,
                float scale_log2e) {
  constexpr int KCH = S / 64;
  constexpr uint32_t Q_BYTES = 2 * 128 * 128;
  constexpr uint32_t KV_CHUNK = S * 128;                    // one 64-wide d-chunk of K or V: [S x 128 B]
  constexpr uint32_t K_BYTES = (2 * KV_CHUNK > KCH * 128 * 128) ? 2 * KV_CHUNK : KCH * 128 * 128;
  constexpr uint32_t V_BYTES = 2 * KV_CHUNK;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smQ = smem;
  uint8_t* smK = smQ + Q_BYTES;                    // later: P
  uint8_t* smV = smK + K_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smV + V_BYTES);   // 0: Q,K landed  1: V landed  2: S ready  3: O ready
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);

  const int t = threadIdx.x;
  const int warp = t >> 5, lane = t & 31;
  const int n = blockIdx.y;
  const int q0 = blockIdx.x * 128;
  const int img_row0 = n * Hp * Wp;
  const int H = S / W;
  const int q_rows = (S - q0 < 128) ? (S - q0) : 128;        // valid query tokens in this tile
  const int qy0 = q0 / W, q_imgrows = q_rows / W;

  if (t == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(bars + i, 1);
    fence_mbar_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  // query rows beyond S (S = 64 case) are never loaded: zero them so the MMA reads defined data
  if (q_rows < 128) {
    for (int i = t; i < (128 - q_rows) * 16; i += kAttnThreads) {
      const int r = q_rows + (i >> 4), g = i & 15;
      sts128(smem_u32(smQ) + (g >> 3) * (128 * 128) + sw128_off(r, g & 7), make_uint4(0, 0, 0, 0));
    }
    fence_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = lds32(smem_u32(tmem_slot));
  const uint32_t tmem_S = tmem_base;
  const uint32_t tmem_O = tmem_base + 256;

  if (t == 0) {
    const uint32_t box = static_cast<uint32_t>(W) * 128u;   // bytes per TMA box
    mbar_arrive_expect_tx(bars + 0, box * 2u * static_cast<uint32_t>(q_imgrows + H));
    for (int c = 0; c < 2; ++c)
      for (int y = 0; y < q_imgrows; ++y)
        tma_load_2d(smQ + c * (128 * 128) + y * box, &tm, bars + 0, c * 64, img_row0 + (qy0 + y) * Wp);
    for (int c = 0; c < 2; ++c)
      for (int y = 0; y < H; ++y)
        tma_load_2d(smK + c * KV_CHUNK + y * box, &tm, bars + 0, kD + c * 64, img_row0 + y * Wp);
    mbar_arrive_expect_tx(bars + 1, box * 2u * static_cast<uint32_t>(H));
    for (int c = 0; c < 2; ++c)
      for (int y = 0; y < H; ++y)
        tma_load_2d(smV + c * KV_CHUNK + y * box, &tm, bars + 1, 2 * kD + c * 64, img_row0 + y * Wp);
    // ---- S = Q K^T
    mbar_wait(bars + 0, 0);
    tc_fence_after();
    constexpr uint32_t idesc = umma_idesc_f16(128, S, kFmtBF16);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const uint64_t da = umma_desc_k_sw128(smem_u32(smQ + c * (128 * 128)));
      const uint64_t db = umma_desc_k_sw128(smem_u32(smK + c * KV_CHUNK));
#pragma unroll
      for (int k = 0; k < 4; ++k) umma_f16(tmem_S, da + 2 * k, db + 2 * k, idesc, (c | k) != 0 ? 1u : 0u);
    }
    umma_commit(bars + 2);
  }
  mbar_wait(bars + 2, 0);
  tc_fence_after();

  // ---- softmax: thread owns query row (warp*32 + lane) == TMEM lane
  const int row = warp * 32 + lane;
  const uint32_t lane_addr = static_cast<uint32_t>(warp * 32) << 16;
  float mx = -INFINITY;
#pragma unroll 1
  for (int c = 0; c < S / 32; ++c) {
    uint32_t v[32];
    tmem_ld_32x32(tmem_S + lane_addr + c * 32, v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(v[j]));
  }
  float sum = 0.f;
  const float mxs = mx * scale_log2e;
#pragma unroll 1
  for (int c = 0; c < S / 32; ++c) {
    uint32_t v[32];
    tmem_ld_32x32(tmem_S + lane_addr + c * 32, v);
    tmem_ld_wait();
    const uint32_t chunk = smem_u32(smK) + (c >> 1) * (128 * 128);   // P tile for keys [64*(c/2), +64)
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float e[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        e[j] = exp2f(fmaf(__uint_as_float(v[g * 8 + j]), scale_log2e, -mxs));
        sum += e[j];
      }
      uint4 o;
      o.x = pack_bf16x2(e[0], e[1]);
      o.y = pack_bf16x2(e[2], e[3]);
      o.z = pack_bf16x2(e[4], e[5]);
      o.w = pack_bf16x2(e[6], e[7]);
      sts128(chunk + sw128_off(row, (c & 1) * 4 + g), o);
    }
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  // ---- O = P V   (A = P K-major; B = V MN-major: N = d contiguous, K = keys)
  if (t == 0) {
    mbar_wait(bars + 1, 0);
    tc_fence_after();
    constexpr uint32_t idesc = umma_idesc_f16(128, kD, kFmtBF16) | (1u << 16);   // bit 16: B is MN-major
#pragma unroll
    for (int c = 0; c < KCH; ++c) {
      const uint64_t da = umma_desc_k_sw128(smem_u32(smK + c * (128 * 128)));
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int key0 = c * 64 + k * 16;
        const uint64_t db = umma_desc_mn_sw128(smem_u32(smV + key0 * 128), KV_CHUNK, 1024);
        umma_f16(tmem_O, da + 2 * k, db, idesc, (c | k) != 0 ? 1u : 0u);
      }
    }
    umma_commit(bars + 3);
  }
  mbar_wait(bars + 3, 0);
  tc_fence_after();

  const float inv = 1.0f / sum;
  const int tok = q0 + row;
  const bool valid = tok < S;
  bf16* orow = out + (valid ? (static_cast<long long>(img_row0) + (tok / W) * Wp + (tok % W)) : 0) * kD;
#pragma unroll 1
  for (int c = 0; c < kD / 32; ++c) {
    uint32_t v[32];
    tmem_ld_32x32(tmem_O + lane_addr + c * 32, v);
    tmem_ld_wait();
    if (valid) {
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint4 o;
        o.x = pack_bf16x2(__uint_as_float(v[g * 8 + 0]) * inv, __uint_as_float(v[g * 8 + 1]) * inv);
        o.y = pack_bf16x2(__uint_as_float(v[g * 8 + 2]) * inv, __uint_as_float(v[g * 8 + 3]) * inv);
        o.z = pack_bf16x2(__uint_as_float(v[g * 8 + 4]) * inv, __uint_as_float(v[g * 8 + 5]) * inv);
        o.w = pack_bf16x2(__uint_as_float(v[g * 8 + 6]) * inv, __uint_as_float(v[g * 8 + 7]) * inv);
        *reinterpret_cast<uint4*>(orow + c * 32 + g * 8) = o;
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

template <int S>
static cudaError_t launch_attn_tma(const CUtensorMap& tm, bf16* out, int batch, int H, int W, float scale,
                                   cudaStream_t stream) {
  constexpr int KCH = S / 64;
  constexpr uint32_t KV_CHUNK = S * 128;
  constexpr uint32_t K_BYTES = (2 * KV_CHUNK > KCH * 128 * 128) ? 2 * KV_CHUNK : KCH * 128 * 128;
  constexpr uint32_t SMEM = 2 * 128 * 128 + K_BYTES + 2 * KV_CHUNK + 64 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(attn_tma_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(SMEM));
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  dim3 grid((S + 127) / 128, batch, 1);
  attn_tma_kernel<S><<<grid, kAttnThreads, SMEM, stream>>>(tm, out, H + 1, W + 1, W, scale * 1.4426950408889634f);
  return cudaGetLastError();
}

cudaError_t launch_attn_v2(const CUtensorMap& tm, bf16* out, int batch, int H, int W, int d, float scale,
                           cudaStream_t stream) {
  if (d != kD) return cudaErrorInvalidValue;
  const int S = H * W;
  if (S == 256) return launch_attn_tma<256>(tm, out, batch, H, W, scale, stream);
  if (S == 64) return launch_attn_tma<64>(tm, out, batch, H, W, scale, stream);
  return cudaErrorInvalidValue;
}

// ---------------------------------------------------------------------------------------------------
// Small-map attention (S = H*W <= 64 tokens with S*d <= 8192, e.g. the 4x4 middle block of a 32x32 model):
// far too little work for the tensor-core pipeline (131 kFLOP per sample at S=16, d=128).  One CTA per sample,
// q, k, v in fp32 shared memory, scores / softmax / PV with plain FMAs.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) attn_small_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int H, int W,
                                                         int d, float scale) {
  extern __shared__ float sm[];
  const int S = H * W, n = blockIdx.x, t = threadIdx.x;
  float* q = sm;
  float* k = q + S * d;
  float* v = k + S * d;
  float* sc = v + S * d;                                  // [S][S]
  const long long img_row0 = static_cast<long long>(n) * (H + 1) * (W + 1);
  for (int i = t; i < S * 3 * d; i += 128) {
    const int tok = i / (3 * d), c = i - tok * 3 * d;
    const long long row = img_row0 + (tok / W) * (W + 1) + (tok % W);
    const float val = __bfloat162float(qkv[row * 3 * d + c]);
    (c < d ? q : (c < 2 * d ? k : v))[tok * d + (c % d)] = val;
  }
  __syncthreads();
  for (int i = t; i < S * S; i += 128) {
    const int a = i / S, b = i - a * S;
    float acc = 0.f;
    for (int c = 0; c < d; ++c) acc = fmaf(q[a * d + c], k[b * d + c], acc);
    sc[i] = acc * scale;
  }
  __syncthreads();
  for (int a = t; a < S; a += 128) {                      // softmax over each row (reference F.softmax, modules.py:156)
    float m = -INFINITY;
    for (int b = 0; b < S; ++b) m = fmaxf(m, sc[a * S + b]);
    float sum = 0.f;
    for (int b = 0; b < S; ++b) { const float e = __expf(sc[a * S + b] - m); sc[a * S + b] = e; sum += e; }
    const float inv = 1.0f / sum;
    for (int b = 0; b < S; ++b) sc[a * S + b] *= inv;
  }
  __syncthreads();
  for (int i = t; i < S * d; i += 128) {
    const int a = i / d, c = i - a * d;
    float acc = 0.f;
    for (int b = 0; b < S; ++b) acc = fmaf(sc[a * S + b], v[b * d + c], acc);
    const long long row = img_row0 + (a / W) * (W + 1) + (a % W);
    out[row * d + c] = __float2bfloat16(acc);
  }
}

cudaError_t launch_attn_small(const bf16* qkv, bf16* out, int batch, int H, int W, int d, float scale, cudaStream_t stream) {
  const int S = H * W;
  if (S > 64 || S * d > 8192 || S <= 0) return cudaErrorInvalidValue;
  const size_t smem = (3 * static_cast<size_t>(S) * d + static_cast<size_t>(S) * S) * sizeof(float);
  static size_t attr = 0;
  if (smem > attr) {
    cudaError_t e = cudaFuncSetAttribute(attn_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    attr = smem;
  }
  attn_small_kernel<<<batch, 128, smem, stream>>>(qkv, out, H, W, d, scale);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// Wide heads (d = 256 / 512: the vanilla Diff model's UNet at ch_mult [1,2,4,8], models.py:746, attention at 256 and 512
// channels).  K and V of one image do not fit next to Q in shared memory at these widths and the tensor-core kernel is
// specialised for d = 128; this CUDA-core kernel keeps the model usable (two-phase sampler, --model vanilla): one CTA
// per (image, 16 queries), scores in shared memory, K / V streamed from L2 with 16-byte loads.  Not on the measured
// InfoDiff path (whose attention is always d = 128).
// ---------------------------------------------------------------------------------------------------
constexpr int kGenQ = 16;
__global__ void __launch_bounds__(256) attn_generic_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int H, int W,
                                                           int d, float scale) {
  extern __shared__ float sm[];
  const int S = H * W, n = blockIdx.y, q0 = blockIdx.x * kGenQ, t = threadIdx.x;
  float* q = sm;                       // [kGenQ][d]
  float* sc = q + kGenQ * d;           // [kGenQ][S]
  const long long img_row0 = static_cast<long long>(n) * (H + 1) * (W + 1);
  auto prow = [&](int tok) -> long long { return img_row0 + (tok / W) * (W + 1) + (tok % W); };
  const int ld = 3 * d;
  for (int i = t; i < kGenQ * d; i += 256) {
    const int a = i / d, c = i - a * d;
    q[i] = (q0 + a < S) ? __bfloat162float(qkv[prow(q0 + a) * ld + c]) : 0.f;
  }
  __syncthreads();
  for (int j = t; j < S; j += 256) {                     // one key per thread
    const uint4* kr = reinterpret_cast<const uint4*>(qkv + prow(j) * ld + d);
    float acc[kGenQ];
#pragma unroll
    for (int a = 0; a < kGenQ; ++a) acc[a] = 0.f;
    for (int c8 = 0; c8 < d / 8; ++c8) {
      const uint4 u = __ldg(kr + c8);
      const float2 k0 = unpack_bf16x2(u.x), k1 = unpack_bf16x2(u.y), k2 = unpack_bf16x2(u.z), k3 = unpack_bf16x2(u.w);
      const float kv[8] = {k0.x, k0.y, k1.x, k1.y, k2.x, k2.y, k3.x, k3.y};
#pragma unroll
      for (int a = 0; a < kGenQ; ++a) {
        const float* qa = q + a * d + c8 * 8;
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[a] = fmaf(qa[e], kv[e], acc[a]);
      }
    }
#pragma unroll
    for (int a = 0; a < kGenQ; ++a) sc[a * S + j] = acc[a] * scale;
  }
  __syncthreads();
  {                                                      // softmax: warp w owns query rows 2w, 2w + 1
    const int warp = t >> 5, lane = t & 31;
    for (int a = 2 * warp; a < 2 * warp + 2; ++a) {
      float m = -INFINITY;
      for (int j = lane; j < S; j += 32) m = fmaxf(m, sc[a * S + j]);
      for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      float sum = 0.f;
      for (int j = lane; j < S; j += 32) { const float e = __expf(sc[a * S + j] - m); sc[a * S + j] = e; sum += e; }
      for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      const float inv = 1.0f / sum;
      for (int j = lane; j < S; j += 32) sc[a * S + j] *= inv;
    }
  }
  __syncthreads();
  for (int c = t; c < d; c += 256) {                     // one output channel per thread and pass
    float acc[kGenQ];
#pragma unroll
    for (int a = 0; a < kGenQ; ++a) acc[a] = 0.f;
    const bf16* vc = qkv + 2 * d + c;
    for (int j = 0; j < S; ++j) {
      const float vv = __bfloat162float(vc[prow(j) * ld]);
#pragma unroll
      for (int a = 0; a < kGenQ; ++a) acc[a] = fmaf(sc[a * S + j], vv, acc[a]);
    }
#pragma unroll
    for (int a = 0; a < kGenQ; ++a)
      if (q0 + a < S) out[prow(q0 + a) * d + c] = __float2bfloat16(acc[a]);
  }
}

cudaError_t launch_attn_generic(const bf16* qkv, bf16* out, int batch, int H, int W, int d, float scale, cudaStream_t stream) {
  const int S = H * W;
  if (S <= 0 || S > 1024 || d % 8 != 0 || d > 1024) return cudaErrorInvalidValue;
  const size_t smem = (static_cast<size_t>(kGenQ) * d + static_cast<size_t>(kGenQ) * S) * sizeof(float);
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  static size_t attr = 0;
  if (smem > attr) {
    cudaError_t e = cudaFuncSetAttribute(attn_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    attr = smem;
  }
  attn_generic_kernel<<<dim3((S + kGenQ - 1) / kGenQ, batch, 1), 256, smem, stream>>>(qkv, out, H, W, d, scale);
  return cudaGetLastError();
}

}  // namespace idf
