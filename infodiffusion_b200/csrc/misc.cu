// HBM-bound helper kernels: layout conversion, head im2col, nearest upsample, space-to-depth,
// stand-alone sampler update, small fp32 linears and the fused MMD loss.
#include "kernels.cuh"

namespace idf {

// ----------------------------------------------------------------------------------------------
// head im2col: x NCHW fp32 [B,C,H,W] -> bf16 pad-flat [rows, 64], k = tap*C + c for 3x3/pad 1
// one thread = one interior pixel x one 16-byte granule (8 k's)
// ----------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(256) im2col_head_kernel(const float* __restrict__ x, bf16* __restrict__ out,
                                                          int batch, int H, int W) {
  // one thread = one pixel: 9*C neighbour loads (coalesced along x across the warp), one 128-byte row out
  const long long total = static_cast<long long>(batch) * H * W;
  const long long pix = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (pix >= total) return;
  const int px = static_cast<int>(pix % W);
  const int py = static_cast<int>((pix / W) % H);
  const int n = static_cast<int>(pix / (static_cast<long long>(W) * H));
  const float* xn = x + static_cast<long long>(n) * C * H * W;
  uint32_t packed[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) packed[i] = 0u;
  float vals[9 * C + 1];
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const int yy = py + tap / 3 - 1, xx = px + tap % 3 - 1;
    const bool in = (yy >= 0) && (yy < H) && (xx >= 0) && (xx < W);
#pragma unroll
    for (int c = 0; c < C; ++c)
      vals[tap * C + c] = in ? __ldg(xn + (static_cast<long long>(c) * H + yy) * W + xx) : 0.f;
  }
  vals[9 * C] = 0.f;
#pragma unroll
  for (int k = 0; k < (9 * C + 1) / 2; ++k) packed[k] = pack_bf16x2(vals[2 * k], vals[2 * k + 1]);
  const long long row = (static_cast<long long>(n) * (H + 1) + py) * (W + 1) + px;
  uint4* o = reinterpret_cast<uint4*>(out + row * 64);
#pragma unroll
  for (int g = 0; g < 8; ++g) o[g] = make_uint4(packed[4 * g], packed[4 * g + 1], packed[4 * g + 2], packed[4 * g + 3]);
}

cudaError_t launch_im2col_head(const float* x, bf16* out, int batch, int C, int H, int W, cudaStream_t stream) {
  const long long total = static_cast<long long>(batch) * H * W;
  const unsigned grid = static_cast<unsigned>((total + 255) / 256);
  switch (C) {
    case 1: im2col_head_kernel<1><<<grid, 256, 0, stream>>>(x, out, batch, H, W); break;
    case 2: im2col_head_kernel<2><<<grid, 256, 0, stream>>>(x, out, batch, H, W); break;
    case 3: im2col_head_kernel<3><<<grid, 256, 0, stream>>>(x, out, batch, H, W); break;
    case 4: im2col_head_kernel<4><<<grid, 256, 0, stream>>>(x, out, batch, H, W); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------
// nearest x2 upsample, pad-flat bf16: one thread = one OUTPUT pixel x one 16-byte granule
// ----------------------------------------------------------------------------------------------
__global__ void upsample2x_kernel(const bf16* __restrict__ in, bf16* __restrict__ out, int batch, int H, int W,
                                  int C) {
  const int V = C >> 3;
  const int Ho = 2 * H, Wo = 2 * W;
  const long long total = static_cast<long long>(batch) * Ho * Wo * V;
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i >= total) return;
  const int v = static_cast<int>(i % V);
  const long long pix = i / V;
  const int ox = static_cast<int>(pix % Wo);
  const int oy = static_cast<int>((pix / Wo) % Ho);
  const int n = static_cast<int>(pix / (static_cast<long long>(Wo) * Ho));
  const long long rin = (static_cast<long long>(n) * (H + 1) + (oy >> 1)) * (W + 1) + (ox >> 1);
  const long long rout = (static_cast<long long>(n) * (Ho + 1) + oy) * (Wo + 1) + ox;
  *reinterpret_cast<uint4*>(out + rout * C + v * 8) = __ldg(reinterpret_cast<const uint4*>(in + rin * C + v * 8));
}

cudaError_t launch_upsample2x(const bf16* in, bf16* out, int batch, int H, int W, int C, cudaStream_t stream) {
  if (C % 8) return cudaErrorInvalidValue;
  const long long total = static_cast<long long>(batch) * 4 * H * W * (C >> 3);
  upsample2x_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(in, out, batch, H, W, C);
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------
// space-to-depth: in [B,H,W,C] -> out[phase=py*2+px][B,H/2,W/2,C] (each phase pad-flat)
// ----------------------------------------------------------------------------------------------
__global__ void space_to_depth_kernel(const bf16* __restrict__ in, bf16* __restrict__ out, int batch, int H, int W,
                                      int C) {
  const int V = C >> 3;
  const long long total = static_cast<long long>(batch) * H * W * V;
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i >= total) return;
  const int v = static_cast<int>(i % V);
  const long long pix = i / V;
  const int x = static_cast<int>(pix % W);
  const int y = static_cast<int>((pix / W) % H);
  const int n = static_cast<int>(pix / (static_cast<long long>(W) * H));
  const int Ho = H >> 1, Wo = W >> 1;
  const long long rows_o = static_cast<long long>(batch) * (Ho + 1) * (Wo + 1);
  const int phase = (y & 1) * 2 + (x & 1);
  const long long rin = (static_cast<long long>(n) * (H + 1) + y) * (W + 1) + x;
  const long long rout = phase * rows_o + (static_cast<long long>(n) * (Ho + 1) + (y >> 1)) * (Wo + 1) + (x >> 1);
  *reinterpret_cast<uint4*>(out + rout * C + v * 8) = __ldg(reinterpret_cast<const uint4*>(in + rin * C + v * 8));
}

cudaError_t launch_space_to_depth(const bf16* in, bf16* out, int batch, int H, int W, int C, cudaStream_t stream) {
  if ((C % 8) || (H & 1) || (W & 1)) return cudaErrorInvalidValue;
  const long long total = static_cast<long long>(batch) * H * W * (C >> 3);
  space_to_depth_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(in, out, batch, H, W, C);
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------
// NCHW fp32 <-> pad-flat bf16 (boundary / test helpers).  Tiled through shared memory so that both
// sides are coalesced: a tile is 32 pixels (along W) x 32 channels.
// ----------------------------------------------------------------------------------------------
__global__ void nchw_to_padflat_kernel(const float* __restrict__ x, bf16* __restrict__ out, int C, int H, int W, int ld) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const int c0 = blockIdx.y * 32;
  const long long p0 = static_cast<long long>(blockIdx.x) * 32;   // pixel index y*W+x
  const long long HW = static_cast<long long>(H) * W;
  const int tx = threadIdx.x, ty = threadIdx.y;                  // 32 x 8
  for (int j = ty; j < 32; j += 8) {
    const int c = c0 + j;
    const long long p = p0 + tx;
    tile[j][tx] = (c < C && p < HW) ? x[(static_cast<long long>(n) * C + c) * HW + p] : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const long long p = p0 + j;
    const int c = c0 + tx;
    if (p < HW && c < C) {
      const int yy = static_cast<int>(p / W), xx = static_cast<int>(p % W);
      const long long row = (static_cast<long long>(n) * (H + 1) + yy) * (W + 1) + xx;
      out[row * ld + c] = __float2bfloat16(tile[tx][j]);
    }
  }
}
__global__ void padflat_to_nchw_kernel(const bf16* __restrict__ in, float* __restrict__ y, int C, int H, int W) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const int c0 = blockIdx.y * 32;
  const long long p0 = static_cast<long long>(blockIdx.x) * 32;
  const long long HW = static_cast<long long>(H) * W;
  const int tx = threadIdx.x, ty = threadIdx.y;
  for (int j = ty; j < 32; j += 8) {
    const long long p = p0 + j;
    const int c = c0 + tx;
    float v = 0.f;
    if (p < HW && c < C) {
      const int yy = static_cast<int>(p / W), xx = static_cast<int>(p % W);
      const long long row = (static_cast<long long>(n) * (H + 1) + yy) * (W + 1) + xx;
      v = __bfloat162float(in[row * C + c]);
    }
    tile[j][tx] = v;   // [pixel][channel]
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const int c = c0 + j;
    const long long p = p0 + tx;
    if (c < C && p < HW) y[(static_cast<long long>(n) * C + c) * HW + p] = tile[tx][j];
  }
}

cudaError_t launch_nchw_to_padflat(const float* x, bf16* out, int batch, int C, int H, int W, int ld,
                                   cudaStream_t stream) {
  dim3 grid(static_cast<unsigned>((static_cast<long long>(H) * W + 31) / 32), (C + 31) / 32, batch);
  nchw_to_padflat_kernel<<<grid, dim3(32, 8), 0, stream>>>(x, out, C, H, W, ld);
  return cudaGetLastError();
}
cudaError_t launch_padflat_to_nchw(const bf16* in, float* y, int batch, int C, int H, int W, cudaStream_t stream) {
  dim3 grid(static_cast<unsigned>((static_cast<long long>(H) * W + 31) / 32), (C + 31) / 32, batch);
  padflat_to_nchw_kernel<<<grid, dim3(32, 8), 0, stream>>>(in, y, C, H, W);
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------
// backward helpers of the layout ops (training)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 add_bf16x8(const uint4& a, const uint4& b) {
  const float2 a0 = unpack_bf16x2(a.x), a1 = unpack_bf16x2(a.y), a2 = unpack_bf16x2(a.z), a3 = unpack_bf16x2(a.w);
  const float2 b0 = unpack_bf16x2(b.x), b1 = unpack_bf16x2(b.y), b2 = unpack_bf16x2(b.z), b3 = unpack_bf16x2(b.w);
  uint4 o;
  o.x = pack_bf16x2(a0.x + b0.x, a0.y + b0.y);
  o.y = pack_bf16x2(a1.x + b1.x, a1.y + b1.y);
  o.z = pack_bf16x2(a2.x + b2.x, a2.y + b2.y);
  o.w = pack_bf16x2(a3.x + b3.x, a3.y + b3.y);
  return o;
}

// d(nearest x2 upsample): din[n,y,x] (+)= sum_{a,b} dout[n, 2y+a, 2x+b]; one thread = one INPUT pixel x granule
__global__ void upsample2x_bwd_kernel(const bf16* __restrict__ dout, bf16* __restrict__ din, int batch, int H, int W,
                                      int C, int accumulate) {
  const int V = C >> 3;
  const long long total = static_cast<long long>(batch) * H * W * V;
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i >= total) return;
  const int v = static_cast<int>(i % V);
  const long long pix = i / V;
  const int x = static_cast<int>(pix % W);
  const int y = static_cast<int>((pix / W) % H);
  const int n = static_cast<int>(pix / (static_cast<long long>(W) * H));
  const int Ho = 2 * H, Wo = 2 * W;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const long long ro = (static_cast<long long>(n) * (Ho + 1) + 2 * y + a) * (Wo + 1) + 2 * x + b;
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(dout + ro * C + v * 8));
      const float2 f0 = unpack_bf16x2(u.x), f1 = unpack_bf16x2(u.y), f2 = unpack_bf16x2(u.z), f3 = unpack_bf16x2(u.w);
      acc[0] += f0.x; acc[1] += f0.y; acc[2] += f1.x; acc[3] += f1.y; acc[4] += f2.x; acc[5] += f2.y; acc[6] += f3.x; acc[7] += f3.y;
    }
  const long long ri = (static_cast<long long>(n) * (H + 1) + y) * (W + 1) + x;
  uint4* dst = reinterpret_cast<uint4*>(din + ri * C + v * 8);
  uint4 o;
  o.x = pack_bf16x2(acc[0], acc[1]); o.y = pack_bf16x2(acc[2], acc[3]); o.z = pack_bf16x2(acc[4], acc[5]); o.w = pack_bf16x2(acc[6], acc[7]);
  *dst = accumulate ? add_bf16x8(*dst, o) : o;
}
cudaError_t launch_upsample2x_bwd(const bf16* dout, bf16* din, int batch, int H, int W, int C, int accumulate,
                                  cudaStream_t stream) {
  if (C % 8) return cudaErrorInvalidValue;
  const long long total = static_cast<long long>(batch) * H * W * (C >> 3);
  upsample2x_bwd_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(dout, din, batch, H, W, C, accumulate);
  return cudaGetLastError();
}

// inverse of space_to_depth: din[n,y,x] (+)= dphase[(y&1)*2+(x&1)][n, y/2, x/2]
__global__ void depth_to_space_kernel(const bf16* __restrict__ dph, bf16* __restrict__ din, int batch, int H, int W,
                                      int C, int accumulate) {
  const int V = C >> 3;
  const long long total = static_cast<long long>(batch) * H * W * V;
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i >= total) return;
  const int v = static_cast<int>(i % V);
  const long long pix = i / V;
  const int x = static_cast<int>(pix % W);
  const int y = static_cast<int>((pix / W) % H);
  const int n = static_cast<int>(pix / (static_cast<long long>(W) * H));
  const int Ho = H >> 1, Wo = W >> 1;
  const long long rows_o = static_cast<long long>(batch) * (Ho + 1) * (Wo + 1);
  const int phase = (y & 1) * 2 + (x & 1);
  const long long rp = phase * rows_o + (static_cast<long long>(n) * (Ho + 1) + (y >> 1)) * (Wo + 1) + (x >> 1);
  const long long ri = (static_cast<long long>(n) * (H + 1) + y) * (W + 1) + x;
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(dph + rp * C + v * 8));
  uint4* dst = reinterpret_cast<uint4*>(din + ri * C + v * 8);
  *dst = accumulate ? add_bf16x8(*dst, u) : u;
}
cudaError_t launch_depth_to_space(const bf16* dph, bf16* din, int batch, int H, int W, int C, int accumulate,
                                  cudaStream_t stream) {
  if ((C % 8) || (H & 1) || (W & 1)) return cudaErrorInvalidValue;
  const long long total = static_cast<long long>(batch) * H * W * (C >> 3);
  depth_to_space_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(dph, din, batch, H, W, C, accumulate);
  return cudaGetLastError();
}

// bias gradient: out[c] += sum_r m[r, c]   (m bf16 [rows, C], C % 8 == 0, C <= 2048).  Thread = one 16-byte
// granule (8 channels) of every rpp-th row, four rows in flight; block partials combined in shared memory,
// one atomicAdd per channel and block.  Ordered: the block partials go to ws[block][C] and the last-arriving block
// adds them to out in block order.
template <bool kOrdered>
__global__ void __launch_bounds__(256) colsum_kernel(const bf16* __restrict__ m, float* __restrict__ out, long long rows,
                                                     int C, float* __restrict__ ws, unsigned* __restrict__ tickets) {
  __shared__ float red[256][9];
  const int VPR = C >> 3, rpp = 256 / VPR;
  const int t = threadIdx.x, vl = t % VPR, rsub = t / VPR;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (t < rpp * VPR) {
    const long long stride = static_cast<long long>(gridDim.x) * rpp;
    for (long long r = static_cast<long long>(blockIdx.x) * rpp + rsub; r < rows; r += 4 * stride) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long rr = r + u * stride;
        v[u] = rr < rows ? __ldg(reinterpret_cast<const uint4*>(m + rr * C) + vl) : make_uint4(0u, 0u, 0u, 0u);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float2 a0 = unpack_bf16x2(v[u].x), a1 = unpack_bf16x2(v[u].y), a2 = unpack_bf16x2(v[u].z), a3 = unpack_bf16x2(v[u].w);
        acc[0] += a0.x; acc[1] += a0.y; acc[2] += a1.x; acc[3] += a1.y;
        acc[4] += a2.x; acc[5] += a2.y; acc[6] += a3.x; acc[7] += a3.y;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[t][j] = acc[j];
  __syncthreads();
  for (int ch = t; ch < C; ch += 256) {
    const int cvl = ch >> 3, j = ch & 7;
    float sum = 0.f;
    for (int rs = 0; rs < rpp; ++rs) sum += red[rs * VPR + cvl][j];
    if constexpr (kOrdered) ws[static_cast<long long>(blockIdx.x) * C + ch] = sum;
    else atomicAdd(out + ch, sum);
  }
  if constexpr (kOrdered) {
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (t == 0) last = atomicAdd(tickets, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    for (int ch = t; ch < C; ch += 256) {
      float sum = 0.f;
      for (unsigned b = 0; b < gridDim.x; ++b) sum += __ldcg(ws + static_cast<long long>(b) * C + ch);
      out[ch] += sum;
    }
    if (t == 0) *tickets = 0u;
  }
}
static long long colsum_grid(long long rows, int C, int num_sms) {
  const int rpp = 256 / (C / 8);
  long long grid = (rows + 16ll * rpp - 1) / (16ll * rpp);          // >= 16 rows per thread
  if (grid > 4ll * num_sms) grid = 4ll * num_sms;
  if (grid < 1) grid = 1;
  return grid;
}
cudaError_t launch_colsum(const bf16* m, float* out, long long rows, int C, int num_sms, cudaStream_t stream) {
  if (C % 8 || C > 2048 || C <= 0) return cudaErrorInvalidValue;
  colsum_kernel<false><<<static_cast<unsigned>(colsum_grid(rows, C, num_sms)), 256, 0, stream>>>(m, out, rows, C, nullptr,
                                                                                                nullptr);
  return cudaGetLastError();
}
int64_t colsum_ws_floats(long long rows, int C, int num_sms) {
  if (C % 8 || C > 2048 || C <= 0) return 0;
  return colsum_grid(rows, C, num_sms) * C;
}
cudaError_t launch_colsum_ordered(const bf16* m, float* out, long long rows, int C, int num_sms, float* ws, unsigned* tickets,
                                  cudaStream_t stream) {
  if (C % 8 || C > 2048 || C <= 0 || ws == nullptr || tickets == nullptr) return cudaErrorInvalidValue;
  colsum_kernel<true><<<static_cast<unsigned>(colsum_grid(rows, C, num_sms)), 256, 0, stream>>>(m, out, rows, C, ws, tickets);
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------
// stand-alone sampler update: x = cx*x + ce*eps + cn*noise (float4 vectorised)
// ----------------------------------------------------------------------------------------------
__global__ void sampler_update_kernel(float* __restrict__ x, const float* __restrict__ eps,
                                      const float* __restrict__ noise, const float* __restrict__ coef,
                                      const int32_t* __restrict__ step_ptr, long long n4, long long n) {
  const int step = step_ptr ? *step_ptr : 0;
  const float cx = coef[3 * step], ce = coef[3 * step + 1], cn = coef[3 * step + 2];
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4; i += stride) {
    float4 xv = reinterpret_cast<float4*>(x)[i];
    const float4 ev = __ldg(reinterpret_cast<const float4*>(eps) + i);
    float4 nv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (noise) nv = __ldg(reinterpret_cast<const float4*>(noise) + i);
    xv.x = cx * xv.x + ce * ev.x + cn * nv.x;
    xv.y = cx * xv.y + ce * ev.y + cn * nv.y;
    xv.z = cx * xv.z + ce * ev.z + cn * nv.z;
    xv.w = cx * xv.w + ce * ev.w + cn * nv.w;
    reinterpret_cast<float4*>(x)[i] = xv;
  }
  // tail (n not a multiple of 4)
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    for (long long i = n4 * 4; i < n; ++i) x[i] = cx * x[i] + ce * eps[i] + cn * (noise ? noise[i] : 0.f);
  }
}

cudaError_t launch_sampler_update(float* x, const float* eps, const float* noise, const float* coef,
                                  const int32_t* step_ptr, int64_t n, cudaStream_t stream) {
  const long long n4 = n / 4;
  long long blocks = (n4 + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  sampler_update_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(x, eps, noise, coef, step_ptr, n4, n);
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------
// small fp32 linear: y[m,n] = sum_k act(x[m,k]) w[n,k] + b[n]; 16x64 output tile, K in chunks of 32
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) linear_f32_kernel(const float* __restrict__ x, long long ldx,
                                                         const float* __restrict__ w, const float* __restrict__ b,
                                                         float* __restrict__ y, long long ldy, int M, int N, int K,
                                                         int silu_in) {
  __shared__ float xs[16][33];
  __shared__ float ws[64][33];
  const int m0 = blockIdx.y * 16, n0 = blockIdx.x * 64;
  const int t = threadIdx.x;
  const int tm = t >> 4;          // 0..15
  const int tn = (t & 15) * 4;    // 0..60
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int k0 = 0; k0 < K; k0 += 32) {
    for (int i = t; i < 16 * 32; i += 256) {
      const int r = i >> 5, c = i & 31;
      float v = 0.f;
      if (m0 + r < M && k0 + c < K) {
        v = x[(m0 + r) * ldx + k0 + c];
        if (silu_in) v = v / (1.0f + expf(-v));
      }
      xs[r][c] = v;
    }
    for (int i = t; i < 64 * 32; i += 256) {
      const int r = i >> 5, c = i & 31;
      ws[r][c] = (n0 + r < N && k0 + c < K) ? w[static_cast<long long>(n0 + r) * K + k0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      const float xv = xs[tm][c];
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j] = fmaf(xv, ws[tn + j][c], acc[j]);
    }
    __syncthreads();
  }
  if (m0 + tm < M) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tn + j;
      if (n < N) y[(m0 + tm) * ldy + n] = acc[j] + (b ? b[n] : 0.f);
    }
  }
}

// larger batches (LatentUNet at sampling batch sizes): 64x64 output tile, 4x4 accumulators per thread, K in
// chunks of 16 staged k-major so the inner loop reads two float4 per 16 FMAs.  Same fp32 FMA order over k.
__global__ void __launch_bounds__(256) linear_f32_tile64_kernel(const float* __restrict__ x, long long ldx,
                                                                const float* __restrict__ w, const float* __restrict__ b,
                                                                float* __restrict__ y, long long ldy, int M, int N, int K,
                                                                int silu_in) {
  __shared__ __align__(16) float xs[16][68];
  __shared__ __align__(16) float ws[16][68];
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int t = threadIdx.x;
  const int tm = (t >> 4) * 4, tn = (t & 15) * 4;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
    for (int i = t; i < 64 * 16; i += 256) {
      const int r = i >> 4, c = i & 15;
      float v = 0.f;
      if (m0 + r < M && k0 + c < K) {
        v = x[(m0 + r) * ldx + k0 + c];
        if (silu_in) v = v / (1.0f + expf(-v));
      }
      xs[c][r] = v;
      ws[c][r] = (n0 + r < N && k0 + c < K) ? w[static_cast<long long>(n0 + r) * K + k0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const float4 xv = *reinterpret_cast<const float4*>(&xs[c][tm]);
      const float4 wv = *reinterpret_cast<const float4*>(&ws[c][tn]);
      const float xa[4] = {xv.x, xv.y, xv.z, xv.w}, wa[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(xa[i], wa[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + tm + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tn + j;
      if (n < N) y[m * ldy + n] = acc[i][j] + (b ? b[n] : 0.f);
    }
  }
}

cudaError_t launch_linear_f32(const float* x, int64_t ldx, const float* w, const float* b, float* y, int64_t ldy,
                              int M, int N, int K, int silu_in, cudaStream_t stream) {
  if (M >= 64) {
    dim3 grid64((N + 63) / 64, (M + 63) / 64, 1);
    linear_f32_tile64_kernel<<<grid64, 256, 0, stream>>>(x, ldx, w, b, y, ldy, M, N, K, silu_in);
    return cudaGetLastError();
  }
  dim3 grid((N + 63) / 64, (M + 15) / 16, 1);
  linear_f32_kernel<<<grid, 256, 0, stream>>>(x, ldx, w, b, y, ldy, M, N, K, silu_in);
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------
// general small fp32 GEMM for the BACKWARD of the fp32 Linears (time / latent MLPs, fc heads, LatentUNet layers):
//   C[M,N] (+)= op(A)[M,K] . op(B)[K,N]     op(X) = X or X^T, all row-major with leading dimensions
// dX = dY . W (A = dY, B = W), dW = dY^T . X (A = dY transposed, B = X), db = 1^T . dY.  64x64 output tile, 4x4
// accumulators per thread, K in chunks of 16 staged k-major; fixed fp32 FMA order over k (deterministic).  These GEMMs
// are tiny (M = batch <= 1024, N, K <= 8192) and weight-bandwidth bound: tensor cores would not help (fp32 operands).
// ----------------------------------------------------------------------------------------------
template <bool kOrdered>
__global__ void __launch_bounds__(256) gemm_f32_kernel(const float* __restrict__ A, long long lda, int transA,
                                                       const float* __restrict__ B, long long ldb, int transB,
                                                       float* __restrict__ Cm, long long ldc, int M, int N, int K,
                                                       int accumulate, float* __restrict__ ws, unsigned* __restrict__ tickets) {
  __shared__ __align__(16) float as[16][68];
  __shared__ __align__(16) float bs[16][68];
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int t = threadIdx.x;
  const int tm = (t >> 4) * 4, tn = (t & 15) * 4;
  float acc[4][4] = {};
  // split-K: blockIdx.z owns the k range [kb, ke); partial tiles are combined with atomicAdd (C pre-zeroed by the
  // launcher).  Used when M x N alone gives too few CTAs (dX of a [batch, 4992] x [4992, 256] Linear: 4 tiles, K = 4992).
  // Ordered: each split stores its 64x64 partial tile to ws[tile][split]; the last split to arrive at a tile sums them
  // in split order.
  const int kchunk = ((K + gridDim.z - 1) / gridDim.z + 15) / 16 * 16;
  const int kb = blockIdx.z * kchunk, ke = min(K, kb + kchunk);
  for (int k0 = kb; k0 < ke; k0 += 16) {
    for (int i = t; i < 64 * 16; i += 256) {
      // pick the index order that walks the operand's contiguous dimension with consecutive threads
      int r, c;
      if (transA) { r = i & 63; c = i >> 6; } else { r = i >> 4; c = i & 15; }
      float v = 0.f;
      if (m0 + r < M && k0 + c < ke) v = transA ? A[static_cast<long long>(k0 + c) * lda + m0 + r] : A[static_cast<long long>(m0 + r) * lda + k0 + c];
      as[c][r] = v;
      if (transB) { r = i >> 4; c = i & 15; } else { r = i & 63; c = i >> 6; }
      v = 0.f;
      if (n0 + r < N && k0 + c < ke) v = transB ? B[static_cast<long long>(n0 + r) * ldb + k0 + c] : B[static_cast<long long>(k0 + c) * ldb + n0 + r];
      bs[c][r] = v;
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const float4 av = *reinterpret_cast<const float4*>(&as[c][tm]);
      const float4 bv = *reinterpret_cast<const float4*>(&bs[c][tn]);
      const float aa[4] = {av.x, av.y, av.z, av.w}, ba[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], ba[j], acc[i][j]);
    }
    __syncthreads();
  }
  if constexpr (kOrdered) {
    if (gridDim.z > 1) {
      const unsigned tile = blockIdx.y * gridDim.x + blockIdx.x;
      float* part = ws + static_cast<long long>(tile) * gridDim.z * 4096;
#pragma unroll
      for (int i = 0; i < 4; ++i)
        *reinterpret_cast<float4*>(part + blockIdx.z * 4096 + (tm + i) * 64 + tn) =
            make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
      __shared__ bool last;
      __threadfence();
      __syncthreads();
      if (t == 0) last = atomicAdd(tickets + tile, 1u) == gridDim.z - 1;
      __syncthreads();
      if (!last) return;
      __threadfence();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float4 v = __ldcg(reinterpret_cast<const float4*>(part + (tm + i) * 64 + tn));
        for (unsigned z = 1; z < gridDim.z; ++z) {
          const float4 u = __ldcg(reinterpret_cast<const float4*>(part + z * 4096 + (tm + i) * 64 + tn));
          v.x += u.x; v.y += u.y; v.z += u.z; v.w += u.w;
        }
        acc[i][0] = v.x; acc[i][1] = v.y; acc[i][2] = v.z; acc[i][3] = v.w;
      }
      if (t == 0) tickets[tile] = 0u;
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + tm + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tn + j;
      if (n < N) {
        float* dst = Cm + static_cast<long long>(m) * ldc + n;
        if (!kOrdered && gridDim.z > 1) atomicAdd(dst, acc[i][j]);
        else *dst = accumulate ? *dst + acc[i][j] : acc[i][j];
      }
    }
  }
}

static int gemm_f32_splits(int M, int N, int K) {
  const int tiles = ((N + 63) / 64) * ((M + 63) / 64);
  int splits = 1;
  if (tiles < 64 && K >= 512) {                       // too few tiles to fill the machine and a long K loop
    splits = 148 / tiles;
    if (splits > K / 128) splits = K / 128;
    if (splits < 1) splits = 1;
  }
  return splits;
}

cudaError_t launch_gemm_f32(const float* A, int64_t lda, int transA, const float* B, int64_t ldb, int transB, float* Cm,
                            int64_t ldc, int M, int N, int K, int accumulate, cudaStream_t stream) {
  dim3 grid((N + 63) / 64, (M + 63) / 64, 1);
  const int splits = gemm_f32_splits(M, N, K);
  if (splits > 1) {
    grid.z = splits;
    if (!accumulate) {                                // the partial tiles are added atomically
      if (ldc == N) {
        cudaError_t e = cudaMemsetAsync(Cm, 0, static_cast<size_t>(M) * N * sizeof(float), stream);
        if (e != cudaSuccess) return e;
      } else {
        cudaError_t e = cudaMemset2DAsync(Cm, static_cast<size_t>(ldc) * sizeof(float), 0, static_cast<size_t>(N) * sizeof(float), M, stream);
        if (e != cudaSuccess) return e;
      }
    }
  }
  gemm_f32_kernel<false><<<grid, 256, 0, stream>>>(A, lda, transA, B, ldb, transB, Cm, ldc, M, N, K, accumulate, nullptr,
                                                   nullptr);
  return cudaGetLastError();
}

int64_t gemm_f32_ws_floats(int M, int N, int K) {
  const int splits = gemm_f32_splits(M, N, K);
  return splits > 1 ? static_cast<int64_t>((N + 63) / 64) * ((M + 63) / 64) * splits * 4096 : 0;
}

cudaError_t launch_gemm_f32_ordered(const float* A, int64_t lda, int transA, const float* B, int64_t ldb, int transB, float* Cm,
                                    int64_t ldc, int M, int N, int K, int accumulate, float* ws, unsigned* tickets,
                                    cudaStream_t stream) {
  dim3 grid((N + 63) / 64, (M + 63) / 64, gemm_f32_splits(M, N, K));
  if (grid.z > 1 && (ws == nullptr || tickets == nullptr)) return cudaErrorInvalidValue;
  gemm_f32_kernel<true><<<grid, 256, 0, stream>>>(A, lda, transA, B, ldb, transB, Cm, ldc, M, N, K, accumulate, ws, tickets);
  return cudaGetLastError();
}

__global__ void gather_rows_kernel(const float* __restrict__ table, const int64_t* __restrict__ idx,
                                   float* __restrict__ y, int N) {
  const int m = blockIdx.x;
  const long long row = idx[m];
  for (int i = threadIdx.x; i < N; i += blockDim.x) y[static_cast<long long>(m) * N + i] = table[row * N + i];
}
cudaError_t launch_gather_rows(const float* table, const int64_t* idx, float* y, int M, int N, cudaStream_t stream) {
  gather_rows_kernel<<<M, 128, 0, stream>>>(table, idx, y, N);
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------
// eval_fid output stage (run.py:288-295 + torchvision.utils.save_image): per image clip(x, -1, 1) -> (x + 1) / 2 ->
// mul 255, add 0.5, clamp(0, 255), truncate to uint8, CHW -> HWC.  Same fp32 operations in the same order (no FMA
// contraction), so the bytes equal what the reference writes into its PNGs.
// ----------------------------------------------------------------------------------------------
__global__ void to_uint8_hwc_kernel(const float* __restrict__ x, uint8_t* __restrict__ out, int C, int HW, long long total) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = i / (static_cast<long long>(HW) * C);
    const long long rem = i - n * HW * C;
    const int pix = static_cast<int>(rem / C), c = static_cast<int>(rem - static_cast<long long>(pix) * C);
    float v = x[(n * C + c) * HW + pix];
    v = fminf(fmaxf(v, -1.0f), 1.0f);
    v = __fdiv_rn(__fadd_rn(v, 1.0f), 2.0f);
    v = __fadd_rn(__fmul_rn(v, 255.0f), 0.5f);
    v = fminf(fmaxf(v, 0.0f), 255.0f);
    out[i] = static_cast<uint8_t>(v);
  }
}
cudaError_t launch_to_uint8_hwc(const float* x, uint8_t* out, int batch, int C, int H, int W, cudaStream_t stream) {
  const long long total = static_cast<long long>(batch) * C * H * W;
  if (total <= 0) return cudaErrorInvalidValue;
  long long blocks = (total + 255) / 256;
  if (blocks > 2368) blocks = 2368;
  to_uint8_hwc_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(x, out, C, H * W, total);
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------
// LatentUNet layer tail (models.py:147-163): out = SiLU(LayerNorm(y * (1 + cond))) over rows of N features.
// One CTA per row; the modulated row is staged in shared memory, mean and variance are two separate
// passes (as ATen's layer_norm), cond may be a single broadcast row (sampling: every sample shares t).
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ float block_sum_128(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  return (red[0] + red[1]) + (red[2] + red[3]);
}
__global__ void __launch_bounds__(128) scale_ln_silu_kernel(const float* __restrict__ y, long long ldy,
                                                            const float* __restrict__ cond, long long cond_stride,
                                                            long long cond_step_stride, const int* __restrict__ step_ptr,
                                                            const float* __restrict__ gamma, const float* __restrict__ beta,
                                                            float eps, float* __restrict__ out, long long ldo, int N,
                                                            int apply_silu) {
  extern __shared__ float row[];
  __shared__ float red[4];
  const long long m = blockIdx.x;
  const float* yr = y + m * ldy;
  const float* cr = cond ? cond + m * cond_stride + (step_ptr ? *step_ptr * cond_step_stride : 0) : nullptr;
  float s = 0.f;
  for (int i = threadIdx.x; i < N; i += 128) {
    float v = yr[i];
    if (cr) v *= 1.0f + cr[i];
    row[i] = v;
    s += v;
  }
  const float mean = block_sum_128(s, red) / static_cast<float>(N);
  float q = 0.f;
  for (int i = threadIdx.x; i < N; i += 128) { const float d = row[i] - mean; q = fmaf(d, d, q); }
  const float rstd = rsqrtf(block_sum_128(q, red) / static_cast<float>(N) + eps);
  for (int i = threadIdx.x; i < N; i += 128) {
    float v = (row[i] - mean) * rstd;
    if (gamma) v = fmaf(v, gamma[i], beta[i]);
    if (apply_silu) v = v / (1.0f + __expf(-v));
    out[m * ldo + i] = v;
  }
}
cudaError_t launch_scale_ln_silu(const float* y, long long ldy, const float* cond, long long cond_stride,
                                 long long cond_step_stride, const int* step_ptr, const float* gamma, const float* beta,
                                 float eps, float* out, long long ldo, int M, int N, int apply_silu, cudaStream_t stream) {
  if (M <= 0 || N <= 0 || N > 8192) return cudaErrorInvalidValue;
  scale_ln_silu_kernel<<<M, 128, N * sizeof(float), stream>>>(y, ldy, cond, cond_stride, cond_step_stride, step_ptr, gamma,
                                                              beta, eps, out, ldo, N, apply_silu);
  return cudaGetLastError();
}

__global__ void copy2d_f32_kernel(const float* __restrict__ src, long long lds, float* __restrict__ dst, long long ldd,
                                  int M, int N) {
  const long long total = static_cast<long long>(M) * N;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = i / N, n = i - m * N;
    dst[m * ldd + n] = src[m * lds + n];
  }
}
cudaError_t launch_copy2d_f32(const float* src, long long lds, float* dst, long long ldd, int M, int N, cudaStream_t stream) {
  if (M <= 0 || N <= 0) return cudaErrorInvalidValue;
  const long long total = static_cast<long long>(M) * N;
  long long blocks = (total + 255) / 256;
  if (blocks > 1184) blocks = 1184;
  const int grid = static_cast<int>(blocks);
  copy2d_f32_kernel<<<grid, 256, 0, stream>>>(src, lds, dst, ldd, M, N);
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------
// Element gather (training): dst[i] (+)= src[idx[i]-1] (+ src[idx2[i]-1]), index 0 = literal zero.
// One launch re-packs every fp32 parameter into the bf16 GEMM operand layouts (forward and data-gradient
// packings) or assembles the parameter-shaped gradients from the weight-gradient arena.  n % 4 == 0.
// ----------------------------------------------------------------------------------------------
template <bool kBf16, bool kAcc>
__global__ void __launch_bounds__(256) gather_elems_kernel(const float* __restrict__ src, const int* __restrict__ idx,
                                                           const int* __restrict__ idx2, void* __restrict__ dst,
                                                           long long n4) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int4 a = reinterpret_cast<const int4*>(idx)[i];
    float v0 = a.x ? src[a.x - 1] : 0.f, v1 = a.y ? src[a.y - 1] : 0.f;
    float v2 = a.z ? src[a.z - 1] : 0.f, v3 = a.w ? src[a.w - 1] : 0.f;
    if (idx2 != nullptr) {
      const int4 b = reinterpret_cast<const int4*>(idx2)[i];
      v0 += b.x ? src[b.x - 1] : 0.f; v1 += b.y ? src[b.y - 1] : 0.f;
      v2 += b.z ? src[b.z - 1] : 0.f; v3 += b.w ? src[b.w - 1] : 0.f;
    }
    if constexpr (kBf16) {
      __nv_bfloat162 lo = __floats2bfloat162_rn(v0, v1), hi = __floats2bfloat162_rn(v2, v3);
      uint2 o;
      o.x = *reinterpret_cast<uint32_t*>(&lo);
      o.y = *reinterpret_cast<uint32_t*>(&hi);
      reinterpret_cast<uint2*>(dst)[i] = o;
    } else {
      float4* d = reinterpret_cast<float4*>(dst) + i;
      if constexpr (kAcc) {
        const float4 o = *d;
        v0 += o.x; v1 += o.y; v2 += o.z; v3 += o.w;
      }
      *d = make_float4(v0, v1, v2, v3);
    }
  }
}
cudaError_t launch_gather_elems(const float* src, const int* idx, const int* idx2, void* dst, long long n, bool dst_bf16,
                                bool accumulate, int num_sms, cudaStream_t stream) {
  const long long n4 = n / 4;
  if (n4 == 0) return cudaSuccess;
  const int grid = static_cast<int>(min(static_cast<long long>(num_sms) * 8, (n4 + 255) / 256));
  if (dst_bf16) gather_elems_kernel<true, false><<<grid, 256, 0, stream>>>(src, idx, idx2, dst, n4);
  else if (accumulate) gather_elems_kernel<false, true><<<grid, 256, 0, stream>>>(src, idx, idx2, dst, n4);
  else gather_elems_kernel<false, false><<<grid, 256, 0, stream>>>(src, idx, idx2, dst, n4);
  return cudaGetLastError();
}

// ----------------------------------------------------------------------------------------------
// MMD (utils.py:74-90): loss = mean k(x,x) + mean k(y,y) - 2 mean k(x,y), k(u,v)=exp(-|u-v|^2/D^2)
// One block per column index j: accumulates sum_i [k(x_i,x_j) + k(y_i,y_j) - 2 k(x_i,y_j)] and
// d loss / d y_j.  The per-block partial is added to *loss with one atomicAdd (loss must be zeroed).
// Ordered: every warp accumulates d loss / d y_j in a shared row of its own (the rows are summed in warp order), the
// per-block partials go to ws[j], and the last-arriving block sums them in block order.
// ----------------------------------------------------------------------------------------------
template <bool kOrdered>
__global__ void __launch_bounds__(128) mmd_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                  float* __restrict__ loss, float* __restrict__ grad_y, int B,
                                                  int D, float* __restrict__ ws, unsigned* __restrict__ tickets) {
  extern __shared__ float sm[];
  float* xj = sm;            // [D]
  float* yj = sm + D;        // [D]
  float* gacc = sm + 2 * D;  // [D] ([4][D] ordered)
  __shared__ float red[4];
  const int j = blockIdx.x;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  for (int d = t; d < D; d += 128) {
    xj[d] = x[static_cast<long long>(j) * D + d];
    yj[d] = y[static_cast<long long>(j) * D + d];
    gacc[d] = 0.f;
    if constexpr (kOrdered) gacc[D + d] = gacc[2 * D + d] = gacc[3 * D + d] = 0.f;
  }
  __syncthreads();
  const float inv_d2 = 1.0f / (static_cast<float>(D) * static_cast<float>(D));
  const float inv_b2 = 1.0f / (static_cast<float>(B) * static_cast<float>(B));
  float part = 0.f;
  // one warp per i; lanes stride over D
  for (int i = warp; i < B; i += 4) {
    const float* xi = x + static_cast<long long>(i) * D;
    const float* yi = y + static_cast<long long>(i) * D;
    float dxx = 0.f, dyy = 0.f, dxy = 0.f;
    for (int d = lane; d < D; d += 32) {
      const float a = xi[d], bb = yi[d];
      const float e0 = a - xj[d], e1 = bb - yj[d], e2 = a - yj[d];
      dxx = fmaf(e0, e0, dxx);
      dyy = fmaf(e1, e1, dyy);
      dxy = fmaf(e2, e2, dxy);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      dxx += __shfl_xor_sync(0xffffffffu, dxx, o);
      dyy += __shfl_xor_sync(0xffffffffu, dyy, o);
      dxy += __shfl_xor_sync(0xffffffffu, dxy, o);
    }
    const float kxx = expf(-dxx * inv_d2), kyy = expf(-dyy * inv_d2), kxy = expf(-dxy * inv_d2);
    if (lane == 0) part += kxx + kyy - 2.0f * kxy;
    if (grad_y != nullptr) {
      // d/dy_j: 2 * k(y_i,y_j) * (-2 (y_j - y_i)/D^2)  -  2 * k(x_i,y_j) * (-2 (y_j - x_i)/D^2), all / B^2
      const float cy = -4.0f * kyy * inv_d2 * inv_b2;
      const float cxy = 4.0f * kxy * inv_d2 * inv_b2;
      for (int d = lane; d < D; d += 32) {
        const float g = cy * (yj[d] - yi[d]) + cxy * (yj[d] - xi[d]);
        if constexpr (kOrdered) gacc[warp * D + d] += g;      // this lane owns element d of its warp's row
        else atomicAdd(&gacc[d], g);
      }
    }
  }
  if (lane == 0) red[warp] = part;
  __syncthreads();
  if constexpr (kOrdered) {
    if (t == 0) ws[j] = (red[0] + red[1] + red[2] + red[3]) * inv_b2;
    if (grad_y != nullptr)
      for (int d = t; d < D; d += 128)
        grad_y[static_cast<long long>(j) * D + d] = (gacc[d] + gacc[D + d]) + (gacc[2 * D + d] + gacc[3 * D + d]);
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (t == 0) last = atomicAdd(tickets, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    float s = 0.f;                                          // fixed order: thread t sums blocks t, t + 128, ...
    for (int b = t; b < B; b += 128) s += __ldcg(ws + b);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __syncthreads();
    if (lane == 0) red[warp] = s;
    __syncthreads();
    if (t == 0) {
      *loss = (red[0] + red[1]) + (red[2] + red[3]);
      *tickets = 0u;
    }
  } else {
    if (t == 0) atomicAdd(loss, (red[0] + red[1] + red[2] + red[3]) * inv_b2);
    if (grad_y != nullptr)
      for (int d = t; d < D; d += 128) grad_y[static_cast<long long>(j) * D + d] = gacc[d];
  }
}

cudaError_t launch_mmd(const float* x, const float* y, float* loss, float* grad_y, int B, int D,
                       cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(loss, 0, sizeof(float), stream);
  if (e != cudaSuccess) return e;
  mmd_kernel<false><<<B, 128, 3 * D * sizeof(float), stream>>>(x, y, loss, grad_y, B, D, nullptr, nullptr);
  return cudaGetLastError();
}

cudaError_t launch_mmd_ordered(const float* x, const float* y, float* loss, float* grad_y, int B, int D, float* ws,
                               unsigned* tickets, cudaStream_t stream) {
  if (ws == nullptr || tickets == nullptr) return cudaErrorInvalidValue;
  const int smem = 6 * D * static_cast<int>(sizeof(float));
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(mmd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 6 * 4096 * 4);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  mmd_kernel<true><<<B, 128, smem, stream>>>(x, y, loss, grad_y, B, D, ws, tickets);
  return cudaGetLastError();
}

}  // namespace idf
