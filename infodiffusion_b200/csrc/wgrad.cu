// Convolution weight gradient on tcgen05:  dW[co, tap, ci] = sum_r dY[r, co] * X[r + off_tap, ci]
// (backward of nn.Conv2d w.r.t. its weight: modules.py:66,81,133-136,216,222,228,231,... under autograd).
//
// GEMM view per tap: D[co, ci] = A[co, r] * B[ci, r]^T with the pixel rows r as the K dimension.  Both
// operands come straight from the pad-flat activation matrices ([rows, C], channels contiguous), i.e.
// they are MN-major for the tensor core: a TMA box {64 channels, KB rows} lands as [K rows x 128 B] and is
// described with LBO = distance between 64-channel atoms, SBO = 1024 B (8 K-rows), +2048 B per K=16 step.
// The taps of one kernel row (kx = 0,1,2) are the SAME X rows shifted by one: one X halo of KB+8 rows per
// stage serves them all (the start address of a descriptor may be any 128-byte row, tools/probe_shift.py).
//
// Work unit = (128-wide co tile, <=128-wide ci chunk, cluster of <=3 taps, slab of K blocks): accumulators
// (<= 3 x 128 fp32 columns) stay in TMEM for the whole slab, then are added to the global fp32 dW with
// red.global.add (split-K across slabs; summation order across slabs is not deterministic).  The ordered variant
// (torch's deterministic mode) stores each slab's tile into its own dW-shaped slice of a partials buffer instead, and
// wgrad_reduce_kernel adds the slices to dW in slab order.
#include "kernels.cuh"

namespace idf {

constexpr int kWgKB = 128;          // K rows per pipeline stage
constexpr int kWgHalo = 8;          // extra X rows per stage (tap shifts 0..7)
constexpr int kWgStages = 3;

__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3fffu);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3fffu) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

template <bool kOrdered>
__global__ void __launch_bounds__(192, 1) wgrad_kernel(const __grid_constant__ WgradKernelParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr uint32_t A_BYTES = 2 * kWgKB * 128;                  // two 64-co atoms
  constexpr uint32_t B_ATOM = (kWgKB + kWgHalo) * 128;           // one 64-ci atom incl. halo rows
  constexpr uint32_t B_BYTES = 2 * B_ATOM;
  constexpr uint32_t STAGE = A_BYTES + B_BYTES;                  // 32 KB + 34 KB
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + kWgStages * STAGE);
  uint64_t* empty = full + kWgStages;
  uint64_t* done = empty + kWgStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int unit = blockIdx.x % p.n_units;
  const int slab = blockIdx.x / p.n_units;
  const int kb_begin = slab * p.kb_per_slab;
  const int kb_end = min(p.n_kb, kb_begin + p.kb_per_slab);
  const int cl = unit % p.n_cl;
  const int co0 = unit / (p.n_cl * p.n_ci) * 128, ci0 = (unit / p.n_cl) % p.n_ci * p.ci_step;
  const int ci_n = min(p.ci_step, p.cin - ci0), ntap = p.c_ntap[cl];
  const int n_ci_atoms = ci_n >> 6;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < kWgStages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
    mbar_init(done, 1);
    fence_mbar_init();
    tma_prefetch_desc(&p.tmDY);
    tma_prefetch_desc(&p.tmX);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = lds32(smem_u32(tmem_slot));

  if (kb_begin < kb_end) {
    if (warp == 0) {
      if (lane == 0) {                       // ---- TMA producer
        int st = 0; uint32_t ph = 0;
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          mbar_wait(empty + st, ph ^ 1u);
          mbar_arrive_expect_tx(full + st, A_BYTES + static_cast<uint32_t>(n_ci_atoms) * B_ATOM);
          uint8_t* a = smem + st * STAGE;
          uint8_t* b = a + A_BYTES;
          const int r0 = kb * kWgKB;
          tma_load_2d(a, &p.tmDY, full + st, co0, r0);                       // channels >= Cout are zero-filled
          tma_load_2d(a + kWgKB * 128, &p.tmDY, full + st, co0 + 64, r0);
          for (int j = 0; j < n_ci_atoms; ++j)
            tma_load_2d(b + j * B_ATOM, &p.tmX, full + st, ci0 + 64 * j, r0 + p.c_base[cl]);
          if (++st == kWgStages) { st = 0; ph ^= 1u; }
        }
      }
    } else if (warp == 1) {
      // ---- UMMA issuer: the whole warp runs the loop on warp-uniform values, only the tcgen05 instructions sit under
      // elect.sync, so descriptors stay in uniform registers (see the issuer of conv_halo_kernel)
      const uint32_t idesc = umma_idesc_f16(128, static_cast<uint32_t>(ci_n), kFmtBF16) | (1u << 15) | (1u << 16);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
      const uint32_t idesc_u = __shfl_sync(0xffffffffu, idesc, 0);
      int st = 0; uint32_t ph = 0;
      for (int kb = kb_begin; kb < kb_end; ++kb) {
        mbar_wait(full + st, ph);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + st * STAGE);
        const uint32_t b_addr = a_addr + A_BYTES;
        for (int t = 0; t < ntap; ++t) {
          // (shuffles from lane 0 tell the compiler these are warp-uniform)
          const uint32_t brow = __shfl_sync(0xffffffffu, b_addr + static_cast<uint32_t>(p.c_rel[cl * 3 + t]) * 128u, 0);
          const uint32_t a_u = __shfl_sync(0xffffffffu, a_addr, 0);
          const uint32_t d = __shfl_sync(0xffffffffu, tmem_u + static_cast<uint32_t>(t * ci_n), 0);
          const uint32_t acc0 = kb > kb_begin ? 1u : 0u;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < kWgKB / 16; ++k) {
              const uint64_t da = umma_desc_mn(a_u + k * 2048, kWgKB * 128);
              const uint64_t db = umma_desc_mn(brow + k * 2048, B_ATOM);
              umma_f16(d, da, db, idesc_u, k > 0 ? 1u : acc0);
            }
            if (t + 1 == ntap) {
              umma_commit(empty + st);
              if (kb + 1 == kb_end) umma_commit(done);
            }
          }
          __syncwarp();
        }
        if (++st == kWgStages) { st = 0; ph ^= 1u; }
      }
    } else {
      // ---- epilogue (warps 2..5): TMEM lane quarter = warp % 4
      const int q = warp & 3;
      mbar_wait(done, 0);
      tc_fence_after();
      const int co = co0 + q * 32 + lane;
      const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
      for (int t = 0; t < ntap; ++t) {
        const int tap = p.c_tap[cl * 3 + t];
        for (int c = 0; c < ci_n; c += 32) {
          uint32_t v[32];
          tmem_ld_32x32(tmem + lane_addr + static_cast<uint32_t>(t * ci_n + c), v);
          tmem_ld_wait();
          if (co < p.cout) {
            const int64_t e = (static_cast<int64_t>(co) * p.ntaps + tap) * p.cin + ci0 + c;
            if constexpr (kOrdered) {
              float4* dst = reinterpret_cast<float4*>(p.partials + static_cast<int64_t>(slab) * p.cout * p.ntaps * p.cin + e);
#pragma unroll
              for (int j = 0; j < 8; ++j)
                dst[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                                     __uint_as_float(v[4 * j + 3]));
              continue;
            }
            float* dst = p.dw + e;
#pragma unroll
            for (int j = 0; j < 8; ++j)      // 16-byte vector reductions: 8 instead of 32 atomics per lane and chunk
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4 * j), "f"(__uint_as_float(v[4 * j])),
                           "f"(__uint_as_float(v[4 * j + 1])), "f"(__uint_as_float(v[4 * j + 2])),
                           "f"(__uint_as_float(v[4 * j + 3]))
                           : "memory");
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// dW[e] += partials[0][e] + partials[1][e] + ... (slab order), one float4 of dW per thread
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float4* __restrict__ partials, float4* __restrict__ dw,
                                                           long long n4, int slabs) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 s = __ldg(partials + i);
    for (int k = 1; k < slabs; ++k) {
      const float4 v = __ldg(partials + k * n4 + i);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    float4 d = dw[i];
    d.x += s.x; d.y += s.y; d.z += s.z; d.w += s.w;
    dw[i] = d;
  }
}

cudaError_t launch_wgrad(const WgradKernelParams& p, int grid, int slabs, int num_sms, cudaStream_t stream) {
  constexpr uint32_t SMEM = kWgStages * (2 * kWgKB * 128 + 2 * (kWgKB + kWgHalo) * 128) + 128 + 1024;
  const bool ordered = p.partials != nullptr && slabs > 1;     // a single slab adds each element once: already ordered
  static bool attr_set[2] = {false, false};
  if (!attr_set[ordered]) {
    cudaError_t e = cudaFuncSetAttribute(ordered ? wgrad_kernel<true> : wgrad_kernel<false>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(SMEM));
    if (e != cudaSuccess) return e;
    attr_set[ordered] = true;
  }
  if (!ordered) {
    wgrad_kernel<false><<<grid, 192, SMEM, stream>>>(p);
    return cudaGetLastError();
  }
  wgrad_kernel<true><<<grid, 192, SMEM, stream>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  const long long n4 = static_cast<long long>(p.cout) * p.ntaps * p.cin / 4;
  long long blocks = (n4 + 255) / 256;
  if (blocks > 8ll * num_sms) blocks = 8ll * num_sms;
  wgrad_reduce_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(reinterpret_cast<const float4*>(p.partials),
                                                                         reinterpret_cast<float4*>(p.dw), n4, slabs);
  return cudaGetLastError();
}

}  // namespace idf
