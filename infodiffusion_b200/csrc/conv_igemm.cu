// Implicit-GEMM convolution for sm_100a, v2: halo-resident A operand, tcgen05.mma, TMEM accumulators.
// See include/idf_b200.h for the contract.
//
// Why v2: the v1 kernel loaded one [128 x 64] A tile per (tap, channel-chunk) and was bound by
// L2->SM operand traffic (ncu: 12 TB/s from L2, tensor pipe 41-44 %).  In the pad-flat layout the nine
// taps of a 3x3 conv are the SAME rows shifted by a constant, and a K-major SWIZZLE_128B UMMA
// descriptor may start at any 128-byte row (the swizzle is a function of the absolute shared-memory
// address; verified with tools/probe_shift.py).  So per 64-channel chunk the CTA loads ONE halo
//   rows [row0 + lo, row0 + 128*MT + hi)        (lo/hi = min/max tap offset, +-(W+2) for 3x3)
// and every (tap, m) operand is a descriptor into it.  One CTA owns MT consecutive 128-row tiles
// (MT accumulators in TMEM), so each streamed weight tile B[BN x 64] feeds MT MMAs as well.
// Operand bytes per MMA drop 3-7x (e.g. 64->64 @64^2: 221 KB -> 33 KB + weights per 128 rows).
//
// Roles (512 threads; 768 in the XF variant), LOW to HIGH warp id -- the SM sub-partition arbiter prefers the highest
// warp id among the eligible warps, so the latency-critical single-warp roles sit on top and are never starved:
//                      XF variant only: warps 0..7 = transform (fused AdaGN + SiLU on the halo, in place)
//                      next 8 warps = drain (TMEM -> bf16 staging tile -> TMA store; two warps per TMEM lane quarter)
//                      next 4 warps = GroupNorm statistics of the staged tiles (one warp per lane quarter)
//                      then: A (halo) TMA producer, B (weights) TMA producer,
//                            TMEM allocator (+ second UMMA issuer when MT >= 2), UMMA issuer
// Pipelines: A halo stages x2 (x3: XF with MT <= 2), B ring x4-8 (full/empty mbarriers), TMEM accumulator sets x2,
// staging tiles x2 per drain warp.  With PAIR the kernel runs as clusters of two CTAs (tcgen05 cta_group::2), see below.
#include <type_traits>

#include "kernels.cuh"

namespace idf {

// Pipeline trace (development builds only, -DIDF_CONV_TRACE; tools/conv_trace.py): CTA 0 records globaltimer stamps of
// every work item's phases into the buffer passed as out_f32 (unused by the bf16 epilogue): [item][8] int64.
#ifdef IDF_CONV_TRACE
#define IDF_TRACE(slot, item)                                                                                     \
  do {                                                                                                            \
    if (blockIdx.x == 0 && p.out_f32 != nullptr && (item) < 64) {                                                 \
      unsigned long long t_;                                                                                      \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                                      \
      reinterpret_cast<unsigned long long*>(p.out_f32)[(item) * 8 + (slot)] = t_;                                 \
    }                                                                                                             \
  } while (0)
#else
#define IDF_TRACE(slot, item) do { } while (0)
#endif

// transform warps of the XF variant (4 rows per warp and pass).  In isolation 12 warps beat 8 (tools/cu/xf_bench.cu: 1.8 vs
// 2.2 us per 648-row halo), inside the kernel they do not: 896 threads leave 72 registers per thread at launch and the
// drain / statistics / producer warps pay for it (64->64 @64^2 fused: 120 vs 105 us).
constexpr int kXfWarps = 8;
constexpr int kXfRows = 4 * kXfWarps;

int g_pdl = 1;     // conv / AdaGN kernels are launched with programmatic dependent launch: their prologue (barriers, TMEM,
                   // bias, weight tiles) overlaps the predecessor's tail.  +6 % sampling rate at 32 images per GPU, neutral
                   // at 256, bitwise neutral; idf_set_option("pdl", 0) disables
int g_xf_debug = 0;  // measurement only: 1 = transform warps forward the halo untouched, 2 = affine without the SiLU,
                     // 5 = full transform but no MMAs are issued

__host__ __device__ constexpr int conv_b_stages(int bn) { return bn == 16 ? 8 : (bn == 64 ? 4 : 6); }
// per-epilogue-warp staging tile: 32 rows x 64 B in the TMA SWIZZLE_64B layout (16-byte chunk c of row r lives at
// chunk c ^ ((r >> 1) & 3)): conflict-free for the row-per-lane 16-byte accesses, for the 4-lanes-per-row coalesced
// residual deposit and for the column-pair reads of the GroupNorm partial sums; the tile leaves through ONE TMA store.
constexpr uint32_t kStageTile = 32 * 64;
// two staging tiles per drain warp: a warp only waits for the TMA store it issued two work items ago (the TMA engine
// also serves the operand loads and drains the staging tiles late) and the statistics warps get a full item of slack
constexpr uint32_t kStageBytes = 16 * kStageTile;
constexpr int kXfMaxRows = 4 * 128 + 256;   // rows of the largest halo (MT = 4 tiles + the widest tap spread)
constexpr uint32_t kRowTabBytes = 3 * 2 * kXfMaxRows;   // XF variant: int16 row table per halo stage
constexpr uint32_t kBiasBytes = 1536 * 4;  // bias vector of the whole conv (cout_pad <= 1536: q|k|v of a 512-wide head), staged once per CTA
__device__ __forceinline__ uint32_t stage_off(int row, int chunk) {
  return static_cast<uint32_t>(row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4));
}

// Halo stages.  The plain kernel is MMA-bound with two (the next halo lands while the MMAs of this one run).  In the
// fused-AdaGN variant load -> transform -> MMAs are serial per stage, so two stages bound the item period by half that
// chain (tools/conv_trace.py: 3.9 + 5.9 + 4.0 us per 512-row item, 7.2 us period); items of at most two tiles leave room
// for a third stage, which lets the load of item i+2 and the transform of item i+1 run under the MMAs of item i.
__host__ __device__ constexpr int conv_a_stages(int mt, bool xf) { return (xf && mt <= 2) ? 3 : 2; }

template <int BN, int MT, bool PAIR = false, bool XF = false>
struct HaloCfg {
  static constexpr int A_STAGES = conv_a_stages(MT, XF);
  static constexpr int B_STAGES = conv_b_stages(BN);
  static constexpr uint32_t B_BYTES = BN * kBK * 2 / (PAIR ? 2 : 1);   // per CTA: a pair splits the weight tile along N
  static constexpr uint32_t ACC_COLS = MT * BN;                       // one accumulator set
  static constexpr uint32_t TMEM_COLS = (2 * ACC_COLS <= 32) ? 32 : (2 * ACC_COLS <= 64) ? 64
                                        : (2 * ACC_COLS <= 128) ? 128 : (2 * ACC_COLS <= 256) ? 256 : 512;
  static_assert(2 * ACC_COLS <= 512, "accumulators do not fit in TMEM");
  static constexpr int NBARS = 3 * A_STAGES + 2 * B_STAGES + 4 + 32;   // + staged / stats-done per drain warp and tile
  static constexpr int NI = (MT >= 2) ? 2 : 1;                        // UMMA issuing threads (accumulators split)
};

__host__ __device__ inline uint32_t conv_smem_bytes(int a_stage_bytes, int a_stages, int b_stages, int b_bytes, bool xf) {
  return static_cast<uint32_t>(a_stages * a_stage_bytes + b_stages * b_bytes + 2048 /*barriers 512 + tap table 1024 + pad*/ +
                               kStageBytes + kBiasBytes + (xf ? kRowTabBytes : 0u) + 1024 /*align*/);
}

// ---------------------------------------------------------------------------------------------------
// epilogue for one (accumulator m, 32-column chunk) work item held in registers
// ---------------------------------------------------------------------------------------------------
// Coalesced residual fetch for one work item: 4 lanes cover one row's 64 bytes, 8 rows per instruction.
// Issued one item ahead of its use so that the DRAM latency hides behind the previous item.
__device__ __forceinline__ void residual_fetch(const ConvKernelParams& p, int64_t warp_row0, int col0, int lane,
                                               uint4 (&res)[4]) {
  const int sub_row = lane >> 2, sub_chunk = lane & 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t rr = warp_row0 + i * 8 + sub_row;
    res[i] = make_uint4(0, 0, 0, 0);
    if (rr < p.rows) res[i] = __ldg(reinterpret_cast<const uint4*>(p.residual + rr * p.res_ld + col0) + sub_chunk);
  }
}

// One (accumulator, 32-column) work item of a drain warp; executed by all 32 lanes.
//   out = bf16(acc + bias (+ residual)), pad rows forced to zero.
// The warp's 32 rows x 64 B pass through one of its two private shared-memory staging tiles (SWIZZLE_64B layout) and
// leave with one TMA store (rows beyond the tensor are clipped by the tensor map); the residual, fetched coalesced one
// item ahead (4 lanes per row), is deposited in the same tile first and read back row-per-lane.  Before the tile is
// rewritten, the TMA store issued from it two items ago must have read it and the statistics warp must be done with it.
// up_row >= 0 (up2 plans): the lane's row goes to row `up_row` of the twice as large output map, columns col0 - up_col0
// (the column tile is the output parity); the staging tile is still written for the statistics warp.
__device__ __forceinline__ void epilogue_drain_chunk(const ConvKernelParams& p, const uint32_t (&v)[32],
                                                     int64_t warp_row0, bool valid, int col0, int lane, uint32_t stage,
                                                     uint32_t bias_sa, const uint4 (&res)[4], uint64_t* staged,
                                                     uint64_t* sdone, uint32_t use, int64_t up_row = -1, int up_col0 = 0,
                                                     int trow = -1) {
  const int sub_row = lane >> 2, sub_chunk = lane & 3;     // coalesced distribution: row = 8 i + sub_row
  if (lane == 0) {
    bulk_wait_read<1>();                     // all but the newest store (which reads the OTHER tile) are done reading
    if (trow >= 0) IDF_TRACE(2, trow);
    mbar_wait(sdone, (use & 1u) ^ 1u);       // the statistics of this tile's previous contents have been taken
    if (trow >= 0) IDF_TRACE(3, trow);
  }
  __syncwarp();
  if (p.residual != nullptr) {
#pragma unroll
    for (int i = 0; i < 4; ++i) sts128(stage + stage_off(i * 8 + sub_row, sub_chunk), res[i]);
    __syncwarp();
  }
  float f[32];
#pragma unroll
  for (int j = 0; j < 8; ++j) {            // bias staged in shared memory once per CTA (warp-uniform address: broadcast)
    const uint4 b = lds128(bias_sa + (col0 + 4 * j) * 4);
    f[4 * j + 0] = __uint_as_float(v[4 * j + 0]) + __uint_as_float(b.x);
    f[4 * j + 1] = __uint_as_float(v[4 * j + 1]) + __uint_as_float(b.y);
    f[4 * j + 2] = __uint_as_float(v[4 * j + 2]) + __uint_as_float(b.z);
    f[4 * j + 3] = __uint_as_float(v[4 * j + 3]) + __uint_as_float(b.w);
  }
  const int sw = (lane >> 1) & 3;
  const uint32_t my_row = stage + lane * 64;
  if (p.residual != nullptr) {             // lane L reads row L, which only lane L overwrites below: no barrier needed
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint4 u = lds128(my_row + ((j ^ sw) << 4));
      const float2 a0 = unpack_bf16x2(u.x), a1 = unpack_bf16x2(u.y), a2 = unpack_bf16x2(u.z), a3 = unpack_bf16x2(u.w);
      f[8 * j + 0] += a0.x; f[8 * j + 1] += a0.y; f[8 * j + 2] += a1.x; f[8 * j + 3] += a1.y;
      f[8 * j + 4] += a2.x; f[8 * j + 5] += a2.y; f[8 * j + 6] += a3.x; f[8 * j + 7] += a3.y;
    }
  }
  // ---- own row -> staging (zeros for pad / out-of-range rows)
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint4 u;
    u.x = valid ? pack_bf16x2(f[8 * j + 0], f[8 * j + 1]) : 0u;
    u.y = valid ? pack_bf16x2(f[8 * j + 2], f[8 * j + 3]) : 0u;
    u.z = valid ? pack_bf16x2(f[8 * j + 4], f[8 * j + 5]) : 0u;
    u.w = valid ? pack_bf16x2(f[8 * j + 6], f[8 * j + 7]) : 0u;
    sts128(my_row + ((j ^ sw) << 4), u);
    if (up_row >= 0 && valid)       // scatter: 64 bytes of this pixel's parity copy (pad rows of the output stay zero)
      *reinterpret_cast<uint4*>(p.out + up_row * p.out_ld + (col0 - up_col0) + 8 * j) = u;
  }
  fence_async_smem();                      // generic-proxy writes -> visible to the TMA store (async proxy)
  __syncwarp();
  // ---- one TMA store for the warp's 32 x 32 tile (pad rows receive zeros, which is what they already hold), and the
  //      hand-over to the statistics warp (release: the tile written by all lanes is ordered before by __syncwarp)
  if (lane == 0) {
    if (warp_row0 < p.rows && p.up2 == 0) tma_store_2d(&p.tmOut, stage, col0, static_cast<int32_t>(warp_row0));
    bulk_commit();
    mbar_arrive(staged);
    if (trow >= 0) IDF_TRACE(4, trow);
  }
}

// GroupNorm partial sums of one staged (bf16-rounded) 32 x 32 tile, taken by a statistics warp (all 32 lanes), so the
// drain warps only move data: column sums written per tile and lane quarter (no cross-warp exchange, fixed summation
// order => deterministic):
//   statsA[(tile*4 + q)][col] = (sum, sumsq) over the window's rows before its last image boundary (all of them when
//                               it has none),
//   statsB[(tile*4 + q)][col] = the same over the rows from that boundary on
//                               (written only when the 32-row window straddles an image boundary).
__device__ __forceinline__ void epilogue_stats_chunk(const ConvKernelParams& p, uint32_t stage, int col0, int n_a, int tile,
                                                     int q, int lane, uint64_t* staged, uint64_t* sdone, uint32_t use) {
  mbar_wait(staged, use & 1u);
  if (p.stats != nullptr && tile < p.m_tiles) {
    // lane -> column pair (2 cp, 2 cp + 1) and row parity hh: rows hh, hh + 2, ..., hh + 30 (even rows occupy banks
    // 0..15, odd rows banks 16..31: conflict-free).  rows < n_a belong to record A, the rest to record B.
    const int cp = lane & 15, hh = lane >> 4;
    const uint32_t col_b = static_cast<uint32_t>((cp & 3) * 4);
    const int cch = cp >> 2;
    uint32_t raw[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int row = 2 * i + hh;       // (row >> 1) & 3 == i & 3
      raw[i] = lds32(stage + static_cast<uint32_t>(row * 64 + ((cch ^ (i & 3)) << 4)) + col_b);
    }
    const int64_t rec = (static_cast<int64_t>(tile) * 4 + q) * p.stats_ld + col0 + 2 * cp;
    if (n_a >= 32) {                                 // warp-uniform fast path: the window lies inside one image
      float sa0 = 0.f, sa1 = 0.f, qa0 = 0.f, qa1 = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float2 w = unpack_bf16x2(raw[i]);
        sa0 += w.x; sa1 += w.y; qa0 = fmaf(w.x, w.x, qa0); qa1 = fmaf(w.y, w.y, qa1);
      }
      sa0 += __shfl_xor_sync(0xffffffffu, sa0, 16); sa1 += __shfl_xor_sync(0xffffffffu, sa1, 16);
      qa0 += __shfl_xor_sync(0xffffffffu, qa0, 16); qa1 += __shfl_xor_sync(0xffffffffu, qa1, 16);
      if (hh == 0) *reinterpret_cast<float4*>(p.stats + 2 * rec) = make_float4(sa0, qa0, sa1, qa1);
    } else {
      float sa0 = 0.f, sa1 = 0.f, qa0 = 0.f, qa1 = 0.f, sb0 = 0.f, sb1 = 0.f, qb0 = 0.f, qb1 = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int row = 2 * i + hh;
        const float2 w = unpack_bf16x2(raw[i]);
        if (row < n_a) { sa0 += w.x; sa1 += w.y; qa0 = fmaf(w.x, w.x, qa0); qa1 = fmaf(w.y, w.y, qa1); }
        else           { sb0 += w.x; sb1 += w.y; qb0 = fmaf(w.x, w.x, qb0); qb1 = fmaf(w.y, w.y, qb1); }
      }
      // combine the two row parities (fixed order: even + odd); lanes 0..15 write 16 B each = 256 B row
      sa0 += __shfl_xor_sync(0xffffffffu, sa0, 16); sa1 += __shfl_xor_sync(0xffffffffu, sa1, 16);
      qa0 += __shfl_xor_sync(0xffffffffu, qa0, 16); qa1 += __shfl_xor_sync(0xffffffffu, qa1, 16);
      sb0 += __shfl_xor_sync(0xffffffffu, sb0, 16); sb1 += __shfl_xor_sync(0xffffffffu, sb1, 16);
      qb0 += __shfl_xor_sync(0xffffffffu, qb0, 16); qb1 += __shfl_xor_sync(0xffffffffu, qb1, 16);
      if (hh == 0) {
        *reinterpret_cast<float4*>(p.stats + 2 * rec) = make_float4(sa0, qa0, sa1, qa1);
        *reinterpret_cast<float4*>(p.stats + p.stats_b_off + 2 * rec) = make_float4(sb0, qb0, sb1, qb1);
      }
    }
  }
  // the sums above consumed every shared-memory load (the global stores precede this asm with its memory clobber)
  __syncwarp();
  if (lane == 0) mbar_arrive(sdone);
}

// Item-level statistics: the same column sums accumulated over ALL tiles of a work item (lane -> column pair and row
// parity as above); a[0..3] = (sum0, sumsq0, sum1, sumsq1) of the rows before `n_a` (record A), a[4..7] of the rest.
__device__ __forceinline__ void epilogue_stats_accum(uint32_t stage, int n_a, int lane, uint64_t* staged, uint64_t* sdone,
                                                     uint32_t use, bool active, float (&a)[8]) {
  mbar_wait(staged, use & 1u);
  if (active) {
    const int cp = lane & 15, hh = lane >> 4;
    const uint32_t col_b = static_cast<uint32_t>((cp & 3) * 4);
    const int cch = cp >> 2;
    uint32_t raw[16];
#pragma unroll
    for (int i = 0; i < 16; ++i)
      raw[i] = lds32(stage + static_cast<uint32_t>((2 * i + hh) * 64 + ((cch ^ (i & 3)) << 4)) + col_b);
    if (n_a >= 32) {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float2 w = unpack_bf16x2(raw[i]);
        a[0] += w.x; a[2] += w.y; a[1] = fmaf(w.x, w.x, a[1]); a[3] = fmaf(w.y, w.y, a[3]);
      }
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float2 w = unpack_bf16x2(raw[i]);
        if (2 * i + hh < n_a) { a[0] += w.x; a[2] += w.y; a[1] = fmaf(w.x, w.x, a[1]); a[3] = fmaf(w.y, w.y, a[3]); }
        else                  { a[4] += w.x; a[6] += w.y; a[5] = fmaf(w.x, w.x, a[5]); a[7] = fmaf(w.y, w.y, a[7]); }
      }
    }
  }
  // all shared-memory loads above have been consumed by the additions: the tile may be rewritten
  asm volatile("" ::"f"(a[0]), "f"(a[1]), "f"(a[2]), "f"(a[3]), "f"(a[4]), "f"(a[5]), "f"(a[6]), "f"(a[7]) : "memory");
  __syncwarp();
  if (lane == 0) mbar_arrive(sdone);
}

__device__ __forceinline__ void epilogue_narrow(const ConvKernelParams& p, const uint32_t (&v)[16], int img, int y,
                                                int x, float cx, float ce, float cn) {
  const int64_t plane = static_cast<int64_t>(p.H) * p.W;
  const int64_t base = static_cast<int64_t>(img) * p.cout * plane + static_cast<int64_t>(y) * p.W + x;
#pragma unroll
  for (int ch = 0; ch < 16; ++ch) {
    if (ch < p.cout) {
      const float e = __uint_as_float(v[ch]) + __ldg(p.bias + ch);
      const int64_t o = base + ch * plane;
      if (p.epilogue == IDF_EPI_SAMPLER) {
        const float xv = p.x_io[o];
        const float nz = (p.noise != nullptr) ? __ldg(p.noise + o) : 0.f;
        p.x_io[o] = cx * xv + ce * e + cn * nz;
        if (p.out_f32 != nullptr) p.out_f32[o] = e;
      } else {
        p.out_f32[o] = e;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// XF = true adds kXfWarps "transform" warps (threads 384..) between the A producer and the UMMA issuers: they
// apply the consumer-side AdaGN (y = act(A*x + B), coefficients per image and channel) to the halo in place, so
// the normalised activation is never written to or read from HBM.
//
// PAIR = true: the kernel runs as clusters of two CTAs (tcgen05 cta_group::2).  A pair owns 2*MT consecutive 128-row
// tiles -- rank r the r-th half, each CTA with its own halo, accumulators and epilogue exactly as in the single-CTA
// kernel -- but every UMMA is one M = 256 instruction issued by the leader (rank 0) over both CTAs' A tiles and a
// weight tile of which each CTA holds HALF (BN/2 rows).  An N = 128 MMA block then reads 16 + 8 KB instead of 16 + 16 KB
// of shared memory per CTA and 256 cycles (N = 64: 16 + 4 instead of 16 + 8 KB per 128 cycles): the operand fetch no
// longer saturates the 128 B/clk shared-memory port, which leaves room for the epilogue staging and the fused-AdaGN
// transform traffic.  Barriers the leader's issuing threads wait on (A ready, B full, accumulator empty) live in the
// leader's shared memory and are signalled by both CTAs; "empty" / "accumulator full" barriers are signalled in both
// CTAs by multicast tcgen05.commit.
// bf16(act(A * x + B)) of one 16-byte granule (8 channels); SiLU(v) = h + h * tanh(h) with h = v / 2 folded into (A, B)
template <bool SILU>
__device__ __forceinline__ uint4 xf_apply(const uint4& u, const float (&A)[8], const float (&B)[8]) {
  const float2 a0 = unpack_bf16x2(u.x), a1 = unpack_bf16x2(u.y), a2 = unpack_bf16x2(u.z), a3 = unpack_bf16x2(u.w);
  float f[8] = {a0.x, a0.y, a1.x, a1.y, a2.x, a2.y, a3.x, a3.y};
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float h = fmaf(f[j], A[j], B[j]);
    if constexpr (SILU) {
      float th;
      asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(h));
      f[j] = fmaf(h, th, h);
    } else {
      f[j] = h;
    }
  }
  uint4 o;
  o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
  o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
  return o;
}

// threads per CTA: [transform warps (XF)] + 8 drain + 4 statistics + A producer, B producer, 2 UMMA issuers / TMEM allocator
__host__ __device__ constexpr int conv_threads(bool xf) { return 32 * ((xf ? kXfWarps : 0) + 8 + 4 + 4); }

template <int BN, int MT, bool XF, bool PAIR>
__global__ void __launch_bounds__(conv_threads(XF), 1) conv_halo_kernel(const __grid_constant__ ConvKernelParams p) {
  using Cfg = HaloCfg<BN, MT, PAIR, XF>;
  constexpr int AS = Cfg::A_STAGES, BS = Cfg::B_STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smA = smem;                                            // AS halo stages
  uint8_t* smB = smem + AS * p.a_stage_bytes;                     // BS weight tiles
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smB + BS * Cfg::B_BYTES);
  uint64_t* a_empty = a_full + AS;
  uint64_t* b_full = a_empty + AS;
  uint64_t* b_empty = b_full + BS;
  uint64_t* tfull = b_empty + BS;
  uint64_t* tempty = tfull + 2;
  uint64_t* a_ready = tempty + 2;                                 // XF: halo transformed (one arrive per transform warp)
  uint64_t* staged = a_ready + AS;                                // [drain warp][tile]: tile written, TMA store issued
  uint64_t* sdone = staged + 16;                                  // [drain warp][tile]: statistics taken
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sdone + 16);
  static_assert(Cfg::NBARS * 8 + 4 <= 2048, "barrier region");
  const uint32_t stage_sa = smem_u32(a_full) + 2048;            // epilogue staging tiles (1024-byte aligned: TMA swizzle)
  const uint32_t bias_sa = stage_sa + kStageBytes;              // bias vector
  const uint32_t rowtab_sa = bias_sa + kBiasBytes;              // XF: row tables

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr int EPI0 = XF ? kXfWarps : 0;          // first of the 8 epilogue warps (multiple of 4: TMEM lane quarters)
  constexpr int STAT0 = EPI0 + 8;                  // four statistics warps, one per lane quarter
  constexpr int W_A = EPI0 + 12, W_B = EPI0 + 13, W_I2 = EPI0 + 14, W_I1 = EPI0 + 15;
  static_assert(EPI0 % 4 == 0, "epilogue warps must start at a multiple of 4");
  // work distribution: `unit0`-th of `n_units` workers (CTAs, or CTA pairs); a pair's super tile is 2 * MT tiles and
  // this CTA owns the `rank`-th half of it
  constexpr int PW = PAIR ? 2 : 1;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;
  const int unit0 = static_cast<int>(blockIdx.x) / PW;
  const int n_units = static_cast<int>(gridDim.x) / PW;

  if (warp == W_A && lane == 0) {
    for (int i = 0; i < p.n_src; ++i) {
      tma_prefetch_desc(&p.tmA[i]);
      if (p.extra_rows[i] > 0) tma_prefetch_desc(&p.tmAx[i]);
    }
    tma_prefetch_desc(&p.tmB);
    if (p.epilogue == IDF_EPI_BF16 && p.up2 == 0) tma_prefetch_desc(&p.tmOut);
  }
  if (warp == W_I1) {
    // ~55 barriers: one per lane and pass instead of a serial loop of one thread (the prologue is on the critical path of
    // every single-round launch, i.e. of every layer at small per-GPU batches).  Layout: a_full[AS] a_empty[AS] b_full[BS]
    // b_empty[BS] tfull[2] tempty[2] a_ready[AS] staged[16] sdone[16]
    for (int i = lane; i < Cfg::NBARS; i += 32) {
      uint32_t cnt = 1;                                               // a_full, b_full, staged, sdone
      if (i >= AS && i < 2 * AS) cnt = Cfg::NI;                        // a_empty
      else if (i >= 2 * AS + BS && i < 2 * AS + 2 * BS + 2) cnt = Cfg::NI;           // b_empty, tfull
      else if (i >= 2 * AS + 2 * BS + 2 && i < 2 * AS + 2 * BS + 4) cnt = PW * 8;    // tempty: one arrive per drain warp
      else if (i >= 2 * AS + 2 * BS + 4 && i < 3 * AS + 2 * BS + 4) cnt = PW * kXfWarps;   // a_ready
      mbar_init(a_full + i, cnt);
    }
    fence_mbar_init();
  }
  if (warp == W_I2) {
    if constexpr (PAIR) {
      tmem_alloc_pair(tmem_slot, Cfg::TMEM_COLS);
      tmem_relinquish_pair();
    } else {
      tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
      tmem_relinquish();
    }
  }
  if (warp >= EPI0 && warp < EPI0 + 8) {   // bias -> shared memory
    const int nb = p.n_tiles * BN;
    for (int i = threadIdx.x - EPI0 * 32; i < nb; i += 256) sts32(bias_sa + 4 * i, __float_as_uint(__ldg(p.bias + i)));
  }
  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all();     // the peer's barriers are initialised before anything signals them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = lds32(smem_u32(tmem_slot));

  const int total = p.m_super * p.n_tiles;    // m_super counts super tiles of PW * MT tiles
  // Programmatic dependent launch: everything above (barriers, TMEM, bias, tap table) touches only constants; the
  // weight (B) producer may also run ahead.  Every other role waits for the producer of its inputs here.
  griddep_launch();
  if (warp != W_B) griddep_wait();

  // Register budget of the XF variant (768 threads: 80 registers each at launch).  The drain warps need ~120 to hold a
  // 32 x 32 fp32 tile plus the prefetched residual without spilling; the single-thread roles and the statistics warps
  // need few.  setmaxnreg (per warpgroup of 4 warps) moves the surplus within the CTA's 6 x 80: 2 x 80 (transform) +
  // 2 x 112 (drain) + 56 (statistics) + 40 (producers, issuers).
  if (warp >= W_A) {
    if constexpr (XF) reg_dec<40>();
  if (warp == W_A) {
    // ------------------------------------------------------------------ A producer: one halo per group
    if (lane == 0) {
      int sa = 0;
      uint32_t pa = 0;
      for (int st = unit0; st < total; st += n_units) {
        const int ms = st / p.n_tiles;
        const int row0 = (ms * PW + static_cast<int>(rank)) * (MT * kBM);
        for (int g = 0; g < p.n_groups; ++g) {
          const int src = p.g_src[g];
          const int ex = p.extra_rows[src];
          mbar_wait(a_empty + sa, pa ^ 1u);
          if (g == 0) IDF_TRACE(0, (st - unit0) / n_units);
          uint8_t* dst = smA + sa * p.a_stage_bytes;
          const int r = row0 + p.g_lo[g];
          const uint32_t bytes = static_cast<uint32_t>((MT * kBM + ex) * 128);
          if constexpr (PAIR && !XF) {
            // the leader's issuing threads wait for BOTH halves: one barrier (the leader's) counts both CTAs' bytes
            const uint32_t bar = mapa_u32(smem_u32(a_full + sa), 0);
            if (leader) mbar_arrive_expect_tx(a_full + sa, 2 * bytes);
#pragma unroll
            for (int m = 0; m < MT; ++m)
              tma_load_2d_pair(dst + m * (kBM * 128), &p.tmA[src], bar, p.g_c0[g], r + m * kBM);
            if (ex > 0) tma_load_2d_pair(dst + MT * (kBM * 128), &p.tmAx[src], bar, p.g_c0[g], r + MT * kBM);
          } else {
            mbar_arrive_expect_tx(a_full + sa, bytes);      // XF: consumed by this CTA's own transform warps
#pragma unroll
            for (int m = 0; m < MT; ++m)
              tma_load_2d(dst + m * (kBM * 128), &p.tmA[src], a_full + sa, p.g_c0[g], r + m * kBM);
            if (ex > 0) tma_load_2d(dst + MT * (kBM * 128), &p.tmAx[src], a_full + sa, p.g_c0[g], r + MT * kBM);
          }
          if (++sa == AS) { sa = 0; pa ^= 1u; }
        }
      }
    }
  } else if (warp == W_B) {
    // ------------------------------------------------------------------ B producer: one weight tile per tap
    if (lane == 0) {
      int sb = 0;
      uint32_t pb = 0;
      for (int st = unit0; st < total; st += n_units) {
        const int nt = st % p.n_tiles;
        for (int t = 0; t < p.n_taps; ++t) {
          mbar_wait(b_empty + sb, pb ^ 1u);
          if constexpr (PAIR) {     // this CTA's half of the weight tile (p.tmB has a box of BN/2 rows); bytes counted by the leader
            if (leader) mbar_arrive_expect_tx(b_full + sb, 2 * Cfg::B_BYTES);
            tma_load_2d_pair(smB + sb * Cfg::B_BYTES, &p.tmB, mapa_u32(smem_u32(b_full + sb), 0), p.t_kb[t] * kBK,
                             nt * BN + static_cast<int>(rank) * (BN / 2));
          } else {
            mbar_arrive_expect_tx(b_full + sb, Cfg::B_BYTES);
            tma_load_2d(smB + sb * Cfg::B_BYTES, &p.tmB, b_full + sb, p.t_kb[t] * kBK, nt * BN);
          }
          if (++sb == BS) { sb = 0; pb ^= 1u; }
        }
      }
    }
  } else if (warp == W_I1 || (warp == W_I2 && Cfg::NI == 2)) {
    // ------------------------------------------------------------------ UMMA issuers
    // One warp per issuer; with MT >= 2 the accumulators are split between two issuing warps so that neither has to
    // sustain more than one MMA per 64 cycles.  Both wait on the same full barriers; every empty / accumulator-full
    // barrier counts one tcgen05.commit per issuer.  The loop runs warp-convergent on warp-uniform values and only
    // the tcgen05 instructions sit under elect.sync: the compiler then keeps descriptors and addresses in uniform
    // registers (3 instructions per MMA).  Inside `if (lane == 0)` every operand went through an ELECT / R2UR.BROADCAST
    // waterfall loop, ~13 instructions per MMA -- the ncu samples showed the issuing thread, not the tensor pipe or the
    // barriers, as the limit of the N = 64 layers.
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_f16(PW * kBM, BN, kFmtBF16);
      constexpr int M_PER = MT / Cfg::NI;
      const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const int m_begin = (warp_u == W_I1) ? 0 : M_PER;
      int sa = 0, sb = 0, iter = 0;
      uint32_t pa = 0, pb = 0;
      const uint32_t b_lo0 = umma_desc_lo(smem_u32(smB));
      for (int st = unit0; st < total; st += n_units, ++iter) {
        const int as = iter & 1;
        if constexpr (PAIR) mbar_wait_cluster(tempty + as, ((iter >> 1) & 1u) ^ 1u);
        else mbar_wait(tempty + as, ((iter >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d0 = tmem_u + static_cast<uint32_t>(as * Cfg::ACC_COLS + m_begin * BN);
        int t = 0;
        // up2 (nearest x2 folded into the conv): column tile nt = output parity (py, px); its taps are the base taps
        // shifted by py rows and px pixels of the input grid
        const int nt_i = st % p.n_tiles;
        const uint32_t nt_shift = p.up2 != 0 ? static_cast<uint32_t>((nt_i >> 1) * p.Wp + (nt_i & 1)) * 8u : 0u;
        uint32_t rel = static_cast<uint32_t>(p.t_rel[0]) * 8u + nt_shift;     // tap view offset in 16-byte units
        for (int g = 0; g < p.n_groups; ++g) {
          if constexpr (PAIR && XF) mbar_wait_cluster(a_ready + sa, pa);   // the peer's transform warps arrive remotely
          else mbar_wait(XF ? a_ready + sa : a_full + sa, pa);
          if constexpr (XF) tc_fence_after();
          if (lane == 0 && g == 0 && warp_u == W_I1) IDF_TRACE(3, iter);
          const uint32_t a_lo0 = umma_desc_lo(smem_u32(smA + sa * p.a_stage_bytes)) +
                                 static_cast<uint32_t>(m_begin * (kBM * 128 / 16));
          const int t_end = t + p.g_ntaps[g];
          for (; t < t_end; ++t) {
            mbar_wait(b_full + sb, pb);
            tc_fence_after();
            const uint32_t a_lo = a_lo0 + rel;           // tap view: any 128-byte row start is legal
            const uint32_t b_lo = b_lo0 + static_cast<uint32_t>(sb) * (Cfg::B_BYTES / 16);
            rel = static_cast<uint32_t>(p.t_rel[t + 1 < IDF_CONV_MAX_KB ? t + 1 : t]) * 8u + nt_shift;   // next tap's offset
            if (elect_one()) {
#pragma unroll
              for (int m = 0; m < M_PER; ++m) {
                if (XF && p.xf_debug == 5) break;      // measurement only: no MMAs (what does the transform cost alone?)
                if constexpr (PAIR)
                  umma_f16_x4_pair(d0 + static_cast<uint32_t>(m * BN), a_lo + static_cast<uint32_t>(m * (kBM * 128 / 16)), b_lo,
                                   idesc, t != 0 ? 1u : 0u);
                else
                  umma_f16_x4(d0 + static_cast<uint32_t>(m * BN), a_lo + static_cast<uint32_t>(m * (kBM * 128 / 16)), b_lo,
                              idesc, t != 0 ? 1u : 0u);
              }
              if constexpr (PAIR) umma_commit_pair(b_empty + sb); else umma_commit(b_empty + sb);
              if (t + 1 == t_end) {
                if constexpr (PAIR) umma_commit_pair(a_empty + sa); else umma_commit(a_empty + sa);
                if (g + 1 == p.n_groups) {
                  if constexpr (PAIR) umma_commit_pair(tfull + as); else umma_commit(tfull + as);
                }
              }
            }
            __syncwarp();
            if (++sb == BS) { sb = 0; pb ^= 1u; }
          }
          if (++sa == AS) { sa = 0; pa ^= 1u; }
        }
        if (lane == 0 && warp_u == W_I1) IDF_TRACE(4, iter);
      }
    }
  }
  } else if (XF && warp < EPI0) {
    // ------------------------------------------------------------------ transform warps (fused AdaGN + SiLU)
    // 32 * kXfWarps threads.  thread -> one physical 16-byte granule column gi and the rows rs, rs + kXfRows, ...; all
    // its rows share (row & 7), so under the 128-byte swizzle it always holds the same logical 8 channels
    // gl = gi ^ (rs & 7).  Per halo the warps first fill a small row table (image of the row relative to the halo's
    // first image, -1 for pad / out-of-range rows) -- each row classified once instead of by every granule's thread --
    // and then stream the halo: one table read, one 16-byte load, 8 x (FMA, tanh, FMA), one 16-byte store per granule.
    // (The first version classified rows inside the streaming loop with float divisions and group shuffles:
    // 114 instructions per granule, and the ncu samples showed the UMMA issuers waiting for these warps 63 % of the time.)
    constexpr int NXT = 32 * kXfWarps;
    const int tt = threadIdx.x;
    const int gi = tt & 7, rs = tt >> 3;
    const int gl = gi ^ (rs & 7);
    const float inv_wp = 1.0f / static_cast<float>(p.Wp), inv_R = 1.0f / static_cast<float>(p.Hp * p.Wp);
    const int R = p.Hp * p.Wp;
    const bool do_silu = p.xf_silu != 0 && p.xf_debug != 2;
    const float cs = do_silu ? 0.5f : 1.0f;          // SiLU(v) = h + h*tanh(h), h = v/2: fold the 1/2 into (A, B)
    const int rows32 = static_cast<int>(p.rows);
    int sa = 0;
    uint32_t pa = 0;
    int cur = -1, cur_cb = -1;           // (image, channel slice) of the coefficients held in A[], B[]
    float A[8], B[8];
    for (int st = unit0; st < total; st += n_units) {
      const int ms = st / p.n_tiles;
      const int row0 = (ms * PW + static_cast<int>(rank)) * (MT * kBM);
      for (int g = 0; g < p.n_groups; ++g) {
        const int cb = p.g_xf[g];
        if (cb != cur_cb) { cur = -1; cur_cb = cb; }
        const int nrows = MT * kBM + p.extra_rows[p.g_src[g]];
        const int rbase = row0 + p.g_lo[g];
        const uint32_t tab = rowtab_sa + static_cast<uint32_t>(sa) * (2u * kXfMaxRows);
        const int rfirst = rbase < 0 ? 0 : rbase;
        const int img0 = __float2int_rd((static_cast<float>(rfirst) + 0.5f) * inv_R);     // image of the halo's first row
        // coefficients of the halo's first image (consecutive items of a CTA lie in different images, so every halo
        // starts with a reload): requested here, consumed after the wait for the halo -- their L2 latency hides behind
        // the row table and the TMA load
        const float2* ctab = p.xf_coef + (cb >= 0 ? cb : 0) + gl * 8;
        const bool pre = cb >= 0 && p.xf_debug != 1 && img0 != cur && rfirst < rows32;
        float4 pc0, pc1, pc2, pc3;
        if (pre) {
          const float4* c4 = reinterpret_cast<const float4*>(ctab + static_cast<int64_t>(img0) * p.xf_ctot);
          pc0 = __ldg(c4); pc1 = __ldg(c4 + 1); pc2 = __ldg(c4 + 2); pc3 = __ldg(c4 + 3);
        }
        if (cb >= 0 && p.xf_debug != 1) {
          // ---- row table (exact float reciprocals: all quotients < 2^22), while the TMA load is still in flight
          for (int i = tt; i < nrows; i += NXT) {
            const int r = rbase + i;
            int inf = -1;
            if (r >= 0 && r < rows32) {                              // outside the tensor: TMA wrote zeros
              const int img = __float2int_rd((static_cast<float>(r) + 0.5f) * inv_R);
              const int rr = r - img * R;
              const int y = __float2int_rd((static_cast<float>(rr) + 0.5f) * inv_wp);
              const int x = rr - y * p.Wp;
              if (x < p.W && y < p.H) inf = img - img0;               // pad rows hold zeros and must keep them
            }
            sts16(tab + 2u * static_cast<uint32_t>(i), static_cast<uint16_t>(inf));
          }
          asm volatile("bar.sync 1, %0;" ::"n"(NXT) : "memory");      // the transform warps only
        }
        mbar_wait(a_full + sa, pa);
        if (tt == 0 && g == 0) IDF_TRACE(1, (st - unit0) / n_units);
        if (pre) {
          cur = img0;
          A[0] = pc0.x * cs; B[0] = pc0.y * cs; A[1] = pc0.z * cs; B[1] = pc0.w * cs;
          A[2] = pc1.x * cs; B[2] = pc1.y * cs; A[3] = pc1.z * cs; B[3] = pc1.w * cs;
          A[4] = pc2.x * cs; B[4] = pc2.y * cs; A[5] = pc2.z * cs; B[5] = pc2.w * cs;
          A[6] = pc3.x * cs; B[6] = pc3.y * cs; A[7] = pc3.z * cs; B[7] = pc3.w * cs;
        }
        if (cb >= 0 && p.xf_debug != 1) {
          const uint32_t base = smem_u32(smA + sa * p.a_stage_bytes) + static_cast<uint32_t>(gi * 16);
          auto reload = [&](int img) {
            cur = img;
            const float4* c4 = reinterpret_cast<const float4*>(ctab + static_cast<int64_t>(img) * p.xf_ctot);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 c = __ldg(c4 + j);
              A[2 * j] = c.x * cs; B[2 * j] = c.y * cs; A[2 * j + 1] = c.z * cs; B[2 * j + 1] = c.w * cs;
            }
          };
          // four rows per trip: table entries and the four loads first; then -- when the valid rows share one image,
          // i.e. in every trip that does not cross an image boundary -- the arithmetic in three phases over 16
          // elements at a time (affines, tanh, second FMA + pack) with predicated stores.  The phases keep 32 independent
          // chains in flight, so that one warp's MUFU phase overlaps the other warps' FMA phases: tools/cu/xf_bench.cu
          // measures 2.09 instead of 2.70 us per 648-row halo for 8 warps (row-by-row code leaves the 8 MUFU results
          // of a granule on the critical path of its store).  The loop exists twice so that the activation is not a
          // per-element branch.
          auto stream = [&](auto silu_tag) {
            constexpr bool SILU = decltype(silu_tag)::value;
#pragma unroll 1
            for (int i0 = rs; i0 < nrows; i0 += 4 * kXfRows) {
              int info[4];
              uint4 u[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const int i = i0 + kXfRows * q;
                const int ic = i < nrows ? i : i0;                    // clamp: the duplicate is never stored
                info[q] = i < nrows ? lds_s16(tab + 2u * static_cast<uint32_t>(ic)) : -1;
                u[q] = lds128(base + static_cast<uint32_t>(ic) * 128u);
              }
              int want = -1;
#pragma unroll
              for (int q = 0; q < 4; ++q) want = info[q] >= 0 ? info[q] : want;      // the last valid row's image
              if (want < 0) continue;
              bool uniform = true;
#pragma unroll
              for (int q = 0; q < 4; ++q) uniform = uniform && (info[q] < 0 || info[q] == want);
              if (uniform) {
                if (want + img0 != cur) reload(want + img0);
#pragma unroll
                for (int q0 = 0; q0 < 4; q0 += 2) {          // two granules (16 independent chains) per phase group
                  float h[2][8];
#pragma unroll
                  for (int q = 0; q < 2; ++q) {
                    const uint4& uu = u[q0 + q];
                    const float2 a0 = unpack_bf16x2(uu.x), a1 = unpack_bf16x2(uu.y), a2 = unpack_bf16x2(uu.z), a3 = unpack_bf16x2(uu.w);
                    const float f[8] = {a0.x, a0.y, a1.x, a1.y, a2.x, a2.y, a3.x, a3.y};
#pragma unroll
                    for (int j = 0; j < 8; ++j) h[q][j] = fmaf(f[j], A[j], B[j]);
                  }
                  if constexpr (SILU) {
                    float th[2][8];
#pragma unroll
                    for (int q = 0; q < 2; ++q)
#pragma unroll
                      for (int j = 0; j < 8; ++j) asm volatile("tanh.approx.f32 %0, %1;" : "=f"(th[q][j]) : "f"(h[q][j]));
#pragma unroll
                    for (int q = 0; q < 2; ++q)
#pragma unroll
                      for (int j = 0; j < 8; ++j) h[q][j] = fmaf(h[q][j], th[q][j], h[q][j]);
                  }
#pragma unroll
                  for (int q = 0; q < 2; ++q) {
                    uint4 o;
                    o.x = pack_bf16x2(h[q][0], h[q][1]); o.y = pack_bf16x2(h[q][2], h[q][3]);
                    o.z = pack_bf16x2(h[q][4], h[q][5]); o.w = pack_bf16x2(h[q][6], h[q][7]);
                    if (info[q0 + q] >= 0) sts128(base + static_cast<uint32_t>(i0 + kXfRows * (q0 + q)) * 128u, o);
                  }
                }
              } else {
#pragma unroll           // (a rolled loop would index u[] / info[] dynamically and push them into local memory)
                for (int q = 0; q < 4; ++q) {
                  if (info[q] < 0) continue;
                  if (info[q] + img0 != cur) reload(info[q] + img0);
                  sts128(base + static_cast<uint32_t>(i0 + kXfRows * q) * 128u, xf_apply<SILU>(u[q], A, B));
                }
              }
            }
          };
          if (do_silu) stream(std::true_type{}); else stream(std::false_type{});
          fence_async_smem();          // generic-proxy writes -> visible to the tensor core's async-proxy reads
        }
        __syncwarp();
        if (tt == 0 && g == 0) IDF_TRACE(2, (st - unit0) / n_units);
        if (lane == 0) {     // hand the stage to the (leader's) UMMA issuers
          if constexpr (PAIR) mbar_arrive_cluster(mapa_u32(smem_u32(a_ready + sa), 0));
          else mbar_arrive(a_ready + sa);
        }
        if (++sa == AS) { sa = 0; pa ^= 1u; }
      }
    }
  } else if (warp >= EPI0 && warp < EPI0 + 8) {
    // ------------------------------------------------------------------ epilogue: 8 drain warps
    if constexpr (XF) reg_inc<112>();
    const int e = warp - EPI0;
    const int q = e & 3;      // TMEM lane quarter (== warp % 4)
    const int half = e >> 2;  // which half of the (m, chunk) work items
    float cx = 0.f, ce = 0.f, cn = 0.f;
    if (p.epilogue == IDF_EPI_SAMPLER) {
      const int step = p.step_ptr ? *p.step_ptr : 0;
      cx = p.coef[3 * step + 0];
      ce = p.coef[3 * step + 1];
      cn = p.coef[3 * step + 2];
    }
    constexpr int CHUNKS = (BN >= 32) ? BN / 32 : 1;
    uint4 res_next[4] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
    if (BN >= 32 && p.residual != nullptr && unit0 < total) {   // first item of the first super tile
      const int ms0 = unit0 / p.n_tiles, nt0 = unit0 - ms0 * p.n_tiles;
      residual_fetch(p, static_cast<int64_t>(ms0 * PW + static_cast<int>(rank)) * MT * kBM + q * 32, nt0 * BN + half * 32, lane,
                     res_next);
    }
    const uint32_t tempty_bar = PAIR ? mapa_u32(smem_u32(tempty), 0) : smem_u32(tempty);   // the leader's barriers
    auto release_acc = [&](int as) {       // all TMEM reads of this warp are complete: one arrive per warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (PAIR) mbar_arrive_cluster_relaxed(tempty_bar + 8u * static_cast<uint32_t>(as));
        else mbar_arrive(tempty + as);
      }
    };
    int iter = 0;
    uint32_t k = 0;         // work items staged so far: tile k & 1, its (k >> 1)-th use
    for (int st = unit0; st < total; st += n_units, ++iter) {
      const int ms = (st / p.n_tiles) * PW + static_cast<int>(rank);     // this CTA's super tile of MT tiles
      const int nt = st % p.n_tiles;
      const int as = iter & 1;
      mbar_wait(tfull + as, (iter >> 1) & 1u);
      tc_fence_after();
      if (e == 0 && lane == 0) IDF_TRACE(5, iter);
      const uint32_t t0 = tmem_base + static_cast<uint32_t>(as * Cfg::ACC_COLS) + (static_cast<uint32_t>(q * 32) << 16);
      if (p.debug_skip_epilogue) {     // measurement only
        release_acc(as);
        continue;
      }
      const float inv_wp = 1.0f / static_cast<float>(p.Wp), inv_hp = 1.0f / static_cast<float>(p.Hp);
#pragma unroll 1
      for (int m = 0; m < MT; ++m) {
        // row bookkeeping once per 128-row tile (exact float reciprocals: all quotients < 2^23)
        const int tile = ms * MT + m;
        const int64_t wr0 = static_cast<int64_t>(tile) * kBM + q * 32;
        const int64_t r = wr0 + lane;
        const int rq = __float2int_rd((static_cast<float>(r) + 0.5f) * inv_wp);
        const int x = static_cast<int>(r) - rq * p.Wp;
        const int img = __float2int_rd((static_cast<float>(rq) + 0.5f) * inv_hp);
        const int y = rq - img * p.Hp;
        const bool valid = (r < p.rows) && (x < p.W) && (y < p.H);
        if constexpr (BN >= 32) {
#pragma unroll 1
          for (int c = half; c < CHUNKS; c += 2) {   // items (m, c) alternate between the halves (CHUNKS is even)
            uint32_t v[32];
            // trace builds: the first drain warp's chunks of the first items go to trace rows 32 + 4 * item + tile
            const int trow = (e == 0 && iter < 8 && m < 4) ? 32 + 4 * iter + m : -1;
            if (lane == 0 && trow >= 0) IDF_TRACE(0, trow);
            tmem_ld_32x32(t0 + static_cast<uint32_t>(m * BN + c * 32), v);
            uint4 res_cur[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) res_cur[i] = res_next[i];
            if (p.residual != nullptr) {             // prefetch the NEXT item's residual (this or the next super tile)
              int nm = m, nc = c + 2, nms = ms, nnt = nt;
              if (nc >= CHUNKS) { nm = m + 1; nc = half; }
              if (nm >= MT) {
                const int nst = st + n_units;
                nms = (nst / p.n_tiles) * PW + static_cast<int>(rank); nnt = nst % p.n_tiles; nm = 0; nc = half;
              }
              residual_fetch(p, (static_cast<int64_t>(nms) * MT + nm) * kBM + q * 32, nnt * BN + nc * 32, lane, res_next);
            }
            tmem_ld_wait();
            if (lane == 0 && trow >= 0) IDF_TRACE(1, trow);
            if (m == MT - 1 && c + 2 >= CHUNKS) release_acc(as);   // last TMEM read of this warp: release the accumulators early
            const uint32_t sl = 2u * e + (k & 1u);
            int64_t up_row = -1;
            if (p.up2 != 0)        // (n, y, x) of the input grid -> parity (nt >> 1, nt & 1) of the (2H) x (2W) output map
              up_row = (static_cast<int64_t>(img) * (2 * p.H + 1) + 2 * y + (nt >> 1)) * (2 * p.W + 1) + 2 * x + (nt & 1);
            epilogue_drain_chunk(p, v, wr0, valid, nt * BN + c * 32, lane, stage_sa + sl * kStageTile, bias_sa, res_cur,
                                 staged + sl, sdone + sl, k >> 1, up_row, nt * BN, trow);
            ++k;
          }
        } else {
          if ((m & 1) == half) {
            uint32_t v[16];
            tmem_ld_32x16(t0 + static_cast<uint32_t>(m * BN), v);
            tmem_ld_wait();
            if (valid) epilogue_narrow(p, v, img, y, x, cx, ce, cn);
          }
        }
      }
      if constexpr (BN < 32) release_acc(as);
    }
    if (BN >= 32 && lane == 0) bulk_wait<0>();     // this warp's TMA stores have been performed
  } else if (warp >= STAT0 && warp < STAT0 + 4) {
    if constexpr (XF) reg_dec<56>();
    if constexpr (BN >= 32) {
    // ------------------------------------------------------------------ statistics (4 warps, one per lane quarter)
    // follows the two drain warps of its quarter through the same item sequence and takes the GroupNorm partial sums
    // of every tile they stage; it runs even when no statistics are wanted so that the tile hand-shake stays in step
    const int q = warp - STAT0;
    constexpr int CHUNKS = BN / 32;
    const int R = p.Hp * p.Wp;
    const float inv_R = 1.0f / static_cast<float>(R);
    uint32_t k = 0;          // items per drain warp so far (both drain warps of a quarter advance in lock step)
    if (!p.debug_skip_epilogue && p.stats_item != 0) {
      // one record per (work item, lane quarter) instead of one per 32-row window: MT times fewer records to write
      // here and to reduce in the consumer's prologue.  Used when an item spans at most two images (rows per image
      // >= rows per item); record index = item * 4 + q, A / B split at the end of the image the ITEM starts in.
      for (int st = unit0; st < total; st += n_units) {
        const int ms = (st / p.n_tiles) * PW + static_cast<int>(rank);
        const int nt = st % p.n_tiles;
        const int64_t item_row0 = static_cast<int64_t>(ms) * (MT * kBM);
        const int img_i = __float2int_rd((static_cast<float>(item_row0) + 0.5f) * inv_R);
        const int64_t boundary = static_cast<int64_t>(img_i + 1) * R;
        const bool active = p.stats != nullptr && item_row0 < p.rows;
        float acc[CHUNKS][8];
#pragma unroll
        for (int c = 0; c < CHUNKS; ++c)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[c][j] = 0.f;
#pragma unroll 1
        for (int m = 0; m < MT; ++m) {
          const int64_t wr0 = item_row0 + m * kBM + q * 32;
          const int64_t left = boundary - wr0;
          const int n_a = left >= 32 ? 32 : (left <= 0 ? 0 : static_cast<int>(left));
#pragma unroll
          for (int c = 0; c < CHUNKS; ++c) {
            const uint32_t kk = k + static_cast<uint32_t>(c >> 1);
            const uint32_t sl = 2u * ((c & 1) * 4 + q) + (kk & 1u);
            epilogue_stats_accum(stage_sa + sl * kStageTile, n_a, lane, staged + sl, sdone + sl, kk >> 1, active, acc[c]);
          }
          k += CHUNKS / 2;
        }
        if (active) {
          const int cp = lane & 15, hh = lane >> 4;
          const bool straddles = boundary < item_row0 + MT * kBM;
#pragma unroll
          for (int c = 0; c < CHUNKS; ++c) {
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[c][j] += __shfl_xor_sync(0xffffffffu, acc[c][j], 16);   // even + odd rows
            if (hh == 0) {
              const int64_t rec = (static_cast<int64_t>(ms) * 4 + q) * p.stats_ld + nt * BN + c * 32 + 2 * cp;
              *reinterpret_cast<float4*>(p.stats + 2 * rec) = make_float4(acc[c][0], acc[c][1], acc[c][2], acc[c][3]);
              if (straddles)
                *reinterpret_cast<float4*>(p.stats + p.stats_b_off + 2 * rec) = make_float4(acc[c][4], acc[c][5], acc[c][6], acc[c][7]);
            }
          }
        }
      }
    } else if (!p.debug_skip_epilogue) {
      for (int st = unit0; st < total; st += n_units) {
        const int ms = (st / p.n_tiles) * PW + static_cast<int>(rank);
        const int nt = st % p.n_tiles;
#pragma unroll 1
        for (int m = 0; m < MT; ++m) {
          const int tile = ms * MT + m;
          const int64_t wr0 = static_cast<int64_t>(tile) * kBM + q * 32;
          // split at the window's LAST image boundary: with R < 32 a window can touch three images, and the rows before
          // an earlier boundary are then pad rows (zeros; the plan rejects geometries where they are not)
          const int64_t wr_last = (wr0 + 31 < p.rows) ? wr0 + 31 : p.rows - 1;
          const int img_l = __float2int_rd((static_cast<float>(wr_last) + 0.5f) * inv_R);
          const int64_t last_bnd = static_cast<int64_t>(img_l) * R;
          const int n_a = last_bnd > wr0 ? static_cast<int>(last_bnd - wr0) : 32;
#pragma unroll 1
          for (int c = 0; c < CHUNKS; ++c, k += (c & 1) ? 0u : 1u) {     // chunk c belongs to drain warp (c & 1) * 4 + q
            const uint32_t sl = 2u * ((c & 1) * 4 + q) + (k & 1u);
            epilogue_stats_chunk(p, stage_sa + sl * kStageTile, nt * BN + c * 32, n_a, tile, q, lane, staged + sl, sdone + sl,
                                 k >> 1);
          }
        }
      }
    }
    }
  }

  tc_fence_before();
  if constexpr (PAIR) cluster_sync_all();    // neither CTA may exit (or free TMEM) while the other still uses its memory
  else __syncthreads();
  if (warp == W_I2) {
    tc_fence_after();
    if constexpr (PAIR) tmem_dealloc_pair(tmem_base, Cfg::TMEM_COLS);
    else tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int BN, int MT, bool XF, bool PAIR>
static cudaError_t launch_cfg(const ConvKernelParams& p, int grid, cudaStream_t stream) {
  using Cfg = HaloCfg<BN, MT, PAIR, XF>;
  const uint32_t smem = conv_smem_bytes(p.a_stage_bytes, Cfg::A_STAGES, Cfg::B_STAGES, Cfg::B_BYTES, XF);
  static uint32_t attr_smem = 0;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(conv_halo_kernel<BN, MT, XF, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    attr_smem = smem;
  }
  return launch_kernel(conv_halo_kernel<BN, MT, XF, PAIR>, dim3(grid), dim3(conv_threads(XF)), smem, stream, g_pdl != 0,
                       PAIR ? 2 : 0, p);
}

template <bool XF, bool PAIR>
static cudaError_t launch_sel(const ConvKernelParams& p, int block_n, int mt, int grid, cudaStream_t stream) {
  const int key = block_n * 10 + mt;
  switch (key) {
    case 1281: return launch_cfg<128, 1, XF, PAIR>(p, grid, stream);
    case 1282: return launch_cfg<128, 2, XF, PAIR>(p, grid, stream);
    case 641: return launch_cfg<64, 1, XF, PAIR>(p, grid, stream);
    case 642: return launch_cfg<64, 2, XF, PAIR>(p, grid, stream);
    case 644: return launch_cfg<64, 4, XF, PAIR>(p, grid, stream);
    default: break;
  }
  if constexpr (!PAIR) {
    switch (key) {
      case 161: return launch_cfg<16, 1, XF, false>(p, grid, stream);
      case 164: return launch_cfg<16, 4, XF, false>(p, grid, stream);
      default: break;
    }
  }
  return cudaErrorInvalidValue;
}

cudaError_t launch_conv_igemm(const ConvKernelParams& p, int block_n, int mt, bool xform, bool pair, int grid,
                              cudaStream_t stream) {
  if (pair) return xform ? launch_sel<true, true>(p, block_n, mt, grid, stream) : launch_sel<false, true>(p, block_n, mt, grid, stream);
  return xform ? launch_sel<true, false>(p, block_n, mt, grid, stream) : launch_sel<false, false>(p, block_n, mt, grid, stream);
}

// shared-memory need of a configuration (host side, for plan validation)
uint32_t conv_config_smem(int block_n, int mt, int a_stage_bytes, bool pair, bool xf) {
  return conv_smem_bytes(a_stage_bytes, conv_a_stages(mt, xf), conv_b_stages(block_n), block_n * kBK * 2 / (pair ? 2 : 1), xf);
}

}  // namespace idf
