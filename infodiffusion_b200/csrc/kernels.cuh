// Internal declarations shared by the kernel translation units and the C-ABI shim (capi.cu).
#pragma once
#include "../../include/idf_b200.h"
#include "ptx.cuh"

namespace idf {

typedef __nv_bfloat16 bf16;

constexpr int kBM = 128;  // output rows (pixels) per tile == UMMA M
constexpr int kBK = 64;   // K elements per k-block == one 128-byte swizzle row

constexpr int kMaxGroups = 40;   // halo loads per work item: (source, 64-channel slice, tap cluster); 1024 + 1024 channels = 32

struct alignas(64) ConvKernelParams {
  CUtensorMap tmA[IDF_CONV_MAX_SRC];    // box {64, 128 rows}
  CUtensorMap tmAx[IDF_CONV_MAX_SRC];   // box {64, extra_rows[src]} -- tail of the halo
  CUtensorMap tmB;                      // box {64, BN} (CTA pairs: {64, BN/2}, each CTA loads its half)
  CUtensorMap tmOut;                    // bf16 epilogue: output [rows, out_ld], box {32 cols, 32 rows}, SWIZZLE_64B (TMA store)
  int32_t n_src;
  int32_t extra_rows[IDF_CONV_MAX_SRC]; // halo rows beyond 128*MT (multiple of 8, 0 for 1x1 sources)
  // K loop = groups (one halo load each: source, 64-channel slice, cluster of taps) x taps
  int32_t n_groups;
  int32_t g_src[kMaxGroups];
  int32_t g_c0[kMaxGroups];
  int32_t g_lo[kMaxGroups];             // row offset of the halo start relative to the tile's first row
  int32_t g_ntaps[kMaxGroups];
  int32_t n_taps;                       // total taps == number of 64-wide k-blocks
  int32_t t_rel[IDF_CONV_MAX_KB];       // tap row offset relative to its group's halo start (>= 0)
  int32_t t_kb[IDF_CONV_MAX_KB];        // k-block index of the tap in the packed weight matrix
  int32_t a_stage_bytes;                // bytes of one halo stage (multiple of 1024)
  int32_t m_super, n_tiles;             // super tiles of MT*128 rows (CTA pairs: 2*MT*128 rows); N tiles
  int32_t m_tiles;                      // 128-row tiles
  float* stats;                         // optional GroupNorm partial sums: records A then records B, each
                                        // [m_tiles*4 (32-row windows)][out_ld][2] fp32 (sum, sumsq)
  int64_t stats_b_off;                  // float offset of the B records
  int32_t stats_ld;                     // columns of a statistics record row (out_ld; up2: cout_pad = 4 parity planes)
  int32_t up2;                          // nearest x2 upsampling folded in: column tile = output parity, scatter epilogue
  int32_t stats_item;                   // 1: one record per (work item of MT tiles, lane quarter) instead of per window
  int32_t debug_skip_epilogue;          // measurement only: epilogue warps drain nothing (main-loop ceiling)
  int64_t rows;
  int32_t Hp, Wp, H, W;
  int32_t cout;
  int32_t epilogue;
  const float* bias;
  bf16* out;
  int32_t out_ld;
  const bf16* residual;
  int32_t res_ld;
  float* out_f32;
  float* x_io;
  const float* noise;
  const float* coef;
  const int32_t* step_ptr;
  // fused AdaGN (+SiLU) on the A operand: halo groups with g_xf[g] >= 0 are rewritten in shared memory as
  // bf16(act(A*x + B)) with (A, B) = xf_coef[image][g_xf[g] + channel] before the MMAs read them
  const float2* xf_coef;                // [batch][xf_ctot] (A, B)
  int32_t xf_ctot;
  int32_t xf_silu;
  int32_t g_xf[kMaxGroups];             // channel base of the group's 64-channel slice in xf_coef, or -1
  int32_t xf_debug;                     // measurement only (idf_set_option "xf_debug")
};

constexpr int kWgMaxClusters = 9;
struct alignas(64) WgradKernelParams {
  CUtensorMap tmDY;                 // dY [rows, Cout]  box {64, 128}
  CUtensorMap tmX;                  // X  [rowsX, Cin]  box {64, 136}
  // work unit u = (128-wide co tile u / (n_ci * n_cl), ci chunk (u / n_cl) % n_ci of ci_step channels, tap cluster u % n_cl)
  int32_t n_units, n_cl, n_ci, ci_step;
  int32_t c_ntap[kWgMaxClusters], c_base[kWgMaxClusters];           // per tap cluster: taps, X row offset of the halo
  int32_t c_rel[kWgMaxClusters * 3], c_tap[kWgMaxClusters * 3];     // ... each tap's row shift within it and its index
  int32_t n_kb, kb_per_slab;
  int32_t cout, cin, ntaps;
  float* dw;                        // fp32 [Cout, ntaps, Cin], accumulated with atomics
  float* partials;                  // ordered variant: fp32 [slabs][Cout, ntaps, Cin], reduced into dw in slab order
};
// partials == nullptr or a single slab: one launch; otherwise the ordered kernel and the slab reduction
cudaError_t launch_wgrad(const WgradKernelParams& p, int grid, int slabs, int num_sms, cudaStream_t stream);

static_assert(sizeof(ConvKernelParams) <= 4000, "kernel parameters are limited to 4 KB");

// library-wide options (idf_set_option), defined in conv_igemm.cu
extern int g_pdl;
extern int g_xf_debug;

// kernel<<<grid, block, smem, stream>>>(args...), with programmatic dependent launch when `pdl` is set (the kernel's
// prologue may overlap its predecessor's tail; it orders its dependent reads with griddepcontrol.wait) and as clusters
// of `cluster` CTAs along x when `cluster` > 0.  The arguments are converted to the kernel's parameter types, as by
// cudaLaunchKernelEx, not deduced against them.
template <typename... KernelParams, typename... Args>
cudaError_t launch_kernel(void (*kernel)(KernelParams...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                          bool pdl, int cluster, const Args&... args) {
  cudaLaunchAttribute attr[2];
  unsigned na = 0;
  if (pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  if (cluster > 0) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = cluster;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cfg.attrs = attr;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

cudaError_t launch_conv_igemm(const ConvKernelParams& p, int block_n, int mt, bool xform, bool pair, int grid, cudaStream_t stream);
cudaError_t launch_adagn_coef(const idf_adagn_args& a, float* coef_out, cudaStream_t stream);
uint32_t conv_config_smem(int block_n, int mt, int a_stage_bytes, bool pair, bool xf);
cudaError_t launch_adagn(const idf_adagn_args& a, cudaStream_t stream);
cudaError_t launch_adagn_bwd(const idf_adagn_bwd_args& b, int num_sms, cudaStream_t stream);
int64_t adagn_bwd_ws_floats(int batch, int C);
cudaError_t launch_attn_small(const bf16* qkv, bf16* out, int batch, int H, int W, int d, float scale, cudaStream_t stream);
cudaError_t launch_attn_generic(const bf16* qkv, bf16* out, int batch, int H, int W, int d, float scale, cudaStream_t stream);
cudaError_t launch_attn_v2(const CUtensorMap& tm, bf16* out, int batch, int H, int W, int d, float scale,
                           cudaStream_t stream);
cudaError_t launch_attn_bwd(const CUtensorMap& tmQKV, const CUtensorMap& tmDO, const CUtensorMap& tmPr,
                            const CUtensorMap& tmDSr, const CUtensorMap& tmDSc, bf16* P, bf16* dS, bf16* dqkv, int batch,
                            int H, int W, int d, float scale, cudaStream_t stream);
cudaError_t launch_attn_small_bwd(const bf16* qkv, const bf16* dout, bf16* dqkv, int batch, int H, int W, int d, float scale,
                                  cudaStream_t stream);
cudaError_t launch_linear_f32(const float* x, int64_t ldx, const float* w, const float* b, float* y, int64_t ldy,
                              int M, int N, int K, int silu_in, cudaStream_t stream);
cudaError_t launch_gemm_f32(const float* A, int64_t lda, int transA, const float* B, int64_t ldb, int transB, float* Cm,
                            int64_t ldc, int M, int N, int K, int accumulate, cudaStream_t stream);
struct ClipAdamWParams {
  void* const* params; const void* const* grads; void* const* exp_avg; void* const* exp_avg_sq;
  const long long* numel; const int* chunk_tensor; const int* chunk_offset;
  int n_chunks;
  const float* bias_corrections;
  float lr, beta1, beta2, eps, weight_decay, max_norm;
  float* partial; float* norm_out;
};
cudaError_t launch_clip_adamw(const ClipAdamWParams& p, cudaStream_t stream);
cudaError_t launch_scale_ln_silu(const float* y, long long ldy, const float* cond, long long cond_stride,
                                 long long cond_step_stride, const int* step_ptr, const float* gamma, const float* beta,
                                 float eps, float* out, long long ldo, int M, int N, int apply_silu, cudaStream_t stream);
cudaError_t launch_to_uint8_hwc(const float* x, uint8_t* out, int batch, int C, int H, int W, cudaStream_t stream);
cudaError_t launch_copy2d_f32(const float* src, long long lds, float* dst, long long ldd, int M, int N, cudaStream_t stream);
cudaError_t launch_gather_elems(const float* src, const int* idx, const int* idx2, void* dst, long long n, bool dst_bf16,
                                bool accumulate, int num_sms, cudaStream_t stream);
cudaError_t launch_gather_rows(const float* table, const int64_t* idx, float* y, int M, int N, cudaStream_t stream);
cudaError_t launch_im2col_head(const float* x, bf16* out, int batch, int C, int H, int W, cudaStream_t stream);
cudaError_t launch_upsample2x(const bf16* in, bf16* out, int batch, int H, int W, int C, cudaStream_t stream);
cudaError_t launch_space_to_depth(const bf16* in, bf16* out, int batch, int H, int W, int C, cudaStream_t stream);
cudaError_t launch_nchw_to_padflat(const float* x, bf16* out, int batch, int C, int H, int W, int ld, cudaStream_t stream);
cudaError_t launch_upsample2x_bwd(const bf16* dout, bf16* din, int batch, int H, int W, int C, int accumulate, cudaStream_t stream);
cudaError_t launch_depth_to_space(const bf16* dph, bf16* din, int batch, int H, int W, int C, int accumulate, cudaStream_t stream);
cudaError_t launch_colsum(const bf16* m, float* out, long long rows, int C, int num_sms, cudaStream_t stream);
// ordered variants (torch's deterministic mode): partials in `ws`, combined in index order by the last-arriving CTA, which
// takes a ticket from the caller-zeroed `tickets` and resets it to zero
int64_t colsum_ws_floats(long long rows, int C, int num_sms);
cudaError_t launch_colsum_ordered(const bf16* m, float* out, long long rows, int C, int num_sms, float* ws, unsigned* tickets,
                                  cudaStream_t stream);
int64_t gemm_f32_ws_floats(int M, int N, int K);
cudaError_t launch_gemm_f32_ordered(const float* A, int64_t lda, int transA, const float* B, int64_t ldb, int transB, float* Cm,
                                    int64_t ldc, int M, int N, int K, int accumulate, float* ws, unsigned* tickets,
                                    cudaStream_t stream);
cudaError_t launch_mmd_ordered(const float* x, const float* y, float* loss, float* grad_y, int B, int D, float* ws,
                               unsigned* tickets, cudaStream_t stream);
cudaError_t launch_padflat_to_nchw(const bf16* in, float* y, int batch, int C, int H, int W, cudaStream_t stream);
cudaError_t launch_sampler_update(float* x, const float* eps, const float* noise, const float* coef,
                                  const int32_t* step_ptr, int64_t n, cudaStream_t stream);
cudaError_t launch_mmd(const float* x, const float* y, float* loss, float* grad_y, int B, int D, cudaStream_t stream);

}  // namespace idf
