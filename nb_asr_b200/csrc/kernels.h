// Internal declarations shared between the translation units of libnbasr.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/nbasr.h"

// Environment switches are read ONCE, when the library is loaded (api.cu), never on the call path.
enum NbasrEnvFlag { NBASR_ENV_FORCE_SIMT = 0, NBASR_ENV_NO_PDL, NBASR_ENV_GCONV_NO_PREFETCH, NBASR_ENV_LSTM_SS, NBASR_ENV_DEBUG,
                    NBASR_ENV_GEMM_DIRECT_EPI, NBASR_ENV_COUNT };
bool nbasr_env_flag(int which);
int nbasr_env_gemm_bn();          // NBASR_GEMM_BN tuning override (0 = cost model)
int nbasr_env_gemm_l2pf();        // NBASR_GEMM_L2PF: K blocks the GEMM producer L2-prefetches ahead of its loads

// "Do once per device" latch for cudaFuncSetAttribute(MaxDynamicSharedMemorySize): the attribute is per (function, device),
// so a process that drives several GPUs (Trainer(gpus=[k]) with k != 0) must opt in on each of them.
// Usage keeps the classic shape:  static DevOnce attr; if (!attr) { ...set...; attr = true; }
struct DevOnce {
  unsigned long long mask = 0;
  static int dev() { int d = 0; cudaGetDevice(&d); return d & 63; }
  bool operator!() const { return !((mask >> dev()) & 1ull); }
  DevOnce& operator=(bool v) { if (v) mask |= 1ull << dev(); return *this; }
};

// Launch with the programmatic-stream-serialization attribute (see pdl_wait() in common.cuh) and an optional cluster
// width.  NBASR_NO_PDL=1 disables the attribute (plain stream ordering).
#ifdef __CUDACC__
#include <utility>
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster_x,
                              Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[2];
  int n = 0;
  if (!nbasr_env_flag(NBASR_ENV_NO_PDL)) {
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (cluster_x > 1) {
    at[n].id = cudaLaunchAttributeClusterDimension;
    at[n].val.clusterDim.x = cluster_x; at[n].val.clusterDim.y = 1; at[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = at; cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}
#endif

// C[i, j] = sum_{kb, kr} A[ib*a_ib + ir*a_ir + kb*a_kb + kr*a_kr] * B[j*b_j + kb*b_kb + kr*b_kr]
// with i = (ib, ir); output row rho = o_r0 + ib*o_bs + ir*o_rs.
struct SimtGemmArgs {
  const void* a;
  int a_dtype;
  int64_t a_ib, a_ir, a_kb, a_kr;
  int nib, nir;
  const void* b;
  int b_dtype;
  int64_t b_j, b_kb, b_kr;
  int nkb, nkr, N;
  int64_t o_r0, o_bs, o_rs;
  nbasr_epilogue epi;
};
int simt_gemm_launch(const SimtGemmArgs& a, cudaStream_t st);

// tcgen05 dense GEMMs on CTA pairs, cta_group::2 (gemm2_sm100.cu)
int sm100_gemm_tn_pair(const nbasr_gemm* p, cudaStream_t st);
int sm100_gemm_wgrad_pair(const nbasr_wgrad* p, cudaStream_t st);

// cached TMA descriptor of 2-byte elements (rank 2/3, 128B swizzle); strides in elements for dims 1..rank-1 (tma_maps.cu)
struct CUtensorMap_st;
int sm100_get_map(const void* base, int rank, const uint64_t* dims, const int64_t* strides_el, const uint32_t* box,
                  CUtensorMap_st* out, int swizzle128 = 1);

// tcgen05 grouped conv (gconv_sm100.cu)
int sm100_gconv_fwd(const nbasr_gconv* p, cudaStream_t st);
// x_f16: x is fp16 holding x / x_scale, converted to bf16 in shared memory (otherwise bf16, x_scale unused)
int sm100_gconv_wgrad(const void* dz, const void* x, int x_f16, float x_scale, int B, int T, int Tp, int C, int cpg, int ktaps,
                      int off0, int dstep, float* dw, float* dbias, cudaStream_t st);

// cluster / tcgen05 LSTM recurrence (lstm_sm100.cu)
int sm100_lstm_fwd(const float* gx, const void* w_packed, int T, int B, int H, void* h_seq, int h_dtype, int64_t h_bs, int64_t h_rs,
                   float* gates, float* cstate, cudaStream_t st);
int sm100_lstm_bwd(const float* dh_seq, int64_t dh_bs, int64_t dh_rs, const void* w_packed, const float* gates, const float* cstate,
                   int T, int B, int H, float* dgx, void* dgx_bf16, cudaStream_t st);

// packed-fp32x2 16-bit LayerNorm (layernorm2.cu); f16 / x_f16: the forward activations are scaled fp16 (see nbasr.h)
int ln2_fwd(const void* x, void* y, int f16, int B, int T, int Tp, int C, const float* gamma, const float* beta, float eps, float* mean,
            float* rstd, float out_scale, void* y2, cudaStream_t st);
int ln2_bwd(const void* dy, const void* x, int x_f16, float x_scale, const float* mean, const float* rstd, const float* gamma, int B, int T,
            int Tp, int C, void* dx, void* dx2, const uint32_t* mask2, float scale2, int64_t mask_rows, int mask2_w, float* dgamma,
            float* dbeta, cudaStream_t st);
