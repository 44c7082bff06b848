// Grouped conv edges (ops.py:73-76: Conv1d(C, C, k, dilation, groups=100) -> cpg = C/100 in {6,8,10,12}).
// Channels-last SIMT kernels: forward (also used for the input gradient with group-transposed
// weights and negated tap offsets) and weight gradient.  ~15-42 FLOP/B: HBM-bound in bf16.
#include <algorithm>

#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int G_TT = 64;   // frames per CTA tile
constexpr int G_FB = 16;   // frames per thread work item
constexpr int G_MAXHALO = 12;
constexpr int G_NT = 256;

__host__ __device__ inline int slab_channels(int cpg) {
  // multiple of 32 (epilogue chunk) and of cpg (whole groups)
  return cpg == 10 ? 160 : 96;
}
__host__ __device__ inline int wpitch(int cpg, int ktaps) {
  int p = cpg * ktaps;
  return (p & 1) ? p : p + 1;
}

template <typename T>
__global__ void __launch_bounds__(G_NT) gconv_fwd_kernel(nbasr_gconv p) {
  extern __shared__ float smem[];
  const int CS = slab_channels(p.cpg);
  const int halo = (p.ktaps - 1) * p.dstep;
  const int WP = wpitch(p.cpg, p.ktaps);
  float* xs = smem;                                  // (G_TT + halo) x CS
  float* ws = xs + (G_TT + G_MAXHALO) * CS;          // CS x WP
  float* os = ws + CS * WP;                          // G_TT x (CS+1)
  const int tid = threadIdx.x;
  const int c_lo = blockIdx.x * CS;
  const int cs = min(CS, p.C - c_lo);                // valid channels in this slab (multiple of cpg)
  const int t0 = blockIdx.y * G_TT;
  const int b = blockIdx.z;
  const T* __restrict__ x = reinterpret_cast<const T*>(p.x);

  // stage weights of the slab: w[(c_lo+co)][i][j]
  for (int idx = tid; idx < cs * p.cpg * p.ktaps; idx += G_NT) {
    int co = idx / (p.cpg * p.ktaps), rem = idx % (p.cpg * p.ktaps);
    ws[co * WP + rem] = reinterpret_cast<const float*>(p.w)[(int64_t)(c_lo + co) * p.cpg * p.ktaps + rem];
  }
  // stage input rows t0+off0 .. t0+off0+G_TT+halo-1 (zero outside [0,T))
  const int nrow = G_TT + halo;
  const int vec = cs >> 3;  // cs % 8 == 0 for every (C, cpg) of the search space
  for (int idx = tid; idx < nrow * vec; idx += G_NT) {
    int r = idx / vec, g8 = idx % vec;
    int t = t0 + p.off0 + r;
    float v[8];
    if (t >= 0 && t < p.T) load8(x + ((int64_t)b * p.Tp + NBASR_PAD_L + t) * p.C + c_lo + g8 * 8, v);
    else {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = 0.f;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) xs[r * CS + g8 * 8 + i] = v[i];
  }
  __syncthreads();

  const int nfb = G_TT / G_FB;
  for (int item = tid; item < cs * nfb; item += G_NT) {
    int co = item % cs, fb = item / cs;
    int g0 = (co / p.cpg) * p.cpg;
    float acc[G_FB];
#pragma unroll
    for (int f = 0; f < G_FB; ++f) acc[f] = 0.f;
    for (int i = 0; i < p.cpg; ++i) {
      float xw[G_FB + G_MAXHALO];
#pragma unroll
      for (int f = 0; f < G_FB + G_MAXHALO; ++f)
        xw[f] = (f < G_FB + halo) ? xs[(fb * G_FB + f) * CS + g0 + i] : 0.f;
      const float* wr = ws + co * WP + i * p.ktaps;
      if (p.dstep == 1) {
#pragma unroll
        for (int j = 0; j < 7; ++j) {
          if (j < p.ktaps) {
            float w = wr[j];
#pragma unroll
            for (int f = 0; f < G_FB; ++f) acc[f] = fmaf(xw[f + j], w, acc[f]);
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < 7; ++j) {
          if (j < p.ktaps) {
            float w = wr[j];
#pragma unroll
            for (int f = 0; f < G_FB; ++f) acc[f] = fmaf(xw[f + 2 * j], w, acc[f]);
          }
        }
      }
    }
#pragma unroll
    for (int f = 0; f < G_FB; ++f) os[(fb * G_FB + f) * (CS + 1) + co] = acc[f];
  }
  __syncthreads();
  const int nch = (cs + 31) >> 5;
  for (int item = tid; item < G_TT * nch; item += G_NT) {
    int r = item / nch, ch = item % nch;
    int t = t0 + r;
    if (t >= p.T) continue;
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = (ch * 32 + i < cs) ? os[r * (CS + 1) + ch * 32 + i] : 0.f;
    int64_t rho = (int64_t)b * p.Tp + NBASR_PAD_L + t;
    epilogue_chunk(p.epi, rho, c_lo + ch * 32, p.C, v);
  }
}

constexpr int W_PAIRS = 7;  // (co,i) pairs per thread: slab pairs <= 160*10 = 1600 <= 7*256
constexpr int W_FB = 8;

// X is staged as x * x_scale (x_scale = 1/S for the forward's scaled fp16 activations)
template <typename TD, typename TX>
__global__ void __launch_bounds__(G_NT) gconv_wgrad_kernel(const TD* __restrict__ dz, const TX* __restrict__ x, float x_scale,
                                                           int B, int Tt, int Tp, int C, int cpg, int ktaps, int off0,
                                                           int dstep, float* __restrict__ dw) {
  extern __shared__ float smem[];
  const int CS = slab_channels(cpg);
  const int halo = (ktaps - 1) * dstep;
  float* xs = smem;                                 // (G_TT + halo) x CS
  float* ds = xs + (G_TT + G_MAXHALO) * CS;         // G_TT x CS
  const int tid = threadIdx.x;
  const int c_lo = blockIdx.x * CS;
  const int cs = min(CS, C - c_lo);
  const int b = blockIdx.y;
  const int npairs = cs * cpg;
  float acc[W_PAIRS][7];
#pragma unroll
  for (int q = 0; q < W_PAIRS; ++q)
#pragma unroll
    for (int j = 0; j < 7; ++j) acc[q][j] = 0.f;
  const int vec = cs >> 3;
  for (int t0 = 0; t0 < Tt; t0 += G_TT) {
    __syncthreads();
    for (int idx = tid; idx < (G_TT + halo) * vec; idx += G_NT) {
      int r = idx / vec, g8 = idx % vec;
      int t = t0 + off0 + r;
      float v[8];
      if (t >= 0 && t < Tt) load8(x + ((int64_t)b * Tp + NBASR_PAD_L + t) * C + c_lo + g8 * 8, v);
      else {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = 0.f;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) xs[r * CS + g8 * 8 + i] = v[i] * x_scale;
    }
    for (int idx = tid; idx < G_TT * vec; idx += G_NT) {
      int r = idx / vec, g8 = idx % vec;
      int t = t0 + r;
      float v[8];
      if (t < Tt) load8(dz + ((int64_t)b * Tp + NBASR_PAD_L + t) * C + c_lo + g8 * 8, v);
      else {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = 0.f;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) ds[r * CS + g8 * 8 + i] = v[i];
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < W_PAIRS; ++q) {
      int pair = tid + q * G_NT;
      if (pair < npairs) {
        int co = pair / cpg, i = pair % cpg;
        int gi = (co / cpg) * cpg + i;
        for (int fb = 0; fb < G_TT / W_FB; ++fb) {
          float xw[W_FB + G_MAXHALO], dv[W_FB];
#pragma unroll
          for (int f = 0; f < W_FB + G_MAXHALO; ++f) xw[f] = (f < W_FB + halo) ? xs[(fb * W_FB + f) * CS + gi] : 0.f;
#pragma unroll
          for (int f = 0; f < W_FB; ++f) dv[f] = ds[(fb * W_FB + f) * CS + co];
          if (dstep == 1) {
#pragma unroll
            for (int j = 0; j < 7; ++j)
#pragma unroll
              for (int f = 0; f < W_FB; ++f) acc[q][j] = fmaf(dv[f], xw[f + j], acc[q][j]);
          } else {
#pragma unroll
            for (int j = 0; j < 7; ++j)
#pragma unroll
              for (int f = 0; f < W_FB; ++f) acc[q][j] = fmaf(dv[f], xw[f + 2 * j], acc[q][j]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int q = 0; q < W_PAIRS; ++q) {
    int pair = tid + q * G_NT;
    if (pair < npairs) {
      int co = pair / cpg, i = pair % cpg;
#pragma unroll
      for (int j = 0; j < 7; ++j)
        if (j < ktaps) atomicAdd(dw + ((int64_t)(c_lo + co) * cpg + i) * ktaps + j, acc[q][j]);
    }
  }
}

__global__ void pack_gconv_dgrad_kernel(const float* __restrict__ w, float* __restrict__ wt, int C, int cpg, int ktaps) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  int total = C * cpg * ktaps;
  if (idx >= total) return;
  int j = idx % ktaps, o = (idx / ktaps) % cpg, ci = idx / (ktaps * cpg);
  int g = ci / cpg, i = ci % cpg;
  wt[idx] = w[((int64_t)(g * cpg + o) * cpg + i) * ktaps + (ktaps - 1 - j)];  // group-transposed, taps flipped
}

size_t fwd_smem(int cpg, int ktaps) {
  int CS = slab_channels(cpg);
  return sizeof(float) * ((size_t)(G_TT + G_MAXHALO) * CS + (size_t)CS * wpitch(cpg, ktaps) + (size_t)G_TT * (CS + 1));
}
size_t wgrad_smem(int cpg) {
  int CS = slab_channels(cpg);
  return sizeof(float) * ((size_t)(G_TT + G_MAXHALO) * CS + (size_t)G_TT * CS);
}

}  // namespace

extern "C" {

int nbasr_gconv_fwd(const nbasr_gconv* p, void* stream) {
  NBASR_REQUIRE(p->C % p->cpg == 0 && p->C % 8 == 0, "channels");
  if (p->B <= 0 || p->T <= 0) return 0;
  if (p->w_packed & 1) {
    NBASR_REQUIRE(p->dtype != NBASR_F32, "packed grouped-conv weights need 16-bit activations");
    return sm100_gconv_fwd(p, as_stream(stream));
  }
  NBASR_REQUIRE(p->ktaps <= 7 && (p->dstep == 1 || p->dstep == 2), "taps");
  NBASR_REQUIRE(p->cpg == 6 || p->cpg == 8 || p->cpg == 10 || p->cpg == 12, "cpg (slab must stay 8-aligned)");
  int CS = slab_channels(p->cpg);
  dim3 grid((p->C + CS - 1) / CS, (p->T + G_TT - 1) / G_TT, p->B);
  size_t sm = fwd_smem(p->cpg, p->ktaps);
  if (p->dtype == NBASR_BF16) {
    static DevOnce attr;
    if (!attr) { cudaFuncSetAttribute(gconv_fwd_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); attr = true; }
    gconv_fwd_kernel<bf16><<<grid, G_NT, sm, as_stream(stream)>>>(*p);
  } else {
    static DevOnce attr;
    if (!attr) { cudaFuncSetAttribute(gconv_fwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); attr = true; }
    gconv_fwd_kernel<float><<<grid, G_NT, sm, as_stream(stream)>>>(*p);
  }
  NBASR_CHECK_LAUNCH();
  return 0;
}

int nbasr_gconv_chain(const nbasr_gconv* nodes, int n, int fused, void* work, int64_t work_bytes, void* stream) {
  NBASR_REQUIRE(nodes != nullptr && n >= 1 && n <= 3, "chain of 1..3 grouped-conv edges");
  if (nodes[0].B <= 0 || nodes[0].T <= 0) return 0;
  bool packed = true;
  for (int i = 0; i < n; ++i) packed = packed && (nodes[i].w_packed & 1) && nodes[i].dtype != NBASR_F32;
  if (packed) return sm100_gconv_chain(nodes, n, fused, work, work_bytes, as_stream(stream));
  for (int i = 0; i < n; ++i)       // fp32 / unpacked weights: the SIMT kernel, node by node
    if (nbasr_gconv_fwd(nodes + i, stream)) return 1;
  return 0;
}

int64_t nbasr_gconv_chain_work_bytes(int B, int T, int C, int cpg, int n) { return sm100_gconv_chain_work_bytes(B, T, C, cpg, n); }

int nbasr_pack_gconv_dgrad(const float* w, float* wt, int C, int cpg, int ktaps, void* stream) {
  int total = C * cpg * ktaps;
  pack_gconv_dgrad_kernel<<<(total + 255) / 256, 256, 0, as_stream(stream)>>>(w, wt, C, cpg, ktaps);
  NBASR_CHECK_LAUNCH();
  return 0;
}

int nbasr_gconv_wgrad_x(int dz_dtype, const void* dz, const void* x, int x_dtype, float x_scale, int B, int T, int Tp, int C,
                        int cpg, int ktaps, int off0, int dstep, float* dw, float* dbias, void* stream) {
  NBASR_REQUIRE(cpg == 6 || cpg == 8 || cpg == 10 || cpg == 12, "cpg");
  NBASR_REQUIRE(ktaps <= 7 && (dstep == 1 || dstep == 2), "taps");
  NBASR_REQUIRE(dz_dtype == NBASR_BF16 ? (x_dtype == NBASR_BF16 || x_dtype == NBASR_F16) : (dz_dtype == NBASR_F32 && x_dtype == NBASR_F32),
                "dtypes: bf16 dz with bf16 / fp16 x, or fp32 dz and x");
  if (B <= 0 || T <= 0) return 0;
  if (dz_dtype == NBASR_BF16 && !nbasr_env_flag(NBASR_ENV_FORCE_SIMT))
    return sm100_gconv_wgrad(dz, x, x_dtype == NBASR_F16, x_scale, B, T, Tp, C, cpg, ktaps, off0, dstep, dw, dbias, as_stream(stream));
  if (dbias && nbasr_colsum(dz_dtype, dz, B, T, Tp, C, dbias, stream)) return 1;
  int CS = slab_channels(cpg);
  dim3 grid((C + CS - 1) / CS, B);
  size_t sm = wgrad_smem(cpg);
  auto launch = [&](auto kern, auto dzp, auto xp) {
    static DevOnce attr;     // one latch per kernel instantiation (the lambda is instantiated per argument types)
    if (!attr) { cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); attr = true; }
    kern<<<grid, G_NT, sm, as_stream(stream)>>>(dzp, xp, x_scale, B, T, Tp, C, cpg, ktaps, off0, dstep, dw);
  };
  if (dz_dtype == NBASR_F32) launch(gconv_wgrad_kernel<float, float>, (const float*)dz, (const float*)x);
  else if (x_dtype == NBASR_F16) launch(gconv_wgrad_kernel<bf16, f16>, (const bf16*)dz, (const f16*)x);
  else launch(gconv_wgrad_kernel<bf16, bf16>, (const bf16*)dz, (const bf16*)x);
  NBASR_CHECK_LAUNCH();
  return 0;
}

int nbasr_gconv_wgrad(int dtype, const void* dz, const void* x, int B, int T, int Tp, int C, int cpg, int ktaps,
                      int off0, int dstep, float* dw, float* dbias, void* stream) {
  return nbasr_gconv_wgrad_x(dtype, dz, x, dtype, 1.f, B, T, Tp, C, cpg, ktaps, off0, dstep, dw, dbias, stream);
}

}  // extern "C"
