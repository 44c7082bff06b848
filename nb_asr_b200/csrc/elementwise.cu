// HBM-bound row kernels: LayerNorm fwd/bwd, element-wise epilogue pass, column sums, input
// transpose, weight packing.  One warp per frame row for the norm kernels (a row of C <= 1280
// channels lives in registers), 16-byte vector accesses everywhere.
#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int LN_MAXG = 5;  // groups of 8 channels per lane -> C <= 1280

template <typename T>
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, int B, int Tt,
                                                            int Tp, int C, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float eps,
                                                            float* __restrict__ mean_o, float* __restrict__ rstd_o) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int ngroups = C >> 3;
  const int64_t nrows = (int64_t)B * Tt;
  for (int64_t r = warp; r < nrows; r += nwarps) {
    int b = (int)(r / Tt), t = (int)(r % Tt);
    int64_t rho = (int64_t)b * Tp + NBASR_PAD_L + t;
    const T* xr = x + rho * C;
    float v[LN_MAXG][8];
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < LN_MAXG; ++q) {
      int g = lane + 32 * q;
      if (g < ngroups) {
        load8(xr + g * 8, v[q]);
#pragma unroll
        for (int i = 0; i < 8; ++i) s += v[q][i];
      }
    }
    float mean = warp_sum(s) / C;
    float ss = 0.f;
#pragma unroll
    for (int q = 0; q < LN_MAXG; ++q) {
      int g = lane + 32 * q;
      if (g < ngroups) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float d = v[q][i] - mean;
          ss += d * d;
        }
      }
    }
    float rstd = rsqrtf(warp_sum(ss) / C + eps);
    if (lane == 0 && mean_o) {
      mean_o[rho] = mean;
      rstd_o[rho] = rstd;
    }
    T* yr = y + rho * C;
#pragma unroll
    for (int q = 0; q < LN_MAXG; ++q) {
      int g = lane + 32 * q;
      if (g < ngroups) {
        float ga[8], be[8], o[8];
        load8(gamma + g * 8, ga);
        load8(beta + g * 8, be);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = (v[q][i] - mean) * rstd * ga[i] + be[i];
        store8(yr + g * 8, o);
      }
    }
  }
}

// Backward: per-warp rows, dgamma/dbeta partials live in warp-private shared memory (layout [i][group] so
// that the 32 lanes of a warp hit 32 different banks), which keeps registers low enough for 16 warps / SM.
template <typename T>
__global__ void __launch_bounds__(256, 2) layernorm_bwd_kernel(
    const T* __restrict__ dy, const T* __restrict__ x, const float* __restrict__ mean_i,
    const float* __restrict__ rstd_i, const float* __restrict__ gamma, int B, int Tt, int Tp, int C,
    T* __restrict__ dx, T* __restrict__ dx2, const uint32_t* __restrict__ mask2, float scale2, int64_t mask_rows, int mask2_w,
    float* __restrict__ dgamma, float* __restrict__ dbeta) {
  extern __shared__ float red[];  // 8 warps x 2 x (8 x GP) floats, GP = padded group count
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int ngroups = C >> 3;
  const int GP = 32 * LN_MAXG;
  const int64_t nrows = (int64_t)B * Tt;
  float* my_dg = red + (size_t)wib * 2 * 8 * GP;
  float* my_db = my_dg + 8 * GP;
  for (int i = lane; i < 2 * 8 * GP; i += 32) my_dg[i] = 0.f;
  __syncwarp();
  // plane-major gate-bit mask: per-lane byte offsets are row independent up to "+ rho * entry_bytes"
  int64_t moff[LN_MAXG];
  const int meb = (mask2_w == 32) ? 4 : 8;
#pragma unroll
  for (int q = 0; q < LN_MAXG; ++q) moff[q] = mask_byte_addr(0, (lane + 32 * q) * 8, mask2_w, mask_rows);
  for (int64_t r = warp; r < nrows; r += nwarps) {
    int b = (int)(r / Tt), t = (int)(r % Tt);
    int64_t rho = (int64_t)b * Tp + NBASR_PAD_L + t;
    float mean = mean_i[rho], rstd = rstd_i[rho];
    float xh[LN_MAXG][8], gy[LN_MAXG][8];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int q = 0; q < LN_MAXG; ++q) {
      int g = lane + 32 * q;
      if (g < ngroups) {
        float xv[8], dv[8], ga[8];
        load8(x + rho * C + g * 8, xv);
        load8(dy + rho * C + g * 8, dv);
        load8(gamma + g * 8, ga);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          xh[q][i] = (xv[i] - mean) * rstd;
          my_dg[i * GP + g] += dv[i] * xh[q][i];
          my_db[i * GP + g] += dv[i];
          gy[q][i] = dv[i] * ga[i];
          s1 += gy[q][i];
          s2 += gy[q][i] * xh[q][i];
        }
      }
    }
    s1 = warp_sum(s1) / C;
    s2 = warp_sum(s2) / C;
#pragma unroll
    for (int q = 0; q < LN_MAXG; ++q) {
      int g = lane + 32 * q;
      if (g < ngroups) {
        float o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = rstd * (gy[q][i] - s1 - xh[q][i] * s2);
        if (dx) store8(dx + rho * C + g * 8, o);
        if (dx2) {
          uint32_t w = mask2 ? reinterpret_cast<const uint8_t*>(mask2)[moff[q] + rho * meb] : 0xffu;
          float o2[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) o2[i] = ((w >> i) & 1u) ? o[i] * scale2 : 0.f;
          store8(dx2 + rho * C + g * 8, o2);
        }
      }
    }
  }
  __syncthreads();
  // block reduction over the 8 warps, then one atomic per channel per block
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    int g = c >> 3, i = c & 7;
    float a = 0.f, bsum = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      a += red[(size_t)w * 2 * 8 * GP + i * GP + g];
      bsum += red[(size_t)w * 2 * 8 * GP + 8 * GP + i * GP + g];
    }
    atomicAdd(dgamma + c, a);
    atomicAdd(dbeta + c, bsum);
  }
}


__global__ void eltwise_kernel(int src_dtype, const void* __restrict__ src, int64_t ld_src, int B, int Tt, int Tp, int C,
                               nbasr_epilogue e) {
  const int nch = (C + 31) >> 5;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)B * Tt * nch;
  if (idx >= total) return;
  int ch = (int)(idx % nch);
  int64_t r = idx / nch;
  int b = (int)(r / Tt), t = (int)(r % Tt);
  int64_t rho = (int64_t)b * Tp + NBASR_PAD_L + t;
  int c0 = ch * 32;
  float v[32];
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    int nrem = C - c0 - g * 8;
    if (src && nrem > 0) load8_dt_n(src, src_dtype, rho * ld_src + c0 + g * 8, v + g * 8, nrem);
    else {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[g * 8 + i] = 0.f;
    }
  }
  epilogue_chunk(e, rho, c0, C, v);
}

constexpr int CS_MAXG = 8;  // C <= 2048

// column sums: warp per row (16-byte vector loads, fully coalesced), register partials, block reduce, atomics
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ x, int B, int Tt, int Tp, int C, float* __restrict__ out) {
  extern __shared__ float red[];  // C floats
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int ngroups = C >> 3;
  const int64_t nrows = (int64_t)B * Tt;
  for (int i = threadIdx.x; i < C; i += blockDim.x) red[i] = 0.f;
  __syncthreads();
  float acc[CS_MAXG][8];
#pragma unroll
  for (int q = 0; q < CS_MAXG; ++q)
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[q][i] = 0.f;
  for (int64_t r = warp; r < nrows; r += nwarps) {
    int b = (int)(r / Tt), t = (int)(r % Tt);
    const T* xr = x + ((int64_t)b * Tp + NBASR_PAD_L + t) * C;
#pragma unroll
    for (int q = 0; q < CS_MAXG; ++q) {
      int g = lane + 32 * q;
      if (g < ngroups) {
        float v[8];
        load8(xr + g * 8, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[q][i] += v[i];
      }
    }
  }
#pragma unroll
  for (int q = 0; q < CS_MAXG; ++q) {
    int g = lane + 32 * q;
    if (g < ngroups) {
#pragma unroll
      for (int i = 0; i < 8; ++i) atomicAdd(&red[g * 8 + i], acc[q][i]);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(out + i, red[i]);
}

template <typename T>
__global__ void transpose_in_kernel(const float* __restrict__ a, T* __restrict__ out, int B, int F, int Tt, int Tp, float scale) {
  __shared__ float tile[32][33];
  int b = blockIdx.z;
  int t0 = blockIdx.x * 32, f0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int f = f0 + i, t = t0 + threadIdx.x;
    tile[i][threadIdx.x] = (f < F && t < Tt) ? a[((int64_t)b * F + f) * Tt + t] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int t = t0 + i, f = f0 + threadIdx.x;
    if (t < Tt && f < F) out[((int64_t)b * Tp + NBASR_PAD_L + t) * F + f] = static_cast<T>(tile[threadIdx.x][i] * scale);
  }
}

// the inverse layout change: padded channels-last fp32 (B, Tp, F) -> (B, F, T) fp32
__global__ void transpose_out_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int F, int Tt, int Tp) {
  __shared__ float tile[32][33];
  int b = blockIdx.z;
  int t0 = blockIdx.x * 32, f0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int t = t0 + i, f = f0 + threadIdx.x;
    tile[i][threadIdx.x] = (t < Tt && f < F) ? in[((int64_t)b * Tp + NBASR_PAD_L + t) * F + f] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int f = f0 + i, t = t0 + threadIdx.x;
    if (f < F && t < Tt) out[((int64_t)b * F + f) * Tt + t] = tile[threadIdx.x][i];
  }
}

template <typename T>
__global__ void pack_weight_kernel(const float* __restrict__ w, T* __restrict__ out, int M, int N, int nq, int t0,
                                   int tstep, int64_t ws_m, int64_t ws_n, int64_t ws_t) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)N * nq * M;
  if (idx >= total) return;
  int m = (int)(idx % M);
  int q = (int)((idx / M) % nq);
  int n = (int)(idx / ((int64_t)M * nq));
  out[idx] = static_cast<T>(w[m * ws_m + n * ws_n + (int64_t)(t0 + q * tstep) * ws_t]);
}

template <typename T>
__global__ void convert_kernel(const float* __restrict__ s, T* __restrict__ d, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) d[i] = static_cast<T>(s[i]);
}

__global__ void fill_u32_kernel(uint32_t* p, uint32_t v, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

}  // namespace

extern "C" {

int nbasr_layernorm_fwd(int dtype, const void* x, void* y, int B, int T, int Tp, int C, const float* gamma,
                        const float* beta, float eps, float* mean, float* rstd, float out_scale, void* y2, void* stream) {
  NBASR_REQUIRE(C % 8 == 0 && C <= 8 * 32 * LN_MAXG, "C");
  int64_t rows = (int64_t)B * T;
  int blocks = (int)std::min<int64_t>((rows + 7) / 8, 148 * 8);
  if (blocks < 1) return 0;
  if (out_scale == 0.f) out_scale = 1.f;
  const bool small = rows * (int64_t)C < (int64_t)1 << 40 && (int64_t)B * Tp < (int64_t)1 << 30;
  if (dtype != NBASR_F32 && small)      // packed-fp32x2 kernels (layernorm2.cu)
    return ln2_fwd(x, y, dtype == NBASR_F16, B, T, Tp, C, gamma, beta, eps, mean, rstd, out_scale, y2, as_stream(stream));
  NBASR_REQUIRE(dtype != NBASR_F16 && out_scale == 1.f && !y2, "generic LayerNorm kernel: fp32 / bf16, unscaled, single output");
  if (dtype == NBASR_BF16)
    layernorm_fwd_kernel<bf16><<<blocks, 256, 0, as_stream(stream)>>>((const bf16*)x, (bf16*)y, B, T, Tp, C, gamma, beta, eps, mean, rstd);
  else
    layernorm_fwd_kernel<float><<<blocks, 256, 0, as_stream(stream)>>>((const float*)x, (float*)y, B, T, Tp, C, gamma, beta, eps, mean, rstd);
  NBASR_CHECK_LAUNCH();
  return 0;
}

int nbasr_layernorm_bwd(int dtype, const void* dy, const void* x, int x_dtype, float x_scale, const float* mean, const float* rstd,
                        const float* gamma, int B, int T, int Tp, int C, void* dx, void* dx2, const uint32_t* mask2,
                        float scale2, int64_t mask_rows, int mask2_w, float* dgamma, float* dbeta, void* stream) {
  NBASR_REQUIRE(C % 8 == 0 && C <= 8 * 32 * LN_MAXG, "C");
  int64_t rows = (int64_t)B * T;
  int blocks = (int)std::min<int64_t>((rows + 7) / 8, 148 * 2);
  if (blocks < 1) return 0;
  if (x_scale == 0.f) x_scale = 1.f;
  size_t sm = (size_t)8 * 2 * 8 * 32 * LN_MAXG * sizeof(float);   // 80 KB
  static DevOnce attr;
  if (!attr) {
    cudaFuncSetAttribute(layernorm_bwd_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    cudaFuncSetAttribute(layernorm_bwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    attr = true;
  }
  const bool small = (int64_t)B * Tp < (int64_t)1 << 30 && mask_rows * 8 * ((C + 31) / 32 + 1) < (int64_t)1 << 31;
  if (dtype == NBASR_BF16 && x_dtype != NBASR_F32 && small)
    return ln2_bwd(dy, x, x_dtype == NBASR_F16, x_scale, mean, rstd, gamma, B, T, Tp, C, dx, dx2, mask2, scale2, mask_rows, mask2_w, dgamma,
                   dbeta, as_stream(stream));
  NBASR_REQUIRE(x_dtype == dtype && x_scale == 1.f && dtype != NBASR_F16, "generic LayerNorm backward: one unscaled dtype (fp32 / bf16)");
  if (dtype == NBASR_BF16)
    layernorm_bwd_kernel<bf16><<<blocks, 256, sm, as_stream(stream)>>>((const bf16*)dy, (const bf16*)x, mean, rstd, gamma, B, T, Tp, C, (bf16*)dx, (bf16*)dx2, mask2, scale2, mask_rows, mask2_w, dgamma, dbeta);
  else
    layernorm_bwd_kernel<float><<<blocks, 256, sm, as_stream(stream)>>>((const float*)dy, (const float*)x, mean, rstd, gamma, B, T, Tp, C, (float*)dx, (float*)dx2, mask2, scale2, mask_rows, mask2_w, dgamma, dbeta);
  NBASR_CHECK_LAUNCH();
  return 0;
}

int nbasr_eltwise(int src_dtype, const void* src, int64_t ld_src, int B, int T, int Tp, int C,
                  const nbasr_epilogue* epi, void* stream) {
  int64_t total = (int64_t)B * T * ((C + 31) / 32);
  if (total == 0) return 0;
  eltwise_kernel<<<(unsigned)((total + 127) / 128), 128, 0, as_stream(stream)>>>(src_dtype, src, ld_src, B, T, Tp, C, *epi);
  NBASR_CHECK_LAUNCH();
  return 0;
}

int nbasr_colsum(int dtype, const void* x, int B, int T, int Tp, int C, float* out, void* stream) {
  NBASR_REQUIRE(C % 8 == 0 && C <= 8 * 32 * CS_MAXG, "C");
  int64_t rows = (int64_t)B * T;
  if (rows < 1) return 0;
  int grid = (int)std::min<int64_t>((rows + 7) / 8, 148 * 4);
  size_t sm = C * sizeof(float);
  if (dtype == NBASR_BF16) colsum_kernel<bf16><<<grid, 256, sm, as_stream(stream)>>>((const bf16*)x, B, T, Tp, C, out);
  else colsum_kernel<float><<<grid, 256, sm, as_stream(stream)>>>((const float*)x, B, T, Tp, C, out);
  NBASR_CHECK_LAUNCH();
  return 0;
}

int nbasr_transpose_in(const float* audio, void* out, int dtype, int B, int F, int T, int Tp, float scale, void* stream) {
  dim3 grid((T + 31) / 32, (F + 31) / 32, B), block(32, 8);
  if (scale == 0.f) scale = 1.f;
  if (dtype == NBASR_BF16) transpose_in_kernel<bf16><<<grid, block, 0, as_stream(stream)>>>(audio, (bf16*)out, B, F, T, Tp, scale);
  else if (dtype == NBASR_F16) transpose_in_kernel<f16><<<grid, block, 0, as_stream(stream)>>>(audio, (f16*)out, B, F, T, Tp, scale);
  else transpose_in_kernel<float><<<grid, block, 0, as_stream(stream)>>>(audio, (float*)out, B, F, T, Tp, scale);
  NBASR_CHECK_LAUNCH();
  return 0;
}

int nbasr_transpose_out(const float* in, float* out, int B, int F, int T, int Tp, void* stream) {
  if (B <= 0 || F <= 0 || T <= 0) return 0;
  dim3 grid((T + 31) / 32, (F + 31) / 32, B), block(32, 8);
  transpose_out_kernel<<<grid, block, 0, as_stream(stream)>>>(in, out, B, F, T, Tp);
  NBASR_CHECK_LAUNCH();
  return 0;
}

int nbasr_pack_weight(const float* w, void* out, int out_dtype, int M, int N, int nq, int t0, int tstep, int64_t ws_m,
                      int64_t ws_n, int64_t ws_t, void* stream) {
  int64_t total = (int64_t)N * nq * M;
  unsigned blocks = (unsigned)((total + 255) / 256);
  if (out_dtype == NBASR_BF16)
    pack_weight_kernel<bf16><<<blocks, 256, 0, as_stream(stream)>>>(w, (bf16*)out, M, N, nq, t0, tstep, ws_m, ws_n, ws_t);
  else if (out_dtype == NBASR_F16)
    pack_weight_kernel<f16><<<blocks, 256, 0, as_stream(stream)>>>(w, (f16*)out, M, N, nq, t0, tstep, ws_m, ws_n, ws_t);
  else
    pack_weight_kernel<float><<<blocks, 256, 0, as_stream(stream)>>>(w, (float*)out, M, N, nq, t0, tstep, ws_m, ws_n, ws_t);
  NBASR_CHECK_LAUNCH();
  return 0;
}

int nbasr_convert(const float* src, void* dst, int dst_dtype, int64_t n, void* stream) {
  unsigned blocks = (unsigned)((n + 255) / 256);
  if (dst_dtype == NBASR_BF16) convert_kernel<bf16><<<blocks, 256, 0, as_stream(stream)>>>(src, (bf16*)dst, n);
  else if (dst_dtype == NBASR_F16) convert_kernel<f16><<<blocks, 256, 0, as_stream(stream)>>>(src, (f16*)dst, n);
  else convert_kernel<float><<<blocks, 256, 0, as_stream(stream)>>>(src, (float*)dst, n);
  NBASR_CHECK_LAUNCH();
  return 0;
}

int nbasr_fill_u32(uint32_t* p, uint32_t val, int64_t n, void* stream) {
  fill_u32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, as_stream(stream)>>>(p, val, n);
  NBASR_CHECK_LAUNCH();
  return 0;
}

}  // extern "C"
