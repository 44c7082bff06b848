// Optimiser tail of Trainer.step (trainer.py:221-225) over flat fp32 buffers:
//   grad += 0.01 * W / ||W||_F for every PadConvRelu weight (gradient of the norm regulariser),
//   coef = min(1, max_norm / (||grad||_2 + 1e-6))   (torch.nn.utils.clip_grad_norm_),
//   Adam(betas, eps) with bias correction (torch.optim.Adam, amsgrad=False, weight_decay=0).
// Step count, lr and every reduction result live in a small device `state` array, so the whole
// step replays inside a CUDA graph.  Every reduction is DETERMINISTIC (per-block partials summed in a fixed order, no
// float atomics): data-parallel replicas that receive the same all-reduced gradient must compute bit-identical clip
// coefficients and updates, or they drift apart.
#include "common.cuh"
#include "kernels.h"

namespace {

__device__ __forceinline__ float block_sum(float v) {
  __shared__ float red[32];
  v = warp_sum(v);
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  v = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
  if (w == 0) v = warp_sum(v);
  return v;
}

__device__ __forceinline__ double block_sum(double v) {
  __shared__ double redd[32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) redd[w] = v;
  __syncthreads();
  v = (threadIdx.x < (blockDim.x >> 5)) ? redd[threadIdx.x] : 0.0;
  if (w == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  }
  return v;
}

// Regularised segments are cut into chunks of SEG_CHUNK elements; block b finds its (segment, chunk) by walking
// the (<= 64) segment lengths -- big tensors get proportionally many blocks.
constexpr int SEG_CHUNK = 16384;

__device__ __forceinline__ bool seg_locate(const int64_t* __restrict__ len, int nseg, int64_t blk, int& s, int64_t& start) {
  for (s = 0; s < nseg; ++s) {
    int64_t nch = (len[s] + SEG_CHUNK - 1) / SEG_CHUNK;
    if (blk < nch) { start = blk * SEG_CHUNK; return true; }
    blk -= nch;
  }
  return false;
}

// (the segment bases are 16-byte aligned in the engine's flat buffer; the scalar loops handle any other caller and the tails)
__device__ __forceinline__ bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

constexpr int SUMSQ_BLOCKS = 592;

__global__ void seg_sumsq_kernel(const float* __restrict__ p, const int64_t* __restrict__ off, const int64_t* __restrict__ len,
                                 int nseg, float* __restrict__ part) {
  int s; int64_t start;
  if (!seg_locate(len, nseg, blockIdx.x, s, start)) return;
  const float* x = p + off[s] + start;
  const int n = (int)(min(len[s], start + SEG_CHUNK) - start);
  float acc = 0.f;
  int i0 = 0;
  if (al16(x)) {
    const int n4 = n >> 2;
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
      const float4 v = reinterpret_cast<const float4*>(x)[i];
      acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
    i0 = n4 << 2;
  }
  for (int i = i0 + threadIdx.x; i < n; i += blockDim.x) acc += x[i] * x[i];
  acc = block_sum(acc);
  if (threadIdx.x == 0) part[blockIdx.x] = acc;
}

// block (s, k): out[s * out_stride + k] = sum of the chunk partials part[k * part_stride + chunk] of segment s, in chunk order
// (the optimiser: one partial per chunk, out = state + 4; nbasr_param_stats: two)
template <typename T>
__global__ void seg_reduce_kernel(const T* __restrict__ part, const int64_t* __restrict__ len, int nseg, T* __restrict__ out,
                                  int64_t part_stride, int out_stride) {
  const int s = blockIdx.x;
  part += blockIdx.y * part_stride;
  int64_t first = 0;
  for (int i = 0; i < s; ++i) first += (len[i] + SEG_CHUNK - 1) / SEG_CHUNK;
  const int nch = (int)((len[s] + SEG_CHUNK - 1) / SEG_CHUNK);
  T acc = 0;
  for (int i = threadIdx.x; i < nch; i += blockDim.x) acc += part[first + i];
  acc = block_sum(acc);
  if (threadIdx.x == 0) out[(int64_t)s * out_stride + blockIdx.y] = acc;
}

// Per-tensor statistics of the zero-cost proxies (nbasr_param_stats): for one chunk of a segment, the fp64 partials
// sum g^2 -> part[blk] and sum |p g| -> part[nchunks + blk].  At initialisation gradients can be ~1e-20: their squares
// are below fp32's normal range, so products are formed and summed in fp64.
__global__ void seg_stats_kernel(const float* __restrict__ p, const float* __restrict__ g, const int64_t* __restrict__ off,
                                 const int64_t* __restrict__ len, int nseg, int64_t nchunks, double* __restrict__ part) {
  int s; int64_t start;
  if (!seg_locate(len, nseg, blockIdx.x, s, start)) return;
  const float* x = p + off[s] + start;
  const float* gg = g + off[s] + start;
  const int n = (int)(min(len[s], start + SEG_CHUNK) - start);
  double sq = 0.0, ab = 0.0;
  int i0 = 0;
  if (al16(x) && al16(gg)) {
    const int n4 = n >> 2;
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
      const float4 v = reinterpret_cast<const float4*>(x)[i];
      const float4 w = reinterpret_cast<const float4*>(gg)[i];
      sq += (double)w.x * w.x + (double)w.y * w.y + (double)w.z * w.z + (double)w.w * w.w;
      ab += fabs((double)v.x * w.x) + fabs((double)v.y * w.y) + fabs((double)v.z * w.z) + fabs((double)v.w * w.w);
    }
    i0 = n4 << 2;
  }
  for (int i = i0 + threadIdx.x; i < n; i += blockDim.x) {
    const double w = gg[i];
    sq += w * w;
    ab += fabs((double)x[i] * w);
  }
  sq = block_sum(sq);
  ab = block_sum(ab);
  if (threadIdx.x == 0) {
    part[blockIdx.x] = sq;
    part[nchunks + blockIdx.x] = ab;
  }
}

// Gradient signal-to-noise of the ZiCo proxy (nbasr_grad_snr): parameter i of a segment has the N fp32 samples
// g[k * g_stride + i]; with m = S / N and var = sum_k (g_k - m)^2 / N (population), r = (A / N) / sqrt(var) when var > 0.
// In fp64 the kernel forms S = sum_k g_k, A = sum_k |g_k| and Q = sum_k (N g_k - S)^2 = N^3 var, and r = sqrt(N) A / sqrt(Q)
// (one reciprocal square root per parameter instead of three divisions and a square root).  For one chunk: sum r ->
// part[blk], number of parameters with Q > 0 -> part[nchunks + blk].  N g_k is exact (24 + 4 significant bits); N equal
// samples sum exactly to N g, so Q = 0; samples that are not all equal leave some N g_k - S != 0, whose square is far
// above fp64's underflow.  So Q > 0 exactly when the samples are not all equal -- the same set as var > 0 in a numpy
// restatement on the same samples.
constexpr int SNR_MAX_N = 16;

// NMAX >= N samples per parameter, VEC = 16 / NMAX parameters per thread and step (elements i, i + 256, ... of the
// chunk): the 16 loads of a step are issued together, so a small N still keeps enough bytes in flight.
template <int NMAX>
__global__ void __launch_bounds__(256) seg_snr_kernel(const float* __restrict__ g, int64_t g_stride, int N,
                                                      const int64_t* __restrict__ off, const int64_t* __restrict__ len,
                                                      int nseg, int64_t nchunks, double* __restrict__ part) {
  constexpr int VEC = SNR_MAX_N / NMAX;
  int s; int64_t start;
  if (!seg_locate(len, nseg, blockIdx.x, s, start)) return;
  const float* x = g + off[s] + start;
  const int n = (int)(min(len[s], start + SEG_CHUNK) - start);
  const double dn = N, sqrt_n = sqrt(dn);
  double rsum = 0.0, cnt = 0.0;
  for (int i0 = threadIdx.x; i0 < n; i0 += VEC * blockDim.x) {
    float v[VEC][NMAX];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const int i = i0 + j * blockDim.x;
#pragma unroll
      for (int k = 0; k < NMAX; ++k) v[j][k] = (k < N && i < n) ? x[k * g_stride + i] : 0.f;
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      if (i0 + j * (int)blockDim.x >= n) break;
      double S = 0.0, A = 0.0;
#pragma unroll
      for (int k = 0; k < NMAX; ++k) {
        if (k < N) {
          S += v[j][k];
          A += fabs((double)v[j][k]);
        }
      }
      double Q = 0.0;
#pragma unroll
      for (int k = 0; k < NMAX; ++k) {
        if (k < N) {
          const double d = fma(dn, (double)v[j][k], -S);
          Q = fma(d, d, Q);
        }
      }
      if (Q > 0.0) {
        rsum = fma(sqrt_n * A, rsqrt(Q), rsum);
        cnt += 1.0;
      }
    }
  }
  rsum = block_sum(rsum);
  cnt = block_sum(cnt);
  if (threadIdx.x == 0) {
    part[blockIdx.x] = rsum;
    part[nchunks + blockIdx.x] = cnt;
  }
}

// Row Gram matrix of nbasr_row_gram: block c covers columns [c * GRAM_CHUNK, (c + 1) * GRAM_CHUNK) of every row and writes
// the fp64 partials of the upper triangle G[i][j] (i <= j, row-major triangle order) and of the row sums.
constexpr int GRAM_CHUNK = 256;
constexpr int GRAM_MAX_B = 128;

__global__ void row_gram_part_kernel(const float* __restrict__ x, int B, int64_t D, int64_t ld, double* __restrict__ part) {
  extern __shared__ float xs[];                     // [B][GRAM_CHUNK + 1] (padded: no bank conflicts along a row)
  const int64_t c0 = (int64_t)blockIdx.x * GRAM_CHUNK;
  const int w = (int)min((int64_t)GRAM_CHUNK, D - c0);
  for (int i = threadIdx.x; i < B * GRAM_CHUNK; i += blockDim.x) {
    const int r = i / GRAM_CHUNK, c = i % GRAM_CHUNK;
    xs[r * (GRAM_CHUNK + 1) + c] = c < w ? x[(int64_t)r * ld + c0 + c] : 0.f;
  }
  __syncthreads();
  const int npair = B * (B + 1) / 2;
  double* out = part + (int64_t)blockIdx.x * (npair + B);
  for (int q = threadIdx.x; q < npair + B; q += blockDim.x) {
    int i, j;
    if (q < npair) {                                 // q -> (i, j), i <= j, row i of the triangle holds B - i entries
      i = 0;
      int r = q;
      while (r >= B - i) { r -= B - i; ++i; }
      j = i + r;
    } else {
      i = q - npair;
      j = -1;
    }
    const float* a = xs + i * (GRAM_CHUNK + 1);
    double acc = 0.0;
    if (j >= 0) {
      const float* bb = xs + j * (GRAM_CHUNK + 1);
      for (int c = 0; c < w; ++c) acc += (double)a[c] * bb[c];
    } else {
      for (int c = 0; c < w; ++c) acc += a[c];
    }
    out[q] = acc;
  }
}

// thread q: the sum of the chunk partials of entry q in chunk order; the triangle is mirrored into the full B x B matrix
__global__ void row_gram_reduce_kernel(const double* __restrict__ part, int B, int nchunks, double* __restrict__ gram,
                                       double* __restrict__ rowsum) {
  const int npair = B * (B + 1) / 2;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= npair + B) return;
  double acc = 0.0;
  for (int c = 0; c < nchunks; ++c) acc += part[(int64_t)c * (npair + B) + q];
  if (q >= npair) {
    rowsum[q - npair] = acc;
    return;
  }
  int i = 0, r = q;
  while (r >= B - i) { r -= B - i; ++i; }
  const int j = i + r;
  gram[i * B + j] = acc;
  gram[j * B + i] = acc;
}

// state[2] = sum of n per-block partials, fixed order
__global__ void total_reduce_kernel(const float* __restrict__ part, int n, float* __restrict__ state) {
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += part[i];
  acc = block_sum(acc);
  if (threadIdx.x == 0) state[2] = acc;
}

// g += k W for one chunk of a regularised segment
__global__ void reg_grad_kernel(const float* __restrict__ p, float* __restrict__ g, const int64_t* __restrict__ off,
                                const int64_t* __restrict__ len, int nseg, const float* __restrict__ state, float reg_coef) {
  int s; int64_t start;
  if (!seg_locate(len, nseg, blockIdx.x, s, start)) return;
  const float nrm = sqrtf(state[4 + s]);
  const float k = nrm > 0.f ? reg_coef / nrm : 0.f;
  const float* x = p + off[s] + start;
  float* gg = g + off[s] + start;
  const int n = (int)(min(len[s], start + SEG_CHUNK) - start);
  int i0 = 0;
  if (al16(x) && al16(gg)) {
    const int n4 = n >> 2;
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
      const float4 v = reinterpret_cast<const float4*>(x)[i];
      float4 w = reinterpret_cast<float4*>(gg)[i];
      w.x += k * v.x; w.y += k * v.y; w.z += k * v.z; w.w += k * v.w;
      reinterpret_cast<float4*>(gg)[i] = w;
    }
    i0 = n4 << 2;
  }
  for (int i = i0 + threadIdx.x; i < n; i += blockDim.x) gg[i] += k * x[i];
}

__global__ void sumsq_kernel(const float* __restrict__ g, int64_t n, float* __restrict__ out) {
  float acc = 0.f;
  int64_t i0 = 0;
  if (al16(g)) {
    const int64_t n4 = n >> 2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
      const float4 v = reinterpret_cast<const float4*>(g)[i];
      acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
    i0 = n4 << 2;
  }
  for (int64_t i = i0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) acc += g[i] * g[i];
  acc = block_sum(acc);
  if (threadIdx.x == 0) out[blockIdx.x] = acc;
}

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            int64_t n, float max_norm, float b1, float b2, float eps, float* __restrict__ state) {
  const float step = state[0] + 1.f;
  const float lr = state[1];
  const float total = sqrtf(state[2]);
  const float coef = fminf(1.f, max_norm / (total + 1e-6f));
  const float bc1 = 1.f - powf(b1, step);
  const float bc2s = sqrtf(1.f - powf(b2, step));
  const float step_size = lr / bc1;
  const int64_t n4 = n >> 2;   // flat buffers are padded to multiples of 64 elements
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 g4 = reinterpret_cast<const float4*>(g)[i];
    float4 m4 = reinterpret_cast<float4*>(m)[i], v4 = reinterpret_cast<float4*>(v)[i], p4 = reinterpret_cast<float4*>(p)[i];
    float* gp = &g4.x; float* mp = &m4.x; float* vp = &v4.x; float* pp = &p4.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float gi = gp[j] * coef;
      mp[j] = b1 * mp[j] + (1.f - b1) * gi;
      vp[j] = b2 * vp[j] + (1.f - b2) * gi * gi;
      pp[j] -= step_size * mp[j] / (sqrtf(vp[j]) / bc2s + eps);
    }
    reinterpret_cast<float4*>(m)[i] = m4;
    reinterpret_cast<float4*>(v)[i] = v4;
    reinterpret_cast<float4*>(p)[i] = p4;
  }
  for (int64_t i = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float gi = g[i] * coef;
    float mi = b1 * m[i] + (1.f - b1) * gi;
    float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] -= step_size * mi / (sqrtf(vi) / bc2s + eps);
  }
}

__global__ void optim_finish_kernel(float* state, int nseg, float max_norm) {
  if (threadIdx.x == 0) {
    state[3] = fminf(1.f, max_norm / (sqrtf(state[2]) + 1e-6f));
    state[0] += 1.f;
  }
}

}  // namespace

extern "C" int nbasr_optim_step(float* param, float* grad, float* m, float* v, int64_t n, const int64_t* seg_off,
                                const int64_t* seg_len, int nseg, int64_t seg_chunks, float reg_coef, float max_norm, float beta1,
                                float beta2, float eps, float* state, void* stream) {
  cudaStream_t st = as_stream(stream);
  float* part_total = state + 8 + nseg;              // SUMSQ_BLOCKS partials of ||grad||^2
  float* part_seg = part_total + SUMSQ_BLOCKS;       // seg_chunks partials of the per-segment ||W||^2
  if (nseg > 0 && reg_coef != 0.f) {
    // seg_chunks = sum_s ceil(seg_len[s] / 16384), computed once by the host that owns the segment table
    seg_sumsq_kernel<<<(unsigned)seg_chunks, 256, 0, st>>>(param, seg_off, seg_len, nseg, part_seg);
    NBASR_CHECK_LAUNCH();
    seg_reduce_kernel<float><<<nseg, 256, 0, st>>>(part_seg, seg_len, nseg, state + 4, 0, 1);
    NBASR_CHECK_LAUNCH();
    reg_grad_kernel<<<(unsigned)seg_chunks, 256, 0, st>>>(param, grad, seg_off, seg_len, nseg, state, reg_coef);
    NBASR_CHECK_LAUNCH();
  }
  sumsq_kernel<<<SUMSQ_BLOCKS, 256, 0, st>>>(grad, n, part_total);
  NBASR_CHECK_LAUNCH();
  total_reduce_kernel<<<1, 256, 0, st>>>(part_total, SUMSQ_BLOCKS, state);
  NBASR_CHECK_LAUNCH();
  adam_kernel<<<1184, 256, 0, st>>>(param, grad, m, v, n, max_norm, beta1, beta2, eps, state);
  NBASR_CHECK_LAUNCH();
  optim_finish_kernel<<<1, 32, 0, st>>>(state, nseg, max_norm);
  NBASR_CHECK_LAUNCH();
  return 0;
}

extern "C" int nbasr_param_stats(const float* param, const float* grad, const int64_t* seg_off, const int64_t* seg_len, int nseg,
                                 int64_t seg_chunks, double* part, double* out, void* stream) {
  if (nseg <= 0) return 0;
  NBASR_REQUIRE(seg_chunks > 0, "seg_chunks = sum of ceil(seg_len / 16384)");
  cudaStream_t st = as_stream(stream);
  seg_stats_kernel<<<(unsigned)seg_chunks, 256, 0, st>>>(param, grad, seg_off, seg_len, nseg, seg_chunks, part);
  NBASR_CHECK_LAUNCH();
  seg_reduce_kernel<double><<<dim3(nseg, 2), 256, 0, st>>>(part, seg_len, nseg, out, seg_chunks, 2);
  NBASR_CHECK_LAUNCH();
  return 0;
}

extern "C" int nbasr_grad_snr(const float* g, int64_t g_stride, int N, const int64_t* seg_off, const int64_t* seg_len,
                              int nseg, int64_t seg_chunks, double* part, double* out, void* stream) {
  NBASR_REQUIRE(N >= 2 && N <= SNR_MAX_N, "2 <= N <= 16 gradient samples");
  if (nseg <= 0) return 0;
  NBASR_REQUIRE(seg_chunks > 0, "seg_chunks = sum of ceil(seg_len / 16384)");
  NBASR_REQUIRE(g_stride >= 0, "snapshot stride");
  cudaStream_t st = as_stream(stream);
  const unsigned grid = (unsigned)seg_chunks;
  if (N == 2)
    seg_snr_kernel<2><<<grid, 256, 0, st>>>(g, g_stride, N, seg_off, seg_len, nseg, seg_chunks, part);
  else if (N <= 4)
    seg_snr_kernel<4><<<grid, 256, 0, st>>>(g, g_stride, N, seg_off, seg_len, nseg, seg_chunks, part);
  else if (N <= 8)
    seg_snr_kernel<8><<<grid, 256, 0, st>>>(g, g_stride, N, seg_off, seg_len, nseg, seg_chunks, part);
  else
    seg_snr_kernel<16><<<grid, 256, 0, st>>>(g, g_stride, N, seg_off, seg_len, nseg, seg_chunks, part);
  NBASR_CHECK_LAUNCH();
  seg_reduce_kernel<double><<<dim3(nseg, 2), 256, 0, st>>>(part, seg_len, nseg, out, seg_chunks, 2);
  NBASR_CHECK_LAUNCH();
  return 0;
}

extern "C" int nbasr_row_gram(const float* x, int B, int64_t D, int64_t ld, double* gram, double* rowsum, double* work,
                              void* stream) {
  if (B <= 0) return 0;
  NBASR_REQUIRE(B <= GRAM_MAX_B, "at most 128 rows");
  NBASR_REQUIRE(D > 0 && ld >= D, "row length / pitch");
  cudaStream_t st = as_stream(stream);
  const int nchunks = (int)((D + GRAM_CHUNK - 1) / GRAM_CHUNK);
  const size_t smem = (size_t)B * (GRAM_CHUNK + 1) * sizeof(float);
  static DevOnce attr;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(row_gram_part_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         GRAM_MAX_B * (GRAM_CHUNK + 1) * (int)sizeof(float));
    if (e != cudaSuccess) return nbasr_fail("row_gram smem attr: %s", cudaGetErrorString(e));
    attr = true;
  }
  row_gram_part_kernel<<<nchunks, 256, smem, st>>>(x, B, D, ld, work);
  NBASR_CHECK_LAUNCH();
  const int nout = B * (B + 1) / 2 + B;
  row_gram_reduce_kernel<<<(nout + 255) / 256, 256, 0, st>>>(work, B, nchunks, gram, rowsum);
  NBASR_CHECK_LAUNCH();
  return 0;
}
