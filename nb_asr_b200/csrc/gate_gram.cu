// NASWOT kernel matrix of the zero-cost proxy `nwot` (nbasr_gate_gram, include/nbasr.h), straight from the plane-major
// ReLU20 gate bits a grad plan's forward pass leaves in HBM:
//   K[i][j] = sum over layers, planes, frames t < min(L_i, L_j), live columns c of [m_i(t, c) == m_j(t, c)].
// One work item is (layer, plane, chunk of GG_TCH frames).  A persistent grid of GG_BLOCKS blocks walks the items
// round-robin: the block stages the item's entries of all B utterances in shared memory (frame-major, each utterance's
// entries are consecutive rows, so the loads are coalesced) with the columns >= C / bits >= w masked off, then every
// thread adds, for each of its pairs (i <= j), the number of equal live bits over the frames valid for both.  Each block
// writes one uint64 partial per pair; a second kernel sums the GG_BLOCKS partials.  Integer sums: the result is exact and
// independent of the order.
#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int GG_TCH = 32;            // frames per work item
constexpr int GG_THREADS = 256;
constexpr int GG_BLOCKS = 296;        // partials per pair (fixed: the work size depends on B alone)
constexpr int GG_MAX_B = 128;
constexpr int GG_PITCH = GG_MAX_B + 1;   // odd pitch of the staged frame rows: conflict-free 8-byte stores along t
constexpr int GG_MAX_LAYERS = 1024;

__device__ __forceinline__ int gg_frames(const nbasr_gate_layer& l, int64_t len) {
  // L = min(T, ceil(len / 2^s)): the model's (T + 1) // 2 frame rule applied s times
  const int64_t v = len > 0 ? (len + ((int64_t)1 << l.s) - 1) >> l.s : 0;
  return (int)min((int64_t)l.T, v);
}

template <int PPT>
__global__ void __launch_bounds__(GG_THREADS) gate_gram_part_kernel(const nbasr_gate_layer* __restrict__ layers, int nlayers,
                                                                    const int64_t* __restrict__ audio_len, int B,
                                                                    uint64_t* __restrict__ part) {
  __shared__ uint64_t xs[GG_TCH * GG_PITCH];        // [t][b]
  __shared__ int64_t len_raw[GG_MAX_B];
  __shared__ int len_s[GG_MAX_B];                   // valid frames of the current item's layer
  __shared__ int item0[GG_MAX_LAYERS + 1];          // first work item of each layer
  const int npair = B * (B + 1) / 2;
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int l = 0; l < nlayers; ++l) {
      item0[l] = acc;
      const nbasr_gate_layer L = layers[l];
      const int planes = L.w > 0 ? (L.C + L.w - 1) / L.w : 0;
      acc += planes * ((L.T + GG_TCH - 1) / GG_TCH);
    }
    item0[nlayers] = acc;
  }
  for (int b = threadIdx.x; b < B; b += GG_THREADS) len_raw[b] = audio_len[b];
  // this thread's pairs q = tid + k * GG_THREADS, unpacked once: i in the low, j in the high half
  int pij[PPT];
#pragma unroll
  for (int k = 0; k < PPT; ++k) {
    const int q = threadIdx.x + k * GG_THREADS;
    int i = 0, r = q;
    if (q < npair)
      while (r >= B - i) { r -= B - i; ++i; }
    pij[k] = q < npair ? (i | ((i + r) << 16)) : -1;
  }
  uint64_t acc[PPT];
#pragma unroll
  for (int k = 0; k < PPT; ++k) acc[k] = 0;
  __syncthreads();
  const int nitems = item0[nlayers];
  int l = 0;
  for (int it = blockIdx.x; it < nitems; it += gridDim.x) {
    while (item0[l + 1] <= it) ++l;
    const nbasr_gate_layer L = layers[l];
    const int nchunk = (L.T + GG_TCH - 1) / GG_TCH;
    const int p = (it - item0[l]) / nchunk;
    const int t0 = ((it - item0[l]) % nchunk) * GG_TCH;
    const int live = min(L.w, L.C - p * L.w);       // live columns of this plane (the last plane of C = 600 / 800, w = 48)
    const uint64_t cm = live >= 64 ? ~0ull : ((1ull << live) - 1);
    const int nt = min(GG_TCH, L.T - t0);
    __syncthreads();                                  // the previous item's staged rows are no longer read
    for (int b = threadIdx.x; b < B; b += GG_THREADS) len_s[b] = gg_frames(L, len_raw[b]);
    __syncthreads();
    // stage entries (t0 + t, b) for t < min(nt, L_b - t0); rows b*Tp + PAD_L + t of plane p
    if (L.w == 32) {
      const uint32_t* src = static_cast<const uint32_t*>(L.mask) + (int64_t)p * L.mask_rows;
      for (int e = threadIdx.x; e < B * GG_TCH; e += GG_THREADS) {
        const int b = e / GG_TCH, t = e % GG_TCH;
        if (t < nt && t0 + t < len_s[b])
          xs[t * GG_PITCH + b] = (uint64_t)(__ldg(src + (int64_t)b * L.Tp + NBASR_PAD_L + t0 + t)) & cm;
      }
    } else {
      const uint64_t* src = static_cast<const uint64_t*>(L.mask) + (int64_t)p * L.mask_rows;
      for (int e = threadIdx.x; e < B * GG_TCH; e += GG_THREADS) {
        const int b = e / GG_TCH, t = e % GG_TCH;
        if (t < nt && t0 + t < len_s[b]) xs[t * GG_PITCH + b] = __ldg(src + (int64_t)b * L.Tp + NBASR_PAD_L + t0 + t) & cm;
      }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < PPT; ++k) {
      if (pij[k] < 0) continue;
      const int i = pij[k] & 0xffff, j = pij[k] >> 16;
      const int n = max(0, min(nt, min(len_s[i], len_s[j]) - t0));   // frames valid for both
      uint32_t d = 0;
      for (int t = 0; t < n; ++t) d += __popcll(xs[t * GG_PITCH + i] ^ xs[t * GG_PITCH + j]);
      acc[k] += (uint64_t)live * n - d;
    }
  }
  uint64_t* out = part + (int64_t)blockIdx.x * npair;
#pragma unroll
  for (int k = 0; k < PPT; ++k)
    if (pij[k] >= 0) out[threadIdx.x + k * GG_THREADS] = acc[k];
}

// thread q: the sum of the block partials of pair q, mirrored into both triangles
__global__ void gate_gram_reduce_kernel(const uint64_t* __restrict__ part, int B, uint64_t* __restrict__ K) {
  const int npair = B * (B + 1) / 2;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= npair) return;
  uint64_t acc = 0;
  for (int c = 0; c < GG_BLOCKS; ++c) acc += part[(int64_t)c * npair + q];
  int i = 0, r = q;
  while (r >= B - i) { r -= B - i; ++i; }
  const int j = i + r;
  K[i * B + j] = acc;
  K[j * B + i] = acc;
}

template <int PPT>
void launch_part(const nbasr_gate_layer* layers, int nlayers, const int64_t* audio_len, int B, uint64_t* work, cudaStream_t st) {
  gate_gram_part_kernel<PPT><<<GG_BLOCKS, GG_THREADS, 0, st>>>(layers, nlayers, audio_len, B, work);
}

}  // namespace

extern "C" int64_t nbasr_gate_gram_work_elems(int B) { return (int64_t)GG_BLOCKS * B * (B + 1) / 2; }

extern "C" int nbasr_gate_gram(const nbasr_gate_layer* layers, int nlayers, const int64_t* audio_len, int B, uint64_t* K,
                               uint64_t* work, void* stream) {
  NBASR_REQUIRE(B >= 1 && B <= GG_MAX_B, "1 <= B <= 128");
  NBASR_REQUIRE(nlayers >= 0 && nlayers <= GG_MAX_LAYERS, "at most 1024 layers");
  cudaStream_t st = as_stream(stream);
  const int ppt = (B * (B + 1) / 2 + GG_THREADS - 1) / GG_THREADS;      // pairs per thread: 1 (B <= 22) .. 33 (B = 128)
  if (ppt <= 1) launch_part<1>(layers, nlayers, audio_len, B, work, st);
  else if (ppt <= 3) launch_part<3>(layers, nlayers, audio_len, B, work, st);
  else if (ppt <= 9) launch_part<9>(layers, nlayers, audio_len, B, work, st);
  else if (ppt <= 17) launch_part<17>(layers, nlayers, audio_len, B, work, st);
  else launch_part<33>(layers, nlayers, audio_len, B, work, st);
  NBASR_CHECK_LAUNCH();
  const int npair = B * (B + 1) / 2;
  gate_gram_reduce_kernel<<<(npair + 255) / 256, 256, 0, st>>>(work, B, K);
  NBASR_CHECK_LAUNCH();
  return 0;
}
