// CTC forced alignment: the Viterbi path of a known target sequence through the CTC trellis (nbasr_ctc_align, definition and
// tie rule in include/nbasr.h; oracle/align_np.py restates it bit-exactly).  One CTA per utterance, one thread per state of
// the extended label sequence, the same layout as ctc_kernel's alpha recursion with max in place of logadd.
#include <math_constants.h>

#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int AL_MAX_THREADS = 1024;                     // one thread per state: 2S + 1 <= 1024
constexpr int AL_MAX_S = (AL_MAX_THREADS - 1) / 2;       // 511
constexpr int AL_PF = 8;                                 // emissions requested this many frames ahead
constexpr int64_t AL_SMEM_MAX = 200 * 1024;

int al_threads(int S) { return ((2 * S + 1 + 31) / 32) * 32; }

// Backpointers: 2 bits per (frame, state), two ballot words (bit 0, bit 1 of the move) per warp and frame = 8 bytes per
// 32 states.  They sit in shared memory beside the two alpha rows (8 bytes per 32 states as well) when both fit.
bool al_bp_in_smem(int T, int S) { return (int64_t)8 * (al_threads(S) / 32) * ((int64_t)T + 32) <= AL_SMEM_MAX; }

__global__ void __launch_bounds__(AL_MAX_THREADS) ctc_align_kernel(
    const float* __restrict__ logp, int T, int V, const int32_t* __restrict__ targets, int S, const int64_t* __restrict__ audio_len,
    int len_div, const int64_t* __restrict__ targets_len, int32_t* labels, int32_t* tok, int32_t* __restrict__ start,
    int32_t* __restrict__ end, float* __restrict__ score, uint2* __restrict__ bp_work, int bp_in_smem) {
  extern __shared__ __align__(16) float al_sm[];
  __shared__ int s_end;
  const int b = blockIdx.x, s = threadIdx.x, lane = s & 31, nw = blockDim.x >> 5;
  float* prev = al_sm;
  float* cur = al_sm + blockDim.x;
  uint2* bp = bp_in_smem ? reinterpret_cast<uint2*>(al_sm + 2 * blockDim.x) : bp_work + (int64_t)b * T * nw;
  const float NEG = -CUDART_INF_F;
  const int Tb = (int)max((int64_t)0, min((int64_t)T, audio_len[b] / len_div));
  const int Sb = (int)max((int64_t)0, min((int64_t)S, targets_len[b]));
  const int L = 2 * Sb + 1;
  const float* lp = logp + (int64_t)b * T * V;
  const int32_t* tg = targets + (int64_t)b * S;
  int32_t* lab = labels + (int64_t)b * T;
  int32_t* tk = tok + (int64_t)b * T;
  int32_t* st0 = start + (int64_t)b * S;
  int32_t* en0 = end + (int64_t)b * S;

  const bool on = s < L;
  const int es = (on && (s & 1)) ? tg[s >> 1] : 0;
  const bool skip_ok = on && (s & 1) && s >= 3 && tg[(s >> 1) - 1] != es;
  // a target id outside [1, V) would index past the log-prob row: the row is refused (score NaN, outputs -1)
  if (__syncthreads_or(on && (s & 1) && (es < 1 || es >= V))) {
    for (int t = s; t < T; t += blockDim.x) { lab[t] = -1; tk[t] = -1; }
    for (int j = s; j < S; j += blockDim.x) { st0[j] = -1; en0[j] = -1; }
    if (s == 0) score[b] = CUDART_NAN_F;
    return;
  }

  prev[s] = (on && s < 2 && Tb > 0) ? __ldg(lp + es) : NEG;
  float ring[AL_PF];
#pragma unroll
  for (int u = 0; u < AL_PF; ++u) ring[u] = (on && 1 + u < Tb) ? __ldg(lp + (int64_t)(1 + u) * V + es) : 0.f;
  __syncthreads();
  // alpha_t(s) = max(alpha(s), alpha(s-1), alpha(s-2) if skip_ok) + logp[t, ext[s]]; strict > keeps the smaller jump on ties
  for (int t0 = 1; t0 < Tb; t0 += AL_PF) {
#pragma unroll
    for (int u = 0; u < AL_PF; ++u) {
      const int t = t0 + u;
      if (t < Tb) {
        float a = prev[s];
        unsigned m = 0;
        if (s >= 1) {
          const float v = prev[s - 1];
          if (v > a) { a = v; m = 1; }
        }
        if (skip_ok) {
          const float v = prev[s - 2];
          if (v > a) { a = v; m = 2; }
        }
        const float e = ring[u];
        if (on && t + AL_PF < Tb) ring[u] = __ldg(lp + (int64_t)(t + AL_PF) * V + es);
        cur[s] = on ? a + e : NEG;
        const unsigned lo = __ballot_sync(0xffffffffu, m & 1u), hi = __ballot_sync(0xffffffffu, m >> 1);
        if (lane == 0) bp[(int64_t)t * nw + (s >> 5)] = make_uint2(lo, hi);
        __syncthreads();
        float* x = prev; prev = cur; cur = x;
      }
    }
  }
  if (s == 0) {          // end state: the trailing blank 2S_b unless the last label is strictly better
    int se = -1;
    float sc = Sb == 0 ? 0.f : NEG;
    if (Tb > 0) {
      se = L - 1;
      sc = prev[L - 1];
      if (L >= 2 && prev[L - 2] > sc) { se = L - 2; sc = prev[L - 2]; }
      if (sc == NEG) se = -1;
    }
    s_end = se;
    score[b] = sc;
  }
  __syncthreads();
  if (s_end < 0) {       // no frames, or no path
    for (int t = s; t < T; t += blockDim.x) { lab[t] = -1; tk[t] = -1; }
    for (int j = s; j < S; j += blockDim.x) { st0[j] = -1; en0[j] = -1; }
    return;
  }
  // Backtrace by warp 0, 32 frames per round: lane k fetches the backpointer words of frame tc - k that the walk can touch
  // (a move is at most 2 states, so 31 moves span at most three 32-state words), then the whole warp walks the 32 frames
  // with shuffles.  The state path is parked in `labels` and rewritten below.
  if (s < 32) {
    int st = s_end;
    for (int tc = Tb - 1; tc >= 0; tc -= 32) {
      const int f = tc - lane;
      const int w0 = max(st - 62, 0) >> 5;
      uint2 q0 = make_uint2(0u, 0u), q1 = q0, q2 = q0;
      if (f >= 1) {
        const uint2* row = bp + (int64_t)f * nw;
        q0 = row[w0];
        if (w0 + 1 < nw) q1 = row[w0 + 1];
        if (w0 + 2 < nw) q2 = row[w0 + 2];
      }
      int mine = 0;
      for (int k = 0; k < 32 && tc - k >= 0; ++k) {
        if (lane == k) mine = st;
        if (tc - k >= 1) {
          const int i = (st >> 5) - w0;
          const uint2 q = i == 0 ? q0 : (i == 1 ? q1 : q2);
          const unsigned lo = __shfl_sync(0xffffffffu, q.x, k), hi = __shfl_sync(0xffffffffu, q.y, k);
          const int bit = st & 31;
          st -= (int)(((lo >> bit) & 1u) | (((hi >> bit) & 1u) << 1));
        }
      }
      if (f >= 0) lab[f] = mine;
    }
  }
  __syncthreads();
  // token of each frame and the half-open frame span of each token (a CTC path visits a label state in one run)
  for (int t = s; t < Tb; t += blockDim.x) {
    const int st = lab[t];
    if (st & 1) {
      const int j = st >> 1;
      tk[t] = j;
      if (t == 0 || lab[t - 1] != st) st0[j] = t;
      if (t == Tb - 1 || lab[t + 1] != st) en0[j] = t + 1;
    } else {
      tk[t] = -1;
    }
  }
  for (int j = Sb + s; j < S; j += blockDim.x) { st0[j] = -1; en0[j] = -1; }
  __syncthreads();
  for (int t = s; t < T; t += blockDim.x) {
    if (t < Tb) {
      const int st = lab[t];
      lab[t] = (st & 1) ? tg[st >> 1] : 0;
    } else {
      lab[t] = -1;
      tk[t] = -1;
    }
  }
}

}  // namespace

extern "C" {

int64_t nbasr_ctc_align_work_bytes(int B, int T, int S) {
  if (B <= 0 || T <= 0 || S < 0 || S > AL_MAX_S || al_bp_in_smem(T, S)) return 0;
  return (int64_t)8 * B * T * (al_threads(S) / 32);
}

int nbasr_ctc_align(const float* logp, int B, int T, int V, const int32_t* targets, int S, const int64_t* audio_len, int len_div,
                    const int64_t* targets_len, int32_t* labels, int32_t* tok, int32_t* start, int32_t* end, float* score,
                    void* work, void* stream) {
  NBASR_REQUIRE(B >= 0 && T >= 0 && V >= 1 && S >= 0 && len_div >= 1, "ctc_align shape");
  if (S > AL_MAX_S)
    return nbasr_fail("ctc_align: S = %d target tokens exceeds the supported %d (one thread per state of the 2S+1 extended "
                      "labels, %d threads per CTA)", S, AL_MAX_S, AL_MAX_THREADS);
  if (B == 0) return 0;
  const int threads = al_threads(S);
  const bool in_smem = al_bp_in_smem(T, S);
  NBASR_REQUIRE(in_smem || work != nullptr, "ctc_align: backpointers exceed shared memory and work is NULL "
                                            "(size it with nbasr_ctc_align_work_bytes)");
  const size_t sm = sizeof(float) * 2 * threads + (in_smem ? (size_t)8 * (threads / 32) * T : 0);
  static DevOnce attr;
  if (!attr) { cudaFuncSetAttribute(ctc_align_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AL_SMEM_MAX); attr = true; }
  ctc_align_kernel<<<B, threads, sm, as_stream(stream)>>>(logp, T, V, targets, S, audio_len, len_div, targets_len, labels, tok,
                                                          start, end, score, reinterpret_cast<uint2*>(work), in_smem ? 1 : 0);
  NBASR_CHECK_LAUNCH();
  return 0;
}

}  // extern "C"
