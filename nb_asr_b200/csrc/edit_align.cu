// Phone error breakdown of a decoded batch: the Levenshtein alignment of each hypothesis against its reference, with
// substitution / deletion / insertion counts, per-position alignments and a confusion matrix (nbasr_edit_align,
// definition and tie rule in include/nbasr.h; oracle/edit_np.py restates it exactly).  One CTA per utterance, threads
// over the cells of an anti-diagonal, the layout of greedy_per_kernel's distance DP.
#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int EA_MAX_LEN = 32767;                 // H, S: cell values n + m fit in 16 bits
constexpr int EA_MAX_V = 64;
constexpr int EA_MAX_THREADS = 1024;
constexpr int64_t EA_SMEM_MAX = 220 * 1024;

int ea_threads(int S) { return std::min(EA_MAX_THREADS, ((S + 1 + 31) / 32) * 32); }
__host__ __device__ int ea_words(int S) { return (S + 1 + 31) / 32; }       // backpointer words (uint2) per anti-diagonal

// hyp and ref as bytes (V <= 64), three rotating anti-diagonals of uint16 cell values, then (16-byte aligned) the
// backpointers when they fit: 2 bits per cell, two ballot words per 32 cells, (H + S + 1) diagonals
__host__ __device__ int64_t ea_fixed_bytes(int H, int S) { return ((int64_t)H + S + 3 * 2 * ((int64_t)S + 1) + 15) & ~(int64_t)15; }
int64_t ea_bp_bytes(int H, int S) { return (int64_t)8 * ((int64_t)H + S + 1) * ea_words(S); }
bool ea_bp_in_smem(int H, int S) { return ea_fixed_bytes(H, S) + ea_bp_bytes(H, S) <= EA_SMEM_MAX; }

// move codes (tie order): diagonal (hit or substitution), deletion (ref token to nothing, j - 1), insertion (i - 1)
constexpr unsigned EA_DIAG = 0, EA_DEL = 1, EA_INS = 2;

__global__ void __launch_bounds__(EA_MAX_THREADS) edit_align_kernel(
    const int32_t* __restrict__ hyp, const int32_t* __restrict__ hyp_len, int H, const int32_t* __restrict__ targets, int S,
    const int64_t* __restrict__ targets_len, const int32_t* __restrict__ lut, int V, int32_t* __restrict__ counts,
    int32_t* __restrict__ ref_at, int32_t* __restrict__ hyp_at, unsigned long long* __restrict__ confusion,
    uint2* __restrict__ bp_work, int bp_in_smem) {
  extern __shared__ __align__(16) unsigned char ea_sm[];
  __shared__ int s_wcnt[EA_MAX_THREADS / 32];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nt = blockDim.x;
  const int nw = ea_words(S);
  uint8_t* hy = ea_sm;
  uint8_t* ref = hy + H;
  uint16_t* dg = reinterpret_cast<uint16_t*>(ea_sm + ((H + S + 1) & ~1));
  uint2* bp = bp_in_smem ? reinterpret_cast<uint2*>(ea_sm + ea_fixed_bytes(H, S))
                         : bp_work + (int64_t)b * (H + S + 1) * nw;
  const int n = max(0, min(H, hyp_len[b]));
  const int mr = (int)max((int64_t)0, min((int64_t)S, targets_len[b]));
  const int32_t* hg = hyp + (int64_t)b * H;
  const int32_t* tg = targets + (int64_t)b * S;
  int32_t* ra = ref_at + (int64_t)b * H;
  int32_t* ha = hyp_at + (int64_t)b * S;

  // hyp as given (folded, no zeros: ids in [1, V)); ref = targets folded through lut with zeros dropped (ids in [0, V)
  // before and after lut), compacted by a block-wide ballot scan.  A row with an id out of range is refused.
  bool bad = false;
  for (int i = tid; i < n; i += nt) {
    const int c = hg[i];
    bad |= c < 1 || c >= V;
    hy[i] = (uint8_t)c;
  }
  int m = 0;
  for (int j0 = 0; j0 < mr; j0 += nt) {
    const int j = j0 + tid;
    int f = 0;
    if (j < mr) {
      const int c = tg[j];
      if (c < 0 || c >= V) {
        bad = true;
      } else {
        f = lut ? lut[c] : c;
        if (f < 0 || f >= V) { bad = true; f = 0; }
      }
    }
    const unsigned keep = __ballot_sync(0xffffffffu, f != 0);
    if (lane == 0) s_wcnt[warp] = __popc(keep);
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < (nt >> 5); ++w) {
      const int c = s_wcnt[w];
      before += w < warp ? c : 0;
      total += c;
    }
    if (f != 0) ref[m + before + __popc(keep & ((1u << lane) - 1u))] = (uint8_t)f;
    m += total;
    __syncthreads();
  }
  if (__syncthreads_or(bad)) {
    for (int i = tid; i < H; i += nt) ra[i] = -1;
    for (int j = tid; j < S; j += nt) ha[j] = -1;
    if (tid < 4) counts[(int64_t)b * 4 + tid] = -1;
    return;
  }
  for (int i = n + tid; i < H; i += nt) ra[i] = -1;
  for (int j = m + tid; j < S; j += nt) ha[j] = -1;

  // D(i, j) over anti-diagonals k = i + j, cell (i, j) at index j of diagonal k (i over hyp, j over ref):
  //   D = min(D(i-1, j-1) + [hyp[i-1] != ref[j-1]], D(i, j-1) + 1, D(i-1, j) + 1); the first of diagonal, deletion,
  //   insertion that attains the minimum is the cell's move (on the borders the only move there is)
  uint16_t* pm2 = dg;
  uint16_t* pm1 = dg + (S + 1);
  uint16_t* cur = dg + 2 * (S + 1);
  for (int k = 0; k <= n + m; ++k) {
    const int jlo = max(0, k - n), jhi = min(m, k);
    uint2* row = bp + (int64_t)k * nw;
    for (int j0 = 0; j0 <= jhi; j0 += nt) {
      const int wj = j0 + (warp << 5);
      if (wj > jhi || wj + 31 < jlo) continue;            // warp-uniform: no cell of this warp is on the diagonal
      const int j = wj + lane, i = k - j;
      unsigned mv = 0;
      if (j >= jlo && j <= jhi) {
        int v;
        if (j == 0) {
          v = i; mv = EA_INS;
        } else if (i == 0) {
          v = j; mv = EA_DEL;
        } else {
          const int dia = pm2[j - 1] + (hy[i - 1] != ref[j - 1] ? 1 : 0);
          const int del = pm1[j - 1] + 1;
          const int ins = pm1[j] + 1;
          v = dia; mv = EA_DIAG;
          if (del < v) { v = del; mv = EA_DEL; }
          if (ins < v) { v = ins; mv = EA_INS; }
        }
        cur[j] = (uint16_t)v;
      }
      const unsigned lo = __ballot_sync(0xffffffffu, mv & 1u), hi = __ballot_sync(0xffffffffu, mv >> 1);
      if (lane == 0) row[wj >> 5] = make_uint2(lo, hi);
    }
    __syncthreads();
    uint16_t* x = pm2; pm2 = pm1; pm1 = cur; cur = x;
  }
  if (tid != 0) return;
  // backtrace from (n, m): every hyp and every ref position is written exactly once
  int i = n, j = m, hits = 0, subs = 0, dels = 0, ins = 0;
  while (i > 0 || j > 0) {
    const uint2 w = bp[(int64_t)(i + j) * nw + (j >> 5)];
    const int bit = j & 31;
    const unsigned mv = ((w.x >> bit) & 1u) | (((w.y >> bit) & 1u) << 1);
    int rc, hc;
    if (mv == EA_DIAG) {
      --i; --j;
      rc = ref[j]; hc = hy[i];
      ra[i] = j; ha[j] = i;
      if (rc == hc) ++hits; else ++subs;
    } else if (mv == EA_DEL) {
      --j;
      rc = ref[j]; hc = 0;
      ha[j] = -1;
      ++dels;
    } else {
      --i;
      rc = 0; hc = hy[i];
      ra[i] = -1;
      ++ins;
    }
    atomicAdd(confusion + rc * V + hc, 1ull);
  }
  int32_t* cb = counts + (int64_t)b * 4;
  cb[0] = hits; cb[1] = subs; cb[2] = dels; cb[3] = ins;
}

}  // namespace

extern "C" {

int64_t nbasr_edit_align_work_bytes(int B, int H, int S) {
  if (B <= 0 || H < 0 || S < 0 || H > EA_MAX_LEN || S > EA_MAX_LEN || ea_bp_in_smem(H, S)) return 0;
  return (int64_t)B * ea_bp_bytes(H, S);
}

int nbasr_edit_align(const int32_t* hyp, const int32_t* hyp_len, int H, const int32_t* targets, int S,
                     const int64_t* targets_len, const int32_t* lut, int B, int V, int32_t* counts, int32_t* ref_at,
                     int32_t* hyp_at, uint64_t* confusion, void* work, void* stream) {
  NBASR_REQUIRE(B >= 0 && H >= 0 && S >= 0 && V >= 1, "edit_align shape");
  if (H > EA_MAX_LEN || S > EA_MAX_LEN)
    return nbasr_fail("edit_align: H = %d hypothesis / S = %d reference tokens; each must stay below %d (cell values "
                      "are 16-bit)", H, S, EA_MAX_LEN + 1);
  if (V > EA_MAX_V)
    return nbasr_fail("edit_align: V = %d classes exceeds the supported %d (tokens are kept as bytes)", V, EA_MAX_V);
  if (ea_fixed_bytes(H, S) > EA_SMEM_MAX)
    return nbasr_fail("edit_align: H = %d, S = %d need %lld bytes of shared memory for the sequences and three "
                      "anti-diagonals; at most %lld are available", H, S, (long long)ea_fixed_bytes(H, S),
                      (long long)EA_SMEM_MAX);
  if (B == 0) return 0;
  const bool in_smem = ea_bp_in_smem(H, S);
  NBASR_REQUIRE(in_smem || work != nullptr, "edit_align: backpointers exceed shared memory and work is NULL "
                                            "(size it with nbasr_edit_align_work_bytes)");
  const size_t sm = (size_t)ea_fixed_bytes(H, S) + (in_smem ? (size_t)ea_bp_bytes(H, S) : 0);
  static DevOnce attr;
  if (!attr) { cudaFuncSetAttribute(edit_align_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EA_SMEM_MAX); attr = true; }
  edit_align_kernel<<<B, ea_threads(S), sm, as_stream(stream)>>>(
      hyp, hyp_len, H, targets, S, targets_len, lut, V, counts, ref_at, hyp_at,
      reinterpret_cast<unsigned long long*>(confusion), reinterpret_cast<uint2*>(work), in_smem ? 1 : 0);
  NBASR_CHECK_LAUNCH();
  return 0;
}

}  // extern "C"
