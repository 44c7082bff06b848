// Grouped conv edges (ops.py:73-76, groups=100, cpg = C/100 in {6,8,10,12}) on tcgen05 tensor cores.
//
// A grouped conv is HBM-bound (15-42 FLOP/B in bf16) but CUDA-core FMA cannot reach the HBM roofline
// (SURVEY.md 7.3), so the groups are evaluated as BLOCK-DIAGONAL MMAs: a slab of OUT = 48 (40 for
// cpg = 10) consecutive channels = 8/6/4/4 whole groups is one 128 x 48 x 48 MMA per tap whose weight
// tile is zero outside the diagonal blocks (8x..4x redundant tensor FLOPs, still far below the HBM time).
//
//  * The input tile (128 frames + halo) x 64 channels is TMA-loaded ONCE per (frame tile, slab) in the
//    128B-swizzled K-major layout; every (dilated) tap is the SAME tile addressed through a UMMA
//    descriptor whose start address is advanced by whole 128-byte rows (swizzle is a function of the
//    absolute smem address, verified on B200 with tools/experiments/dbg.cu) -- no im2col, no per-tap reload.
//  * A CTA keeps one slab's block-diagonal weights (<= 7 taps x 6 KB) in smem and walks frame tiles;
//    2 CTAs / SM, 3-stage TMA ring, 4 TMEM accumulator stages.  Warps 0..11: epilogue (three column thirds x four TMEM
//    lane quadrants, each quadrant staging and storing on its own), warp 12: TMA producer, warp 13: MMA issue (last =
//    highest issue priority; warp-uniform loop, one elected lane issues).
//  * Forward and input-gradient share the kernel (different weight pack / tap offsets); the fused
//    epilogue (bias, ReLU20, dropout, skip-sum, gradient mask) works on 8-column groups because slab
//    boundaries are only 8-aligned.
//  * Weight gradient: dW_j[co][ci] = sum_t dZ[t][co] X[t+off_j][ci], both operands MN-major (frames
//    are the reduction index).  ALL taps share one M=128 x N=64*ceil(k/2) MMA per 16-frame K step: the A
//    descriptor's "leading byte offset" makes rows 64..127 the same dZ tile shifted by `dstep` frames, the
//    B descriptor's makes N atom i the same X tile shifted by 2 i dstep frames, so (atom i, rows 64-127)
//    gives tap 2i and (atom i, rows 0-63) tap 2i+1.  Diagonal blocks are extracted from TMEM, assembled into the slab's
//    contiguous gradient run in shared memory and added to the fp32 gradient with 16-byte reductions.  X may be the forward's scaled fp16 activation: the drain warps convert each landed tile
//    to bf16 in place before the MMAs read it, so a 16-bit plan keeps no bf16 copy of it.
#include <cuda.h>

#include "common.cuh"
#include "kernels.h"
#include "sm100_ptx.cuh"

using namespace sm100;

namespace {

constexpr int GT = 128;                    // frames per tile
constexpr int AROWS = 144;                 // 128 + max halo 12, multiple of 8
constexpr int A_BYTES = AROWS * 128;       // 18432
constexpr int NW = 48;                     // MMA N (and K window) of a slab
constexpr int WTAP_BYTES = NW * 128;       // 6144
constexpr int NSTAGE = 3;                  // (weight-gradient kernel)
constexpr int NACC = 4;
constexpr int GC_THREADS = 192;            // weight-gradient kernel: 4 drain warps, producer, MMA
constexpr int FWD_THREADS = 448;           // forward kernel: 12 epilogue warps, producer, MMA
constexpr int NEPI = 384;                  // (three column thirds x four TMEM lane quadrants)
constexpr int OSTAGE_BYTES = GT * NW * 2;  // 12288: bf16 output tile staged for the TMA store
constexpr int FWD_SMEM_BUDGET = 112 * 1024;
constexpr int GCONV_SLOTS = 2;             // resident CTAs per SM the grouped-conv kernels size their persistent grids for

__host__ __device__ inline int slab_out(int cpg) { return cpg == 10 ? 40 : 48; }
// weight-gradient slabs: as many whole groups as fit in 56 channels: 54 / 56 / 50 / 48 for cpg 6 / 8 / 10 / 12 -> fewer,
// fuller 128-byte loads.  TMA boxes must start on a 16-byte (8-channel) boundary, so the box starts at c0 & ~7 and the
// slab sits at offset c0 & 7 inside the 64-channel window; channel 63 of the window is never part of a slab and carries
// the ones column of the fused bias gradient.
__host__ __device__ inline int wg_slab_out(int cpg) { return (56 / cpg) * cpg; }
__host__ __device__ inline int fwd_nstage(int ktaps) {
  int n = (FWD_SMEM_BUDGET - 3072 - ktaps * WTAP_BYTES - 2 * OSTAGE_BYTES) / A_BYTES;
  return n > 4 ? 4 : n;
}

struct GcFwdArgs {
  int B, T, C, OUT, ktaps, dstep, off0;
  int nslabs, ntiles, tiles_per_utt, nlanes, nstage, no_prefetch, w_stable, f16;
  nbasr_epilogue epi;
  int64_t Tp;
};


// Epilogue of the forward / input-gradient kernel.  12 warps: warps (w, w+4, w+8) share a TMEM lane quadrant and split the
// 48 accumulator columns in thirds of 16 (the 40-column slabs of C = 1000: 16 + 16 + 8).  ncu r2: with 8 warps the kernel sat
// at IPC 2.0 with 4 epilogue warps per scheduler, each issuing one instruction per ~9 cycles (fixed-latency, scoreboard and
// barrier stalls) while the MMAs + loads alone ran at the 88-cycle issue floor -- the epilogue lacked warps, not pipes.  Results are staged in shared memory as a dense
// [128][OUT] bf16 tile and written with ONE TMA store per output tensor (coalesced, asynchronous); only the
// gate-bit bytes and optional skip-sum reads stay per-thread accesses.
__global__ void __launch_bounds__(FWD_THREADS, 2)
gconv_mma_fwd_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW,
                     const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmO2, const GcFwdArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* al = smem_raw + (base - smem_u32(smem_raw));
  const int NS = p.nstage;
  const uint32_t wsm = base;
  const uint32_t asm0 = base + p.ktaps * WTAP_BYTES;
  const uint32_t osm = asm0 + NS * A_BYTES;          // out staging, then out2 staging
  const uint32_t bar0 = osm + 2 * OSTAGE_BYTES;
  uint8_t* ost = al + p.ktaps * WTAP_BYTES + NS * A_BYTES;
  uint8_t* mst = ost + 2 * OSTAGE_BYTES + 256;    // 128 x 8-byte gate-bit entries
  const uint32_t wbar = bar0;
  auto full_bar = [&](int s) { return bar0 + 8u * (1 + s); };
  auto empty_bar = [&](int s) { return bar0 + 8u * (1 + 4 + s); };
  auto tfull_bar = [&](int s) { return bar0 + 8u * (1 + 8 + s); };
  auto tempty_bar = [&](int s) { return bar0 + 8u * (1 + 8 + NACC + s); };
  uint32_t* tptr = reinterpret_cast<uint32_t*>(ost + 2 * OSTAGE_BYTES + 8 * (1 + 8 + 2 * NACC));
  const int warp = uniform_warp_idx(), lane = threadIdx.x & 31;
  // Warp roles: 0 .. 11 epilogue, 12 producer, 13 MMA issue.  The issue arbiter of a scheduler prefers the HIGHEST warp id
  // (B300_MICROARCH.md, multi-warp arbiter), so the single thread that issues the MMAs must not sit below twelve busy
  // epilogue warps: as warp 1 it was starved by them (ablation r2: MMAs + loads alone ran at the 88-cycle issue floor, 62 us per
  // three nodes; any epilogue arithmetic pushed the kernel to 124 us whatever its pipe mix or warp count).
  constexpr int W_PROD = NEPI / 32, W_MMA = NEPI / 32 + 1;
  const int slab = blockIdx.x % p.nslabs;
  const int lane_id = blockIdx.x / p.nslabs;
  const int c0 = slab * p.OUT;

  if (warp == W_PROD && lane == 0) {
    prefetch_tmap(&tmX);
    prefetch_tmap(&tmW);
    mbar_init(wbar, 1);
    for (int s = 0; s < NS; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < NACC; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), NEPI); }
    fence_barrier_init();
  }
  if (warp == W_MMA) tmem_alloc(smem_u32(tptr), 256);
  pdl_launch_dependents();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tm = *tptr;
  // w_packed bit 1 (NBASR_W_STABLE): the caller states that the weight pack was NOT written by the launch this one depends
  // on (the engine re-packs in the optimiser tail of the previous step, many launches earlier), so its load may start before
  // the dependency wait and overlap the previous kernel's tail.
  auto load_weights = [&]() {
    mbar_expect_tx(wbar, p.ktaps * WTAP_BYTES);
    for (int j = 0; j < p.ktaps; ++j) tma_load_2d(wsm + j * WTAP_BYTES, &tmW, wbar, 0, (slab * p.ktaps + j) * NW);
  };
  if (p.w_stable && warp == W_PROD && lane == 0) load_weights();
  pdl_wait();                                  // everything above overlapped the previous kernel's tail
  if (!p.w_stable && warp == W_PROD && lane == 0) load_weights();

  if (warp == W_PROD) {
    // The epilogue's per-thread operands (skip-sum tensors, gate bits of the second output) are loaded AFTER the accumulator
    // is ready, so their latency sits on the epilogue's critical path (1 skip operand: 55 -> 92 us per launch).  The whole
    // producer warp therefore L2-prefetches them for each tile at the moment that tile's input load is issued, i.e. NS tiles
    // ahead of their use (the register prefetch tried earlier spilled).
    const int esz = p.epi.add_dtype == NBASR_F32 ? 4 : 2;
    const bool pf_mask = p.epi.out2 && p.epi.mask2;
    const int pl2 = pf_mask ? c0 / p.epi.mask2_w : 0;
    const int eb2 = p.epi.mask2_w == 32 ? 4 : 8;
    int stage = 0, it = 0;
    uint32_t phase = 0;
    for (int tile = lane_id; tile < p.ntiles; tile += p.nlanes, ++it) {
      const int b = tile / p.tiles_per_utt, t0 = (tile % p.tiles_per_utt) * GT;
      if (lane == 0) {
        mbar_wait(empty_bar(stage), phase ^ 1);
        mbar_expect_tx(full_bar(stage), A_BYTES);
        tma_load_3d(asm0 + stage * A_BYTES, &tmX, full_bar(stage), c0, NBASR_PAD_L + t0 + p.off0, b);
      }
      __syncwarp();
      if (!p.no_prefetch) {
        const int64_t rho0 = (int64_t)b * p.Tp + NBASR_PAD_L + t0;
        const int nr = min(GT, p.T - t0);
        const int ncols = min(p.OUT, p.C - c0);
        for (int a = 0; a < p.epi.n_add; ++a) {
          const char* base = reinterpret_cast<const char*>(p.epi.add[a]) + (rho0 * p.epi.ld_out + c0) * esz;
          for (int r = lane; r < nr; r += 32) {
            const char* q = base + (int64_t)r * p.epi.ld_out * esz;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(q));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(q + ncols * esz - 1));
          }
        }
        if (pf_mask) {
          // this slab's 8 column groups may straddle two mask planes when the widths differ: prefetch both row ranges
          const char* m0 = reinterpret_cast<const char*>(p.epi.mask2) + ((int64_t)pl2 * p.epi.mask_rows + rho0) * eb2;
          const char* m1 = reinterpret_cast<const char*>(p.epi.mask2) +
                           ((int64_t)((c0 + ncols - 1) / p.epi.mask2_w) * p.epi.mask_rows + rho0) * eb2;
          const int nb = nr * eb2;
          for (int o = lane * 128; o < nb + 127; o += 32 * 128) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(m0 + min(o, nb - 1)));
            if (m1 != m0) asm volatile("prefetch.global.L2 [%0];" ::"l"(m1 + min(o, nb - 1)));
          }
        }
      }
      if (++stage == NS) { stage = 0; phase ^= 1; }
    }
  } else if (warp == W_MMA) {
    // the whole warp walks the tile loop (uniform control flow: loop state and UMMA descriptors in uniform registers); one
    // elected lane issues the MMAs and the commits
    const uint32_t idesc = make_idesc(128, NW, 0, 0, p.f16);
    mbar_wait(wbar, 0);
    int stage = 0, it = 0;
    uint32_t phase = 0;
    // descriptors advance by adding to the 14-bit start-address field (bytes >> 4): no carry can leave it (smem < 256 KB)
    const uint64_t bd0 = make_smem_desc(wsm, 16, 1024);
    for (int tile = lane_id; tile < p.ntiles; tile += p.nlanes, ++it) {
      const int as = it % NACC;
      const uint32_t aphase = (it / NACC) & 1;
      mbar_wait(tempty_bar(as), aphase ^ 1);
      mbar_wait(full_bar(stage), phase);
      tcgen05_fence_after();
      const uint64_t ad0 = make_smem_desc(asm0 + stage * A_BYTES, 16, 1024);
      if (elect_one()) {
        for (int j = 0; j < p.ktaps; ++j) {
#pragma unroll
          for (int k = 0; k < NW / 16; ++k)
            umma_bf16(tm + as * 64, ad0 + (uint64_t)(j * p.dstep * 8 + k * 2), bd0 + (uint64_t)(j * (WTAP_BYTES >> 4) + k * 2), idesc, (j | k) != 0);
        }
        umma_commit(empty_bar(stage));
        umma_commit(tfull_bar(as));
      }
      __syncwarp();
      if (++stage == NS) { stage = 0; phase ^= 1; }
    }
  } else {
    const int ew = warp;                     // 0..11
    const int q = warp & 3;                  // TMEM lane quadrant of this warp
    const int hh = ew >> 2;                  // column third: cols [16*hh, 16*hh + 16)
    const int row = q * 32 + lane;
    const int cbeg = c0 + 16 * hh;
    const int nvalid = max(0, min(16, min(p.C, c0 + p.OUT) - cbeg));     // multiple of 8
    const int OUTB = p.OUT * 2;              // staged row pitch in bytes
    const nbasr_epilogue& epi = p.epi;       // stays in the kernel-parameter bank (a local copy would live on the stack)
    // scaled fp16 activations (nbasr.h): v = acc * acc_scale + bias * bias_scale, clamp at relu_hi
    const float acc_s = epi_acc_scale(epi), bias_s = epi_bias_scale(epi), relu_hi = epi_relu_hi(epi);
    const uint32_t hi_bits = __float_as_uint(relu_hi);
    float bias_r[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) bias_r[i] = (epi.bias && i < nvalid) ? __ldg(epi.bias + cbeg + i) * bias_s : 0.f;
    int it = 0;
    for (int tile = lane_id; tile < p.ntiles; tile += p.nlanes, ++it) {
      const int as = it % NACC;
      const uint32_t aphase = (it / NACC) & 1;
      const int b = tile / p.tiles_per_utt, t0 = (tile % p.tiles_per_utt) * GT;
      const int t = t0 + row;
      // gate bits of the second output (input gradient: dZ of the previous node): requested BEFORE waiting for the
      // accumulator so that their latency overlaps the MMAs instead of sitting between the epilogue's two barriers
      uint32_t w2[2] = {0xffu, 0xffu};
      if (epi.out2 && epi.mask2 && t < p.T) {
        const int64_t rho2 = (int64_t)b * p.Tp + NBASR_PAD_L + t;
#pragma unroll
        for (int g = 0; g < 2; ++g)
          if (g * 8 < nvalid) w2[g] = reinterpret_cast<const uint8_t*>(epi.mask2)[mask_byte_addr(rho2, cbeg + g * 8, epi.mask2_w, epi.mask_rows)];
      }
      mbar_wait(tfull_bar(as), aphase);
      tcgen05_fence_after();
      float v[16];
      const uint32_t ta = tm + ((uint32_t)(q * 32) << 16) + as * 64 + 16 * hh;
      tmem_ld16_nowait(ta, v);
      tmem_ld_wait();
      tcgen05_fence_before();
      mbar_arrive(tempty_bar(as));           // accumulator is in registers: release the TMEM stage early
      const bool rowok = t < p.T;
      const int64_t rho = (int64_t)b * p.Tp + NBASR_PAD_L + t;
      uint32_t m[2] = {0, 0};
      if (rowok) {
        if (nvalid == 16 && epi.drop_p == 0.f && epi.n_add == 0) {
          // lean path (every forward of a skip-free node, most input-gradients): ~6 instructions / element
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            uint32_t mm = 0xffu;
            if (epi.relu20) {
              mm = 0;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float z = fmaf(v[g * 8 + i], acc_s, bias_r[g * 8 + i]);
                // 0 < z <= hi  <=>  bits(z) - 1 < bits(hi) as unsigned (negative z and +0 wrap to huge values)
                mm |= ((__float_as_uint(z) - 1u) < hi_bits) ? (1u << i) : 0u;
                v[g * 8 + i] = fminf(fmaxf(z, 0.f), relu_hi);
              }
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i) v[g * 8 + i] = fmaf(v[g * 8 + i], acc_s, bias_r[g * 8 + i]);
            }
            m[g] = mm;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = fmaf(v[i], acc_s, bias_r[i]);
          if (nvalid == 16) epilogue_compute<16, true, true>(epi, rho, cbeg, 16, v, m);
          else epilogue_compute<16, false, true>(epi, rho, cbeg, nvalid, v, m);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = 0.f;      // rows past the utterance land on zero pad rows / are clipped
      }
      // The four TMEM lane quadrants (32 frames each, three warps) stage, synchronise and store INDEPENDENTLY: quadrant q owns
      // rows 32 q .. 32 q + 31 of the staging tile, named barrier 1 + q (96 threads) and its own TMA stores / bulk groups
      // (leader: lane 0 of warp q), so a slow warp or a pending store only holds up its own quadrant.
      const bool qlead = hh == 0 && lane == 0;
      // the quadrant's staging rows are free once ITS previous TMA stores have finished READING shared memory
      if (qlead) bulk_wait_read0();
      named_bar_sync(1 + q, 96);
      uint8_t* orow = ost + row * OUTB + 32 * hh;
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        if (g * 8 < nvalid) {
          if (epi.out) store8_h(orow + g * 16, epi.out_dtype, v + g * 8);
          if (epi.out2) {
            float t2[8];
            if (epi.mask2) {               // gated second output (input gradient: dZ of the previous node)
              const uint32_t w = w2[g];
#pragma unroll
              for (int i = 0; i < 8; ++i) t2[i] = ((w >> i) & 1u) ? v[g * 8 + i] * epi.scale2 : 0.f;
            } else {                       // plain scaled copy (forward: the weight gradient's bf16 operand): no bit tests
#pragma unroll
              for (int i = 0; i < 8; ++i) t2[i] = v[g * 8 + i] * epi.scale2;
            }
            store8_h(orow + OSTAGE_BYTES + g * 16, epi.out2_dtype, t2);
          }
        }
        if (epi.mask_out) mst[row * 8 + 2 * hh + g] = (g * 8 < nvalid) ? (uint8_t)m[g] : (uint8_t)0;   // 8-byte entry per row
      }
      fence_async_smem();
      named_bar_sync(1 + q, 96);
      if (epi.mask_out && hh == 0 && t < p.T) {
        // 32 consecutive 8-byte entries of this slab's mask plane (warp q = the quadrant's rows): one coalesced store
        const int64_t r2 = (int64_t)b * p.Tp + NBASR_PAD_L + t;
        reinterpret_cast<uint64_t*>(epi.mask_out)[(int64_t)slab * epi.mask_rows + r2] = reinterpret_cast<const uint64_t*>(mst)[row];
      }
      if (qlead) {
        const uint32_t qoff = (uint32_t)(q * 32 * OUTB);
        if (epi.out) tma_store_3d(&tmO, osm + qoff, c0, NBASR_PAD_L + t0 + 32 * q, b);
        if (epi.out2) tma_store_3d(&tmO2, osm + OSTAGE_BYTES + qoff, c0, NBASR_PAD_L + t0 + 32 * q, b);
        bulk_commit();
      }
    }
    if (hh == 0 && lane == 0) bulk_wait0();
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == W_MMA) {
    tcgen05_fence_after();
    tmem_dealloc(tm, 256);
  }
}

// ---------------------------------------------------------------- weight gradient
constexpr int DZROWS = 136;                       // 128 + dstep(<=2), multiple of 8
constexpr int DZ_BYTES = DZROWS * 128;            // 17408
constexpr int WG_STAGE = DZ_BYTES + A_BYTES;      // 35840
constexpr int WG_SMEM = NSTAGE * WG_STAGE + 1024 + 256;

struct GcWgArgs {
  int B, T, C, cpg, OUT, ktaps, dstep, off0;
  int nslabs, nchunks, nunits, nlanes;
  int x_f16;      // X is fp16 holding x / x_scale (the forward's scaled activation): converted to bf16 in shared memory
  float x_scale;
  float* dw;
  float* dbias;   // optional: db[c] += sum_t dZ[t][c], computed by the tensor core against a column of ones
};

__global__ void __launch_bounds__(GC_THREADS, 2)
gconv_mma_wgrad_kernel(const __grid_constant__ CUtensorMap tmDZ, const __grid_constant__ CUtensorMap tmX, const GcWgArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* al = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar0 = base + NSTAGE * WG_STAGE;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (NSTAGE + s); };
  const uint32_t tfull = bar0 + 8u * (2 * NSTAGE);
  auto ready_bar = [&](int s) { return bar0 + 8u * (2 * NSTAGE + 1 + s); };     // X tile converted / ones column written
  uint32_t* tptr = reinterpret_cast<uint32_t*>(al + NSTAGE * WG_STAGE + 8 * (3 * NSTAGE + 2));
  // warp roles: 0..3 drain (and, in the main loop, X tile preparation), 4 producer, 5 MMA issue (highest id: issue priority)
  const int warp = uniform_warp_idx(), lane = threadIdx.x & 31;
  const int slab = blockIdx.x % p.nslabs;
  const int lane_id = blockIdx.x / p.nslabs;
  const int c0 = slab * p.OUT;
  const int cbox = c0 & ~7, coff = c0 - cbox;       // TMA box start (16-byte aligned) and slab offset inside the window
  const int npairs = (p.ktaps + 1) / 2;

  if (warp == 4 && lane == 0) {
    prefetch_tmap(&tmDZ);
    prefetch_tmap(&tmX);
    for (int s = 0; s < NSTAGE; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); mbar_init(ready_bar(s), 4); }
    mbar_init(tfull, 1);
    fence_barrier_init();
  }
  if (warp == 5) tmem_alloc(smem_u32(tptr), 256);
  pdl_launch_dependents();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tm = *tptr;
  pdl_wait();
  const bool has_work = lane_id < p.nunits;

  if (warp == 4) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = lane_id; u < p.nunits; u += p.nlanes) {
        const int b = u / p.nchunks, t0 = (u % p.nchunks) * GT;
        mbar_wait(empty_bar(stage), phase ^ 1);
        mbar_expect_tx(full_bar(stage), DZ_BYTES + A_BYTES);
        const uint32_t sa = base + stage * WG_STAGE;
        tma_load_3d(sa, &tmDZ, full_bar(stage), cbox, NBASR_PAD_L + t0 - p.dstep, b);
        tma_load_3d(sa + DZ_BYTES, &tmX, full_bar(stage), cbox, NBASR_PAD_L + t0 + p.off0, b);
        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 5) {
    if (has_work) {
      // ONE MMA per 16-frame K step covers every tap: the B descriptor's leading-byte offset (2 dstep rows) makes the
      // N atoms 0..npairs-1 the same X tile shifted by 0, 2, 4, .. taps, the A descriptor's (dstep rows) makes rows
      // 64..127 / 0..63 the dZ tile unshifted / shifted by one tap: atom i, rows 64..127 -> tap 2i, rows 0..63 -> tap 2i+1.
      // (A tcgen05.mma costs ~88 cycles of issue whatever N <= 176 is, 96 at N = 192, 128 at N = 256: tools/dbg_bench.py.)
      // Uniform control flow, one elected lane issues: the descriptors stay in uniform registers (one add per MMA).
      const uint32_t idesc = make_idesc(128, 64 * npairs, 1, 1);
      int stage = 0;
      uint32_t phase = 0;
      bool first = true;
      for (int u = lane_id; u < p.nunits; u += p.nlanes) {
        // with fp16 X or a bias gradient the stage is usable once the drain warps have prepared its X tile (below)
        mbar_wait((p.x_f16 || p.dbias) ? ready_bar(stage) : full_bar(stage), phase);
        const uint32_t sa = base + stage * WG_STAGE;
        tcgen05_fence_after();
        const uint64_t ad0 = make_smem_desc(sa, (uint32_t)p.dstep * 128u, 1024);
        const uint64_t bd0 = make_smem_desc(sa + DZ_BYTES, 2u * (uint32_t)p.dstep * 128u, 1024);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < GT / 16; ++k)
            umma_bf16(tm, ad0 + (uint64_t)(k * 128), bd0 + (uint64_t)(k * 128), idesc, (!first || k > 0) ? 1u : 0u);
          umma_commit(empty_bar(stage));
        }
        __syncwarp();
        first = false;
        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) umma_commit(tfull);
      __syncwarp();
    }
  } else if (has_work) {
    if (p.x_f16 || p.dbias) {
      // Warps 0..3, idle until the drain, prepare each landed X tile for the MMAs, each on its own AROWS / 4 rows, OFF the MMA
      // warp's critical path (ncu r2: tensor pipe 37 % busy with the ones-column write + proxy fence in front of every unit's
      // MMAs when the MMA warp did it itself):
      //  * fp16 X -> bf16 in place, x * x_scale rounded once (x_scale = 1/S is a power of two: exact before the rounding).
      //    Element-wise, so the 128B swizzle (a permutation of whole 16-byte chunks within a row) does not matter.
      //  * bias gradient = dZ^T 1: channel 63 of the X window (never part of a slab) <- 1.0 for every frame row (element 7 of
      //    the 16-byte chunk 7, at its swizzled position chunk ^ (row & 7)).
      constexpr int QROWS = AROWS / 4;
      const int r0 = warp * QROWS;
      int stage = 0;
      uint32_t phase = 0;
      for (int u = lane_id; u < p.nunits; u += p.nlanes) {
        mbar_wait(full_bar(stage), phase);
        uint8_t* xb = al + stage * WG_STAGE + DZ_BYTES;
        if (p.x_f16) {
#pragma unroll 3
          for (int i = lane; i < QROWS * 8; i += 32) {          // 16-byte chunks, 8 per row: 9 per lane
            const int r = r0 + (i >> 3), ch = i & 7;
            uint4* cp = reinterpret_cast<uint4*>(xb + r * 128 + ch * 16);
            uint4 w = *cp;
            uint32_t* h = &w.x;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = f16x2_to_f2(h[e]);
              h[e] = f2_to_bf16x2(f.x * p.x_scale, f.y * p.x_scale);
            }
            if (p.dbias && ch == (7 ^ (r & 7))) w.w = (w.w & 0xffffu) | (0x3F80u << 16);
            *cp = w;
          }
        } else {
          for (int r = r0 + lane; r < r0 + QROWS; r += 32)
            *reinterpret_cast<uint16_t*>(xb + r * 128 + ((7 ^ (r & 7)) << 4) + 14) = 0x3F80;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(ready_bar(stage));
        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
      }
    }
    const int q = warp & 3;
    const int m = q * 32 + lane;
    const int half = m >> 6, co_l = m & 63;
    const int co = cbox + co_l;
    const bool row_ok = co_l >= coff && co_l < coff + p.OUT && co < p.C;
    const int g_l = (co_l - coff) / p.cpg;
    // The slab's gradient dw[c0 .. c0 + nco)[cpg][ktaps] is ONE contiguous run of nco * cpg * ktaps floats (<= 16 KB).  The
    // drain warps assemble it in the stage buffers, idle once every MMA has completed (tfull) -- each element is written
    // exactly once: a thread owns one output channel, the two TMEM halves hold disjoint taps -- and add it to global memory
    // with 16-byte reductions, 4x fewer than one fp32 atomic per element (those were ~15 % of the kernel's time).  The run
    // starts `pad` floats into shared memory so that its 16-byte-aligned global stretch is 16-byte aligned there too.
    const int nco = min(p.OUT, p.C - c0);
    const int nrun = nco * p.cpg * p.ktaps;
    float* g = p.dw + (int64_t)c0 * p.cpg * p.ktaps;
    const int head = min(nrun, (int)(((16u - (uint32_t)(reinterpret_cast<uintptr_t>(g) & 15u)) & 15u) >> 2));
    float* run = reinterpret_cast<float*>(al) + ((4 - head) & 3);
    mbar_wait(tfull, 0);
    tcgen05_fence_after();
    for (int pr = 0; pr < npairs; ++pr) {
      float v[64];
      const uint32_t ta = tm + ((uint32_t)(q * 32) << 16) + pr * 64;
      tmem_ld32(ta, v);
      tmem_ld32(ta + 32, v + 32);
      const int tap = half ? 2 * pr : 2 * pr + 1;
      // column 63 of atom 0, rows 64..127 (tap 0, unshifted dZ) = sum_t dZ[t][co]
      if (pr == 0 && p.dbias && row_ok && half) atomicAdd(p.dbias + co, v[63]);
      if (row_ok && tap < p.ktaps) {
        float* dst = run + (co_l - coff) * p.cpg * p.ktaps + tap;
#pragma unroll
        for (int i = 0; i < 64; ++i) {
          const int il = i - coff - g_l * p.cpg;
          if (il >= 0 && il < p.cpg) dst[il * p.ktaps] = v[i];
        }
      }
    }
    named_bar_sync(1, 128);
    const int tid = threadIdx.x;                      // 0 .. 127: the drain warps
    const int nvec = (nrun - head) >> 2, tail = head + 4 * nvec;
    if (tid < head) atomicAdd(g + tid, run[tid]);
    for (int j = tid; j < nvec; j += 128)
      atomicAdd(reinterpret_cast<float4*>(g + head) + j, reinterpret_cast<const float4*>(run + head)[j]);
    if (tail + tid < nrun) atomicAdd(g + tail + tid, run[tail + tid]);
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 5) {
    tcgen05_fence_after();
    tmem_dealloc(tm, 256);
  }
}

// ---------------------------------------------------------------- weight packs (fp32 master -> bf16 block diagonal)
// out[slab][tap][n (48 rows)][kk (64 cols)], transposed=0: forward  (n = c_out, kk = c_in, tap j)
//                                            transposed=1: dgrad    (n = c_in, kk = c_out, tap k-1-j)
template <typename T>
__global__ void pack_gconv_mma_kernel(const float* __restrict__ w, T* __restrict__ out, int C, int cpg, int ktaps, int OUT,
                                      int nslabs, int transposed) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)nslabs * ktaps * NW * 64;
  if (idx >= total) return;
  int kk = (int)(idx % 64);
  int n = (int)((idx / 64) % NW);
  int j = (int)((idx / (64 * NW)) % ktaps);
  int s = (int)(idx / ((int64_t)64 * NW * ktaps));
  int c0 = s * OUT;
  int cn = c0 + n, ck = c0 + kk;
  float v = 0.f;
  if (n < OUT && cn < C && ck < C && kk < NW && (cn / cpg) == (ck / cpg)) {
    if (!transposed) v = w[((int64_t)cn * cpg + (ck % cpg)) * ktaps + j];
    else v = w[((int64_t)ck * cpg + (cn % cpg)) * ktaps + (ktaps - 1 - j)];
  }
  out[idx] = static_cast<T>(v);
}

}  // namespace

int sm100_gconv_fwd(const nbasr_gconv* g, cudaStream_t st) {
  GcFwdArgs a{};
  a.B = g->B; a.T = g->T; a.Tp = g->Tp; a.C = g->C; a.OUT = slab_out(g->cpg);
  a.ktaps = g->ktaps; a.dstep = g->dstep; a.off0 = g->off0;
  NBASR_REQUIRE(a.off0 >= -NBASR_PAD_L && (a.ktaps - 1) * a.dstep <= AROWS - GT, "tap reach");
  NBASR_REQUIRE(g->epi.ld_out == g->C, "grouped conv writes dense (B,Tp,C) tensors");
  NBASR_REQUIRE((!g->epi.out || g->epi.out_dtype != NBASR_F32) && (!g->epi.out2 || g->epi.out2_dtype != NBASR_F32) &&
                    !g->epi.accumulate, "tcgen05 grouped conv stores 16-bit tensors");
  NBASR_REQUIRE(g->epi.n_add == 0 || g->epi.add_dtype != NBASR_F32, "tcgen05 grouped conv adds 16-bit skip tensors");
  a.f16 = g->dtype == NBASR_F16 ? 1 : 0;
  a.nslabs = (g->C + a.OUT - 1) / a.OUT;
  a.tiles_per_utt = (g->T + GT - 1) / GT;
  a.ntiles = a.tiles_per_utt * g->B;
  a.nstage = fwd_nstage(a.ktaps);
  int slots = GCONV_SLOTS * nbasr_sm_count();
  a.nlanes = std::max(1, std::min(a.ntiles, slots / a.nslabs));
  a.epi = g->epi;
  a.no_prefetch = nbasr_env_flag(NBASR_ENV_GCONV_NO_PREFETCH) ? 1 : 0;
  a.w_stable = (g->w_packed & 2) ? 1 : 0;
  CUtensorMap tmX, tmW, tmO, tmO2;
  uint64_t dx[3] = {(uint64_t)g->C, (uint64_t)g->Tp, (uint64_t)g->B};
  int64_t sx[3] = {1, g->C, (int64_t)g->Tp * g->C};
  uint32_t bx[3] = {64, AROWS, 1};
  if (sm100_get_map(g->x, 3, dx, sx, bx, &tmX)) return 1;
  uint64_t dw[2] = {64, (uint64_t)a.nslabs * a.ktaps * NW};
  int64_t sw[2] = {1, 64};
  uint32_t bw[2] = {64, NW};
  if (sm100_get_map(g->w, 2, dw, sw, bw, &tmW)) return 1;
  uint32_t bo[3] = {(uint32_t)a.OUT, 32, 1};             // one store per TMEM lane quadrant (32 frames)
  const void* o1 = g->epi.out ? g->epi.out : g->x;       // unused maps still need a valid descriptor
  const void* o2 = g->epi.out2 ? g->epi.out2 : g->x;
  if (sm100_get_map(o1, 3, dx, sx, bo, &tmO, 0)) return 1;
  if (sm100_get_map(o2, 3, dx, sx, bo, &tmO2, 0)) return 1;
  NBASR_REQUIRE(!g->epi.mask_out || g->epi.mask_w == a.OUT, "grouped-conv mask planes are slab wide");
  size_t smem = (size_t)a.ktaps * WTAP_BYTES + (size_t)a.nstage * A_BYTES + 2 * OSTAGE_BYTES + 1024 + 256 + 1024;
  static DevOnce attr;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(gconv_mma_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM_BUDGET);
    if (e != cudaSuccess) return nbasr_fail("gconv_mma_fwd smem attr: %s", cudaGetErrorString(e));
    attr = true;
  }
  cudaError_t le = launch_pdl(gconv_mma_fwd_kernel, dim3(a.nslabs * a.nlanes), dim3(FWD_THREADS), smem, st, 1, tmX, tmW, tmO, tmO2, a);
  if (le != cudaSuccess) return nbasr_fail("gconv_mma_fwd launch: %s", cudaGetErrorString(le));
  return 0;
}

int sm100_gconv_wgrad(const void* dz, const void* x, int x_f16, float x_scale, int B, int T, int Tp, int C, int cpg, int ktaps,
                      int off0, int dstep, float* dw, float* dbias, cudaStream_t st) {
  GcWgArgs a{};
  a.x_f16 = x_f16;
  a.x_scale = x_scale;
  a.B = B; a.T = T; a.C = C; a.cpg = cpg; a.OUT = wg_slab_out(cpg); a.ktaps = ktaps; a.dstep = dstep; a.off0 = off0;
  NBASR_REQUIRE(off0 >= -NBASR_PAD_L && (ktaps - 1) * dstep <= AROWS - GT && dstep <= DZROWS - GT, "tap reach");
  a.nslabs = (C + a.OUT - 1) / a.OUT;
  a.nchunks = (T + dstep + GT - 1) / GT;
  a.nunits = a.nchunks * B;
  int slots = GCONV_SLOTS * nbasr_sm_count();
  a.nlanes = std::max(1, std::min(a.nunits, slots / a.nslabs));
  a.dw = dw;
  a.dbias = dbias;
  CUtensorMap tmDZ, tmX;
  uint64_t dd[3] = {(uint64_t)C, (uint64_t)Tp, (uint64_t)B};
  int64_t sd[3] = {1, C, (int64_t)Tp * C};
  uint32_t bz[3] = {64, DZROWS, 1};
  uint32_t bx[3] = {64, AROWS, 1};
  if (sm100_get_map(dz, 3, dd, sd, bz, &tmDZ)) return 1;
  if (sm100_get_map(x, 3, dd, sd, bx, &tmX)) return 1;
  static DevOnce attr;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(gconv_mma_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM);
    if (e != cudaSuccess) return nbasr_fail("gconv_mma_wgrad smem attr: %s", cudaGetErrorString(e));
    attr = true;
  }
  cudaError_t le = launch_pdl(gconv_mma_wgrad_kernel, dim3(a.nslabs * a.nlanes), dim3(GC_THREADS), (size_t)WG_SMEM, st, 1, tmDZ, tmX, a);
  if (le != cudaSuccess) return nbasr_fail("gconv_mma_wgrad launch: %s", cudaGetErrorString(le));
  return 0;
}

extern "C" int nbasr_pack_gconv_mma(const float* w, void* out, int out_dtype, int C, int cpg, int ktaps, int transposed, void* stream) {
  int OUT = slab_out(cpg);
  int nslabs = (C + OUT - 1) / OUT;
  int64_t total = (int64_t)nslabs * ktaps * NW * 64;
  NBASR_REQUIRE(out_dtype == NBASR_BF16 || out_dtype == NBASR_F16, "16-bit pack");
  const unsigned grid = (unsigned)((total + 255) / 256);
  if (out_dtype == NBASR_F16) pack_gconv_mma_kernel<f16><<<grid, 256, 0, as_stream(stream)>>>(w, (f16*)out, C, cpg, ktaps, OUT, nslabs, transposed);
  else pack_gconv_mma_kernel<bf16><<<grid, 256, 0, as_stream(stream)>>>(w, (bf16*)out, C, cpg, ktaps, OUT, nslabs, transposed);
  NBASR_CHECK_LAUNCH();
  return 0;
}

extern "C" int64_t nbasr_gconv_mma_pack_elems(int C, int cpg, int ktaps) {
  int OUT = slab_out(cpg);
  return (int64_t)((C + OUT - 1) / OUT) * ktaps * NW * 64;
}
