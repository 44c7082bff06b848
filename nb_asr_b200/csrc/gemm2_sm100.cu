// Dense GEMM  C[(b,r), n] = sum_k A[(b,r), k] W[n, k]  on CTA PAIRS (tcgen05 cta_group::2): the time-reduction
// convolutions, `linear` edges, the LSTM input projection and their input-gradients (see include/nbasr.h).
//
// Why pairs: measured on B200 (tools/bench_gemm.py) the 1-CTA kernel (gemm_sm100.cu, 128 x 256 tile) needs ~750 cycles
// per 64-deep K block although its four MMAs take 512 -- an SM ingests ~64 B/clk from L2 and the tile needs
// 16 KB (A) + 32 KB (B) per K block.  With cta_group::2 two SMs of a TPC share one 256 x BN MMA: each CTA loads ITS
// 128 rows of A and only HALF of the B tile (BN/2 rows), so ingest drops to 16 + 16 KB per K block (= 512 cycles at
// 64 B/clk, the MMA time), and a stage is 32 KB, so the TMA ring is 6 deep.
//
// Structure per CTA: 8 (direct epilogue) or 16 (staged epilogue) epilogue warps first, then the TMA producer warp, then the
// MMA issuer (leader CTA only) as the LAST warp -- the issue arbiter prefers the highest warp id -- walking its loop in
// warp-uniform control flow with one elected lane issuing (round 2).  Synchronisation:
//   full[s]   lives in the LEADER: both producers arrive.expect_tx on it (count 2) and both CTAs' TMA loads
//             complete_tx on it (.cta_group::2 lets a load signal the peer's barrier);
//   empty[s]  in each CTA, arrived by the leader's tcgen05.commit multicast to both CTAs;
//   tfull[a]  in each CTA, same multicast commit; each CTA's epilogue drains ITS half (TMEM lanes = its 128 rows);
//   tempty[a] in the leader: one arrive per epilogue warp of both CTAs (count 16, the peer arrives remotely).
#include <cuda.h>

#include <cstdlib>

#include "common.cuh"
#include "kernels.h"
#include "sm100_ptx.cuh"

using namespace sm100;

namespace {

constexpr int BM = 128;                 // rows per CTA (256 per pair)
constexpr int BK = 64;
constexpr int STAGES = 6;
constexpr int A_STAGE_BYTES = BM * BK * 2;          // 16 KB
constexpr int B_STAGE_BYTES = 128 * BK * 2;         // up to BN/2 = 128 rows: 16 KB
constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
constexpr int THREADS = 320;                        // direct epilogue: 8 epilogue warps, producer, MMA
// Staged epilogue (16-bit outputs).  ncu on the direct version (profiles/r2_ncu_gemm_linear800.txt): a `linear` edge
// (K = 600..1200: 3 us of MMAs per 256 x 224 tile) is EPILOGUE-bound -- 8 epilogue warps were busy 86 % of the time, the tensor
// pipe 45 %, and per-thread 16-byte row stores half-use 32-byte sectors.  So:
//  * 16 epilogue warps (4 per TMEM lane quadrant, every 4th 32-column chunk each): twice the latency hiding;
//  * every epilogue warp owns two 32 x 32 boxes of shared memory (64-byte-swizzled TMA layout): the skip operands of a chunk
//    arrive in them by TMA LOAD, are summed into the registers, then the boxes carry `out` / `out2` to a TMA STORE -- global
//    traffic moves in full 64-byte row segments;
//  * the bias of a chunk is one coalesced load per warp, broadcast by shuffles (not 32 loads per thread);
//  * the accumulator stage is released with a RELAXED cluster arrive (a release compiles to MEMBAR.ALL + ERRBAR, 15 % of the
//    epilogue's samples; the TMEM reads are already ordered by tcgen05.wait::ld + fence::before_thread_sync).
constexpr int ST_THREADS = 576;                     // 16 epilogue warps, producer, MMA (<= 112 registers per thread)
constexpr int ST_EPI_WARPS = 16;
constexpr int ST_STAGES = 5;                        // 5 x 32 KB ring + 64 KB staging
constexpr int ST_WARP_BYTES = 4096;
constexpr int ST_BOX_BYTES = 2048;
constexpr int ST_SMEM_BYTES = ST_STAGES * STAGE_BYTES + ST_EPI_WARPS * ST_WARP_BYTES + 1024 + 256;

struct Args {
  int nb, nr, K, N, BN, f16, n_add_staged, l2_prefetch;
  int mt_per_utt, m_tiles, n_tiles, pair_tiles;
  int64_t o_r0, o_bs, o_rs;
  nbasr_epilogue epi;
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive (+ expect_tx) on a barrier that may live in the peer CTA (shared::cluster address)
__device__ __forceinline__ void mbar_expect_tx_cluster(uint32_t bar_cluster, uint32_t bytes) {
  // .relaxed: a cluster-scope release here compiles to MEMBAR + ERRBAR, which waits for the producer's outstanding TMA
  // loads and serialises the whole ring (ncu: ~1 us per K block); the data itself is published by complete_tx.
  asm volatile("mbarrier.arrive.expect_tx.relaxed.cluster.shared::cluster.b64 _, [%0], %1;" ::"r"(bar_cluster), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t bar_cluster) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}
// TMA loads whose completion is signalled on a barrier of either CTA of the pair
__device__ __forceinline__ void tma2_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma2_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          dst),
      "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of all prior MMAs -> one arrive on the barrier at the same offset in both CTAs of the pair
__device__ __forceinline__ void umma2_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}

struct StMaps {      // tensor maps of the staged epilogue: out, out2, up to three skip tensors (all the same geometry)
  CUtensorMap o, o2, a0, a1, a2;
};

template <bool STAGED>
__global__ void __launch_bounds__(STAGED ? ST_THREADS : THREADS, 1)
gemm_tn_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ StMaps sm,
                    const Args p) {
  constexpr int STAGES = STAGED ? ST_STAGES : ::STAGES;
  constexpr int EPI_WARPS = STAGED ? ST_EPI_WARPS : 8;
  constexpr int NSUB = EPI_WARPS / 4;               // epilogue warps per TMEM lane quadrant
  constexpr int STG_BYTES = STAGED ? ST_EPI_WARPS * ST_WARP_BYTES : 0;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + STAGES * STAGE_BYTES + STG_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + 2 + s); };
  auto add_bar = [&](int w) { return bar_base + 8u * (2 * STAGES + 4 + w); };      // one per epilogue warp (staged)
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(smem_al + STAGES * STAGE_BYTES + STG_BYTES + 8 * (2 * STAGES + 4 + 16));

  // Warp roles: 0 .. EPI_WARPS-1 epilogue, then the producer, then the MMA warp LAST: the issue arbiter prefers the highest warp
  // id, and as warp 1 the thread that issues the MMAs was starved by the epilogue warps (see gconv_sm100.cu, r2).
  constexpr int W_PROD = EPI_WARPS, W_MMA = EPI_WARPS + 1;
  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair_id = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int num_kb = (p.K + BK - 1) / BK;
  const int half_bn = p.BN >> 1;

  if (warp == W_PROD && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 2);       // one arrive.expect_tx per CTA of the pair (used in the leader only)
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), 2 * EPI_WARPS);    // every epilogue warp of both CTAs (used in the leader only)
    }
    if (STAGED) {
      prefetch_tmap(&sm.o);
      for (int w = 0; w < EPI_WARPS; ++w) mbar_init(add_bar(w), 1);
    }
    fence_barrier_init();
  }
  if (warp == W_MMA) tmem_alloc2(smem_u32(tmem_ptr_smem), 512);
  pdl_launch_dependents();
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();                  // both CTAs' barriers are initialised before any remote arrive / multicast
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();

  if (warp == W_PROD) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t stage_tx = A_STAGE_BYTES + half_bn * BK * 2;
      // optional L2 prefetch cursor, `l2_prefetch` K blocks ahead of the load cursor (across tile boundaries)
      int ppt = pair_id, pkb = 0;
      auto pf_issue = [&]() {
        if (ppt < p.pair_tiles) {
          const int pn = ppt % p.n_tiles;
          const int pm = min(2 * (ppt / p.n_tiles) + (int)rank, p.m_tiles - 1);
          tma_prefetch_3d(&tmA, pkb * BK, (pm % p.mt_per_utt) * BM, pm / p.mt_per_utt);
          tma_prefetch_2d(&tmB, pkb * BK, pn * p.BN + (int)rank * half_bn);
          if (++pkb == num_kb) { pkb = 0; ppt += npairs; }
        }
      };
      for (int i = 0; i < p.l2_prefetch; ++i) pf_issue();
      for (int pt = pair_id; pt < p.pair_tiles; pt += npairs) {
        const int n_idx = pt % p.n_tiles;
        const int m_idx = min(2 * (pt / p.n_tiles) + (int)rank, p.m_tiles - 1);   // odd tile count: the peer repeats the last tile
        const int b = m_idx / p.mt_per_utt, r0 = (m_idx % p.mt_per_utt) * BM;
        for (int kb = 0; kb < num_kb; ++kb) {
          if (p.l2_prefetch) pf_issue();
          mbar_wait(empty_bar(stage), phase ^ 1);
          const uint32_t sa = smem_base + stage * STAGE_BYTES;
          const uint32_t sb = sa + A_STAGE_BYTES;
          const uint32_t fb = mapa(full_bar(stage), 0);
          mbar_expect_tx_cluster(fb, stage_tx);
          tma2_load_3d(sa, &tmA, fb, kb * BK, r0, b);
          tma2_load_2d(sb, &tmB, fb, kb * BK, n_idx * p.BN + (int)rank * half_bn);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == W_MMA) {
    if (rank == 0) {
      // the whole warp walks the loop (uniform control flow: descriptors in uniform registers, one add per MMA instead of the
      // ELECT / R2UR.BROADCAST sequence ptxas emits inside `if (lane == 0)`); one elected lane issues MMAs and commits
      const uint32_t idesc = make_idesc(2 * BM, p.BN, 0, 0, p.f16);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int pt = pair_id; pt < p.pair_tiles; pt += npairs, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(tempty_bar(as), aphase ^ 1);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + as * 256;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          const uint32_t sa = smem_base + stage * STAGE_BYTES;
          const uint64_t ad0 = make_smem_desc(sa, 16, 1024), bd0 = make_smem_desc(sa + A_STAGE_BYTES, 16, 1024);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) umma2_bf16(d_tmem, ad0 + (uint64_t)(2 * k), bd0 + (uint64_t)(2 * k), idesc, (kb | k) != 0);
            umma2_commit(empty_bar(stage));
            if (kb == num_kb - 1) umma2_commit(tfull_bar(as));
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    const int q = warp & 3;           // TMEM lane quadrant this warp may access
    const int sub = warp >> 2;        // the NSUB warps of a quadrant take every NSUB-th 32-column chunk
    // staged epilogue state: this warp's two 2 KB boxes and its skip-operand barrier
    const int ew = warp;
    uint8_t* stg = smem_al + STAGES * STAGE_BYTES + ew * ST_WARP_BYTES;
    const uint32_t stg_u = smem_base + STAGES * STAGE_BYTES + ew * ST_WARP_BYTES;
    const uint32_t abar = add_bar(ew);
    uint32_t aphase = 0;
    const int na = p.n_add_staged;
    // byte offset of 16-byte chunk j of this lane's row inside a 64-byte-swizzled 32 x 32 box (bits 4-5 ^= bits 7-8)
    const int sw_row = lane * 64, sw_x = (lane >> 1) & 3;
    int it = 0;
    for (int pt = pair_id; pt < p.pair_tiles; pt += npairs, ++it) {
      const int as = it & 1;
      const uint32_t aphase_t = (it >> 1) & 1;
      const int n_idx = pt % p.n_tiles;
      const int m_raw = 2 * (pt / p.n_tiles) + (int)rank;
      const int m_idx = min(m_raw, p.m_tiles - 1);
      const int b = m_idx / p.mt_per_utt, r0 = (m_idx % p.mt_per_utt) * BM;
      const int r = r0 + q * 32 + lane;
      const int n0 = n_idx * p.BN;
      const int ncol = min(p.N, n0 + p.BN);
      const int64_t rho = p.o_r0 + (int64_t)b * p.o_bs + (int64_t)r * p.o_rs;
      if (!STAGED) {
        mbar_wait(tfull_bar(as), aphase_t);
        tcgen05_fence_after();
        for (int c = 32 * sub; c < p.BN; c += 32 * NSUB) {
          if (n0 + c >= ncol) break;   // warp-uniform
          float v[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + as * 256 + c, v);
          if (r < p.nr && m_raw < p.m_tiles) epilogue_chunk(p.epi, rho, n0 + c, ncol, v);
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa(tempty_bar(as), 0));
      } else {
        const nbasr_epilogue& e = p.epi;
        const int rbox = r0 + q * 32;                                   // first row of this warp's 32-row box
        const bool box_ok = m_raw < p.m_tiles && rbox < p.nr;           // warp-uniform
        const float acc_s = epi_acc_scale(e), bias_s = epi_bias_scale(e), relu_hi = epi_relu_hi(e);
        const uint32_t hi_bits = __float_as_uint(relu_hi);
        const bool plain = e.drop_p == 0.f;                              // (dropout goes through the general routine)
        // Skip operands of chunk c -> this warp's boxes.  The boxes also carry the previous chunk's results to their TMA
        // stores, so the stores must have finished READING shared memory first.
        auto load_adds = [&](int c) {
          if (box_ok && na > 0 && lane == 0 && c < p.BN && n0 + c < ncol) {   // (only chunks that will be processed)
            bulk_wait_read0();
            mbar_expect_tx(abar, ST_BOX_BYTES * min(na, 2));
            tma_load_3d(stg_u, &sm.a0, abar, n0 + c, rbox, b);
            if (na > 1) tma_load_3d(stg_u + ST_BOX_BYTES, &sm.a1, abar, n0 + c, rbox, b);
          }
        };
        auto add_box = [&](int box, float* v) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float t[8];
            load8_h(stg + box * ST_BOX_BYTES + sw_row + ((j ^ sw_x) << 4), e.add_dtype, t);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[j * 8 + i] += t[i];
          }
        };
        load_adds(32 * sub);                  // before the accumulator wait: the load overlaps the tile's last MMAs
        mbar_wait(tfull_bar(as), aphase_t);
        tcgen05_fence_after();
        for (int c = 32 * sub; c < p.BN; c += 32 * NSUB) {
          if (n0 + c >= ncol) break;   // warp-uniform
          // bias of this chunk: one coalesced load per warp (lane i <- column c + i), broadcast by shuffles below
          float bl = 0.f;
          if (e.bias && n0 + c + lane < ncol) bl = __ldg(e.bias + n0 + c + lane) * bias_s;
          float v[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + as * 256 + c, v);
          if (box_ok) {
            const int nvalid = min(32, ncol - (n0 + c));
            uint32_t m[4];
            if (plain) {
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                uint32_t mm = 0xffu;
                if (e.relu20) {
                  mm = 0;
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const float z = fmaf(v[g * 8 + i], acc_s, __shfl_sync(0xffffffffu, bl, g * 8 + i));
                    // 0 < z <= hi  <=>  bits(z) - 1 < bits(hi) as unsigned (negative z and +0 wrap to huge values)
                    mm |= ((__float_as_uint(z) - 1u) < hi_bits) ? (1u << i) : 0u;
                    v[g * 8 + i] = fminf(fmaxf(z, 0.f), relu_hi);
                  }
                } else {
#pragma unroll
                  for (int i = 0; i < 8; ++i) v[g * 8 + i] = fmaf(v[g * 8 + i], acc_s, __shfl_sync(0xffffffffu, bl, g * 8 + i));
                }
                m[g] = mm;
              }
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = fmaf(v[i], acc_s, __shfl_sync(0xffffffffu, bl, i));
              if (nvalid == 32) epilogue_compute<32, true, true, true>(e, rho, n0 + c, 32, v, m);
              else epilogue_compute<32, false, true, true>(e, rho, n0 + c, nvalid, v, m);
            }
            if (na > 0) {
              mbar_wait(abar, aphase);
              aphase ^= 1;
              add_box(0, v);
              if (na > 1) add_box(1, v);
              if (na > 2) {                     // third skip tensor: through the first box once everyone has read it
                __syncwarp();
                if (lane == 0) {
                  mbar_expect_tx(abar, ST_BOX_BYTES);
                  tma_load_3d(stg_u, &sm.a2, abar, n0 + c, rbox, b);
                }
                mbar_wait(abar, aphase);
                aphase ^= 1;
                add_box(0, v);
              }
            }
            // gate bits of the second output (backward: dZ of the previous node), one byte per 8 columns
            uint32_t w2[4] = {0xffu, 0xffu, 0xffu, 0xffu};
            if (e.out2 && e.mask2 && r < p.nr) {
#pragma unroll
              for (int g = 0; g < 4; ++g)
                if (g * 8 < nvalid) w2[g] = reinterpret_cast<const uint8_t*>(e.mask2)[mask_byte_addr(rho, n0 + c + g * 8, e.mask2_w, e.mask_rows)];
            }
            // the boxes are free once (a) every lane has read its skip operands and (b) the previous chunk's TMA stores have
            // finished reading them (already waited for by load_adds when there are skip operands)
            if (na == 0 && lane == 0) bulk_wait_read0();
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int off = sw_row + ((j ^ sw_x) << 4);
              if (e.out) store8_h(stg + off, e.out_dtype, v + j * 8);
              if (e.out2) {
                float t2[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) t2[i] = ((w2[j] >> i) & 1u) ? v[j * 8 + i] * e.scale2 : 0.f;
                store8_h(stg + ST_BOX_BYTES + off, e.out2_dtype, t2);
              }
            }
            if (e.mask_out && r < p.nr) {
              uint8_t* mo = reinterpret_cast<uint8_t*>(e.mask_out);
              if (e.mask_w == 32 && ((n0 + c) & 31) == 0) {
                uint32_t word = 0;
#pragma unroll
                for (int g = 0; g < 4; ++g) word |= (g * 8 < nvalid ? m[g] : 0u) << (8 * g);
                *reinterpret_cast<uint32_t*>(mo + mask_byte_addr(rho, n0 + c, 32, e.mask_rows)) = word;
              } else {
#pragma unroll
                for (int g = 0; g < 4; ++g)
                  if (g * 8 < nvalid) mo[mask_byte_addr(rho, n0 + c + g * 8, e.mask_w, e.mask_rows)] = static_cast<uint8_t>(m[g]);
              }
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) {                   // rows >= nr and columns >= N are clipped by the tensor map
              if (e.out) tma_store_3d(&sm.o, stg_u, n0 + c, rbox, b);
              if (e.out2) tma_store_3d(&sm.o2, stg_u + ST_BOX_BYTES, n0 + c, rbox, b);
              bulk_commit();
            }
            load_adds(c + 32 * NSUB);          // next chunk's skip operands (waits for the stores just issued to read the boxes)
          }
        }
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster_relaxed(mapa(tempty_bar(as), 0));
      }
    }
    if (STAGED && lane == 0) bulk_wait0();
  }
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();                  // nobody leaves (or frees TMEM) while the pair's MMAs / multicasts may still touch it
  if (warp == W_MMA) {
    tcgen05_fence_after();
    tmem_dealloc2(tmem_base, 512);
  }
}

// ---------------------------------------------------------------- weight gradient on CTA pairs (MN-major operands)
// dW[m, n] += sum_{b,r} dY[(b,r), m] X[(b,r), n]: frames are the reduction (K) index.  Persistent: ONE wave of CTA pairs walks
// a list of work items (tile, split of the frame range) with TWO TMEM accumulator stages, so the drain of item i overlaps the
// MMAs of item i + 1 and the set-up (barriers, TMEM allocation, cluster sync, pipeline fill) is paid once.  A kernel that pays
// set-up and its ~3 us fp32 `red.global` drain once per (tile, split) CTA pair spends about half of its time there on the
// step's shapes (ncu r2: tensor pipe 43 % busy, 339 CTAs per launch).
//   * tile = 256 output rows (m) x 248 columns (n): the leader CTA feeds N columns 0..127 of the 256-wide MMA, of which
//     0..119 are X columns n0..n0+119 and 120..127 are (for the first column tile, when a bias gradient is wanted) a
//     block of ONES planted by a helper warp, so accumulator column 120 = sum_t dY[t][m] = the bias gradient; the peer CTA feeds
//     columns 128..255 = X columns n0+120..n0+247.  (Without bias those 8 columns duplicate n0+120..n0+127 and are skipped.)
//   * barriers as in the forward kernel: full[] (+ ready[] = "ones planted") and tempty[] in the leader, empty[] / tfull[] in
//     both CTAs by multicast commit; the 4 drain warps of each CTA release a TMEM stage with a relaxed remote arrive.
struct WgArgs3 {
  int nb, nr, M, N;
  int m_pairs, n_tiles, chunks_per_utt, total_units, tiles, span;
  float* dw;
  int64_t ldw;
  float* dbias;
};
constexpr int WG3_TW = 248;                          // X columns per tile
constexpr int WG3_THREADS = 224;                     // 4 drain warps, ones helper, producer, MMA
constexpr int WG3_SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;

__global__ void __launch_bounds__(WG3_THREADS, 1)
gemm_wgrad_persist_kernel(const __grid_constant__ CUtensorMap tmDY, const __grid_constant__ CUtensorMap tmX, const WgArgs3 p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + STAGES * STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto ready_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (3 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (3 * STAGES + 2 + a); };
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(smem_al + STAGES * STAGE_BYTES + 8 * (3 * STAGES + 4));
  // warp roles: 0..3 drain (TMEM lane quadrant = warp), 4 ones helper, 5 producer, 6 MMA issue (highest id: issue priority)
  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair_id = blockIdx.x >> 1;
  if (warp == 5 && lane == 0) {
    prefetch_tmap(&tmDY);
    prefetch_tmap(&tmX);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 2);
      mbar_init(empty_bar(s), 1);
      mbar_init(ready_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 8);       // 4 drain warps x 2 CTAs (used in the leader only)
    }
    fence_barrier_init();
  }
  if (warp == 6) tmem_alloc2(smem_u32(tmem_ptr_smem), 512);
  pdl_launch_dependents();
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();

  // Stream-K: the (tile, frame unit) space is one line of tiles * total_units K blocks, tile-major; pair i owns the contiguous
  // span [i * span, (i + 1) * span) and cuts it at tile boundaries into items (m pair, n tile, unit range).  Every pair does the
  // same number of K blocks (no wave quantisation) and drains ~2 partial tiles instead of one tile per split -- the red.global
  // traffic of a many-way split saturated L2 atomics when every SM drained continuously (r2: 706 vs 817 TFLOP/s).
  const int g_begin = pair_id * p.span, g_end = min(p.tiles * p.total_units, g_begin + p.span);
  const int tile_first = g_begin / p.total_units;
  auto item_geo = [&](int it, int& mp, int& nt, int& u0, int& u1) -> bool {
    const int tile = tile_first + it;
    const int s0 = max(g_begin, tile * p.total_units), s1 = min(g_end, (tile + 1) * p.total_units);
    if (s0 >= s1) return false;
    mp = tile % p.m_pairs;
    nt = tile / p.m_pairs;
    u0 = s0 - tile * p.total_units;
    u1 = s1 - tile * p.total_units;
    return true;
  };

  if (warp == 5) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0;; ++it) {
        int mp, nt, u0, u1;
        if (!item_geo(it, mp, nt, u0, u1)) break;
        const int m0 = mp * 2 * BM + (int)rank * BM;
        const int xc = nt * WG3_TW + (rank ? 120 : 0);
        for (int u = u0; u < u1; ++u) {
          const int b = u / p.chunks_per_utt, r0 = (u % p.chunks_per_utt) * BK;
          mbar_wait(empty_bar(stage), phase ^ 1);
          const uint32_t sa = smem_base + stage * STAGE_BYTES;
          const uint32_t sb = sa + A_STAGE_BYTES;
          const uint32_t fb = mapa(full_bar(stage), 0);
          mbar_expect_tx_cluster(fb, 4 * 64 * 64 * 2);
          tma2_load_3d(sa, &tmDY, fb, m0, r0, b);
          tma2_load_3d(sa + 8192, &tmDY, fb, m0 + 64, r0, b);
          tma2_load_3d(sb, &tmX, fb, xc, r0, b);
          tma2_load_3d(sb + 8192, &tmX, fb, xc + 64, r0, b);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 6) {
    if (rank == 0) {
      // uniform control flow, one elected lane issues (see gemm_tn_pair_kernel)
      const uint32_t idesc = make_idesc(2 * BM, 256, 1, 1);
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0;; ++it) {
        int mp, nt, u0, u1;
        if (!item_geo(it, mp, nt, u0, u1)) break;
        const int as = it & 1;
        mbar_wait(tempty_bar(as), ((it >> 1) & 1) ^ 1);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + as * 256;
        for (int u = u0; u < u1; ++u) {
          // with a bias gradient EVERY stage goes through the helper warp (it arrives on ready[] once per use, after the
          // stage has landed), so that the phases of ready[] stay in lockstep with those of the ring
          mbar_wait(p.dbias != nullptr ? ready_bar(stage) : full_bar(stage), phase);
          tcgen05_fence_after();
          const uint32_t sa = smem_base + stage * STAGE_BYTES;
          const uint64_t ad0 = make_smem_desc(sa, 8192, 1024), bd0 = make_smem_desc(sa + A_STAGE_BYTES, 8192, 1024);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k)
              umma2_bf16(d_tmem, ad0 + (uint64_t)(k * 128), bd0 + (uint64_t)(k * 128), idesc, (u > u0 || k > 0) ? 1u : 0u);
            umma2_commit(empty_bar(stage));
            if (u == u1 - 1) umma2_commit(tfull_bar(as));
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 4) {
    if (rank == 0 && p.dbias != nullptr) {
      // ones block: X columns 120..127 of the leader's half = the last 16-byte chunk of every K row of its second 64-column box
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0;; ++it) {
        int mp, nt, u0, u1;
        if (!item_geo(it, mp, nt, u0, u1)) break;
        for (int u = u0; u < u1; ++u) {
          mbar_wait(full_bar(stage), phase);
          if (nt == 0) {
            uint8_t* xb = smem_al + stage * STAGE_BYTES + A_STAGE_BYTES + 8192;
            for (int r = lane; r < BK; r += 32)
              *reinterpret_cast<uint4*>(xb + r * 128 + ((7 ^ (r & 7)) << 4)) = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
            fence_async_smem();
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(ready_bar(stage));
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    const int q = warp & 3;
    for (int it = 0;; ++it) {
      int mp, nt, u0, u1;
      if (!item_geo(it, mp, nt, u0, u1)) break;
      const bool bias_item = p.dbias != nullptr && nt == 0;
      const int as = it & 1;
      const int m = mp * 2 * BM + (int)rank * BM + q * 32 + lane;
      const int n0 = nt * WG3_TW;
      mbar_wait(tfull_bar(as), (it >> 1) & 1);
      tcgen05_fence_after();
      for (int c = 0; c < 256; c += 32) {
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + as * 256 + c, v);
        if (c == 224) {                       // last chunk is in registers: hand the accumulator stage back before the adds
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster_relaxed(mapa(tempty_bar(as), 0));
        }
        if (m < p.M) {
          // accumulator column j: j < 120 -> X column n0 + j; 120..127 -> ones block (bias) / duplicate; j >= 128 -> n0 + j - 8
          float* row = p.dw + (int64_t)m * p.ldw;
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const int j = c + g * 4;
            if (j >= 120 && j < 128) {
              if (j == 120 && bias_item) atomicAdd(p.dbias + m, v[g * 4]);
              continue;
            }
            const int col = n0 + (j < 120 ? j : j - 8);
            if (col < p.N)
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(row + col), "f"(v[g * 4]), "f"(v[g * 4 + 1]),
                           "f"(v[g * 4 + 2]), "f"(v[g * 4 + 3])
                           : "memory");
          }
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 6) {
    tcgen05_fence_after();
    tmem_dealloc2(tmem_base, 512);
  }
}

// waves x cycles per K block , for the paired tile 256 x BN: four MMAs of max(88, BN/2)
// cycles against 16 KB of A + 64 BN bytes of B ingest per CTA
int pick_bn_pair(int N, int m_tiles, int pairs) {
  int best = 256;
  long best_cost = -1;
  for (int bn = 128; bn <= 256; bn += 32) {
    const long tiles = (long)((m_tiles + 1) / 2) * ((N + bn - 1) / bn);
    const long waves = (tiles + pairs - 1) / pairs;
    const long mma = 4L * std::max(88, bn / 2), ingest = (16384 + 64L * bn) / 64;
    const long cost = waves * std::max(mma, ingest) * 16 + bn / 32;
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = bn; }
  }
  return best;
}

}  // namespace

// persistent pairs: never launch more clusters than can be co-resident (a second wave would double the time)
template <bool STAGED>
static int max_resident_pairs(int smem_bytes, cudaStream_t st) {
  static int cached[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  dev &= 63;
  if (!cached[dev]) {
    const int sms = nbasr_sm_count();
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(STAGED ? ST_THREADS : THREADS);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cfg.gridDim = dim3(sms);
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, gemm_tn_pair_kernel<STAGED>, &cfg) != cudaSuccess || n < 1) n = sms / 2;
    cached[dev] = std::min(n, sms / 2);
    if (nbasr_env_flag(NBASR_ENV_DEBUG))
      fprintf(stderr, "[nbasr] gemm_tn_pair<%d>: %d co-resident CTA pairs on %d SMs\n", (int)STAGED, cached[dev], sms);
  }
  return cached[dev];
}

int sm100_gemm_tn_pair(const nbasr_gemm* g, cudaStream_t st) {
  NBASR_REQUIRE(g->K % 8 == 0, "K must keep 16-byte row alignment");
  Args a{};
  a.nb = g->nb; a.nr = g->nr; a.K = g->K; a.N = g->N;
  a.f16 = g->dtype == NBASR_F16 ? 1 : 0;
  a.l2_prefetch = nbasr_env_gemm_l2pf();
  a.mt_per_utt = (g->nr + BM - 1) / BM;
  a.m_tiles = a.mt_per_utt * g->nb;
  const int sms = nbasr_sm_count();
  a.BN = pick_bn_pair(g->N, a.m_tiles, sms / 2);
  if (nbasr_env_gemm_bn()) a.BN = std::max(64, std::min(256, nbasr_env_gemm_bn() / 32 * 32));   // tuning override (tools/bench_gemm.py)
  a.n_tiles = (g->N + a.BN - 1) / a.BN;
  a.pair_tiles = ((a.m_tiles + 1) / 2) * a.n_tiles;
  a.o_r0 = g->o_r0; a.o_bs = g->o_bs; a.o_rs = g->o_rs;
  a.epi = g->epi;
  CUtensorMap tmA, tmB;
  uint64_t da[3] = {(uint64_t)g->K, (uint64_t)g->nr, (uint64_t)g->nb};
  int64_t sa[3] = {1, g->a_rs, g->a_bs};
  uint32_t ba[3] = {BK, BM, 1};
  if (sm100_get_map(g->a, 3, da, sa, ba, &tmA)) return 1;
  uint64_t db[2] = {(uint64_t)g->K, (uint64_t)g->N};
  int64_t sb[2] = {1, g->ldw};
  uint32_t bb[2] = {BK, (uint32_t)(a.BN / 2)};
  if (sm100_get_map(g->w, 2, db, sb, bb, &tmB)) return 1;

  // Staged (TMA) epilogue: every tensor the epilogue touches row-wise is 16-bit with a 16-byte-aligned pitch.
  const nbasr_epilogue& e = g->epi;
  const int64_t ld = e.ld_out;
  auto h16 = [](int dt) { return dt == NBASR_BF16 || dt == NBASR_F16; };
  auto al16p = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  bool staged = !nbasr_env_flag(NBASR_ENV_GEMM_DIRECT_EPI) && (e.out || e.out2) && !e.accumulate && ld % 8 == 0 &&
                (!e.out || (h16(e.out_dtype) && al16p(e.out))) && (!e.out2 || (h16(e.out2_dtype) && al16p(e.out2))) &&
                (e.n_add == 0 || h16(e.add_dtype)) && g->o_rs >= 1 && g->o_bs >= 0;
  for (int i = 0; i < e.n_add; ++i) staged = staged && al16p(e.add[i]);
  StMaps sm{};
  if (staged) {
    uint64_t dd[3] = {(uint64_t)g->N, (uint64_t)g->nr, (uint64_t)g->nb};
    int64_t sd[3] = {1, g->o_rs * ld, std::max<int64_t>(g->o_bs, 1) * ld};
    uint32_t bx[3] = {32, 32, 1};
    const int64_t off = g->o_r0 * ld * 2;      // bytes: all staged tensors are 16-bit
    auto at = [&](const void* p) { return reinterpret_cast<const char*>(p) + off; };
    const void* any = e.out ? e.out : e.out2;
    if (sm100_get_map(at(e.out ? e.out : any), 3, dd, sd, bx, &sm.o, 2)) return 1;
    if (sm100_get_map(at(e.out2 ? e.out2 : any), 3, dd, sd, bx, &sm.o2, 2)) return 1;
    if (sm100_get_map(at(e.n_add > 0 ? e.add[0] : any), 3, dd, sd, bx, &sm.a0, 2)) return 1;
    if (sm100_get_map(at(e.n_add > 1 ? e.add[1] : any), 3, dd, sd, bx, &sm.a1, 2)) return 1;
    if (sm100_get_map(at(e.n_add > 2 ? e.add[2] : any), 3, dd, sd, bx, &sm.a2, 2)) return 1;
    a.n_add_staged = e.n_add;
  }
  cudaError_t err;
  if (staged) {
    static DevOnce attr;
    if (!attr) {
      cudaError_t e2 = cudaFuncSetAttribute(gemm_tn_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ST_SMEM_BYTES);
      if (e2 != cudaSuccess) return nbasr_fail("gemm_tn_pair<staged> smem attr: %s", cudaGetErrorString(e2));
      attr = true;
    }
    const int npairs = std::max(1, std::min(a.pair_tiles, max_resident_pairs<true>(ST_SMEM_BYTES, st)));
    err = launch_pdl(gemm_tn_pair_kernel<true>, dim3(2 * npairs), dim3(ST_THREADS), (size_t)ST_SMEM_BYTES, st, 2, tmA, tmB, sm, a);
  } else {
    static DevOnce attr;
    if (!attr) {
      cudaError_t e2 = cudaFuncSetAttribute(gemm_tn_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
      if (e2 != cudaSuccess) return nbasr_fail("gemm_tn_pair smem attr: %s", cudaGetErrorString(e2));
      attr = true;
    }
    const int npairs = std::max(1, std::min(a.pair_tiles, max_resident_pairs<false>(SMEM_BYTES, st)));
    err = launch_pdl(gemm_tn_pair_kernel<false>, dim3(2 * npairs), dim3(THREADS), (size_t)SMEM_BYTES, st, 2, tmA, tmB, sm, a);
  }
  if (err != cudaSuccess) return nbasr_fail("gemm_tn_pair launch: %s", cudaGetErrorString(err));
  return 0;
}

int sm100_gemm_wgrad_pair(const nbasr_wgrad* g, cudaStream_t st) {
  NBASR_REQUIRE(g->N % 4 == 0 && g->ldw % 4 == 0, "wgrad N / ldw must be multiples of 4");
  WgArgs3 a{};
  a.nb = g->nb; a.nr = g->nr; a.M = g->M; a.N = g->N;
  a.m_pairs = (g->M + 2 * BM - 1) / (2 * BM);
  a.n_tiles = (g->N + WG3_TW - 1) / WG3_TW;
  a.chunks_per_utt = (g->nr + BK - 1) / BK;
  a.total_units = a.chunks_per_utt * g->nb;
  const int sms = nbasr_sm_count();
  const int slots = std::max(1, sms / 2);
  a.tiles = a.m_pairs * a.n_tiles;
  // one contiguous span of K blocks per pair; a pair should carry >= ~12 K blocks (0.27 us each) per ~3 us drain
  const long total = (long)a.tiles * a.total_units;
  NBASR_REQUIRE(total < (1L << 30), "wgrad problem too large for 32-bit unit indices");
  int npairs = (int)std::max(1L, std::min((long)slots, total / 12));
  a.span = (int)((total + npairs - 1) / npairs);
  npairs = (int)((total + a.span - 1) / a.span);
  a.dw = g->dw; a.ldw = g->ldw; a.dbias = g->dbias;
  CUtensorMap tmDY, tmX;
  uint64_t dd[3] = {(uint64_t)g->M, (uint64_t)g->nr, (uint64_t)g->nb};
  int64_t sd[3] = {1, g->dy_rs, g->dy_bs};
  uint32_t bx[3] = {64, BK, 1};
  if (sm100_get_map(g->dy, 3, dd, sd, bx, &tmDY)) return 1;
  uint64_t dx[3] = {(uint64_t)g->N, (uint64_t)g->nr, (uint64_t)g->nb};
  int64_t sx[3] = {1, g->x_rs, g->x_bs};
  if (sm100_get_map(g->x, 3, dx, sx, bx, &tmX)) return 1;
  static DevOnce attr;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(gemm_wgrad_persist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WG3_SMEM_BYTES);
    if (e != cudaSuccess) return nbasr_fail("gemm_wgrad_persist smem attr: %s", cudaGetErrorString(e));
    attr = true;
  }
  cudaError_t e = launch_pdl(gemm_wgrad_persist_kernel, dim3(2 * npairs), dim3(WG3_THREADS), (size_t)WG3_SMEM_BYTES, st, 2, tmDY, tmX, a);
  if (e != cudaSuccess) return nbasr_fail("gemm_wgrad_persist launch: %s", cudaGetErrorString(e));
  return 0;
}
