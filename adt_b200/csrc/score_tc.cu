// K7 on the 5th-generation tensor cores: bf16 catalog scoring as a TMA-fed tcgen05.mma GEMM with accumulators in
// TMEM and a fused streaming top-K' epilogue; exact fp32 re-score + provable-exactness check behind it.
//
//   warp 0 (1 thread) : TMA producer   - user-feature tile A [128 x H] once, item tiles B [BN x H] in a 2-stage ring
//   warp 1 (1 thread) : MMA issuer     - tcgen05.mma.kind::f16 M=128,N=BN,K=16 into one of two TMEM accumulators
//   warps 2..5        : epilogue       - tcgen05.ld the 128 x BN scores (thread == user row), threshold filter,
//                                        seen-item check, insert into the thread's private top-K' list in smem
//
// Only [splits][U][K'] (score,id) candidates ever reach HBM.  rescore_select_kernel then recomputes the candidates'
// scores in fp32 (same arithmetic as the reference's fp32 matmul), picks the top-K, and flags a user when the bf16
// rounding bound  eps = 2^-7 |f_u| max_i|e_i|  cannot exclude that a non-candidate belongs in the top-K (those users
// are re-run on the exact fp32 kernel by the host, evaluate.py).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/adt_b200.h"
#include "tc.cuh"

using namespace adt;

namespace {

constexpr int BM = 128;
constexpr int TC_THREADS = 192;          // single streaming pass: TMA warp, MMA warp, 4 epilogue warps (thread == user row, lists in smem)
constexpr int TC_THREADS2 = 320;         // two-pass kernels: 8 epilogue warps, two per TMEM lane quarter, each filters half of a tile's columns

struct TcArgs {
  const int* seen_indptr; const int* seen_idx;
  float* part_scores; int* part_ids; float* part_thr;
  unsigned int* gthr;   // [U] best K'-th-best key published by any catalog split of this launch (order-preserving keys, 0 = none)
  const __nv_bfloat16* feats_bf16;   // [U][H] user features (ATM kernels load them straight into tensor memory)
  const float* tau;     // MODE 1: [U] per-user score threshold (from the sample pass): everything above it is a candidate
  int U, n_items, item_offset, KC, n_splits, debug;
  int sstride;          // MODE 2: every sstride-th catalog tile belongs to the sample
  const float* bias;    // BIAS kernels: [n_items] per-item fp32 bias, local index like the catalog rows
};

// Which catalog tiles (BN items each) a CTA walks:
//   MODE 0  streaming top-K' lists over a CONTIGUOUS tile range per split (small catalogs: one pass, thresholds exchanged through gthr)
//   MODE 1  append-only candidate lists against a FIXED per-user threshold tau, tiles interleaved over the splits (tile s, s+S, ...)
//           so that every split sees the same score distribution whatever the id order of the catalog
//   MODE 2  sample pass: streaming top-K' lists over every sstride-th tile (interleaved), from which tau is chosen
template <int MODE>
__device__ __forceinline__ void tc_tile_walk(const TcArgs& a, int BN, int split, int& first, int& step, int& count) {
  const int ntt = (a.n_items + BN - 1) / BN;
  if (MODE == 0) {
    const int tps = (ntt + a.n_splits - 1) / a.n_splits;
    first = split * tps; step = 1;
    count = max(0, min(tps, ntt - first));
  } else if (MODE == 1) {
    first = split; step = a.n_splits;
    count = split < ntt ? (ntt - split + a.n_splits - 1) / a.n_splits : 0;
  } else {
    const int nst = (ntt + a.sstride - 1) / a.sstride;
    first = split * a.sstride; step = a.n_splits * a.sstride;
    count = split < nst ? (nst - split + a.n_splits - 1) / a.n_splits : 0;
  }
}

// first position p in [lo, hi) of the sorted id list with idx[p] >= item
__device__ __forceinline__ int tc_seen_lower_bound(const int* __restrict__ idx, int lo, int hi, int item) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (idx[mid] < item) lo = mid + 1; else hi = mid;
  }
  return lo;
}
// [sb, se): the part of the user's sorted seen list inside this CTA's catalog split, found once per row; usually empty
__device__ __forceinline__ bool tc_is_seen(const TcArgs& a, int sb, int se, int item) {
  if (sb >= se) return false;
  const int p = tc_seen_lower_bound(a.seen_idx, sb, se, item);
  return p < se && a.seen_idx[p] == item;
}

// NS = depth of the TMA ring of catalog tiles (B operand); accumulators are double buffered in TMEM
// MC: the CTA is one of a 2-CTA cluster that walks the SAME catalog tiles for two different user tiles; each CTA fetches half of every
// catalog tile and TMA multicasts it into both CTAs' rings, so every catalog byte leaves L2 once per pair (tmB's box is BN/2 rows then)
// ATM: the user tile (A operand, reused by every MMA of the kernel) lives in TENSOR MEMORY instead of shared memory: the epilogue
// threads store their own feature row with tcgen05.st once, the MMAs read it from TMEM (tcgen05.mma, A from TMEM).  Frees
// KB*16 KB of shared memory for a deeper TMA ring and takes the A fragment reads off the shared-memory port.
// KB > 4 (H = 320 .. 512): a full-K catalog tile (KB*BN*128 B, 128 KB at H = 512) no longer fits two ring stages beside the lists, so
// the ring holds ONE 64-column K block of a catalog tile per stage and the MMA warp consumes KB stages per tile; the user tile always
// sits in tensor memory there (KB*32 <= 256 columns beside two 128-column accumulators).  KB <= 4 keeps the full-K stages.
// BIAS: score = accumulator + bias[item] in fp32, added to every value as it leaves tcgen05.ld and before any comparison, in all three
// modes (so the streaming lists, the published gthr keys, tau and the appended candidates are all in biased scores).  Every epilogue
// warp stages the bias of its columns once per tile in its own smem row (loaded from global one tile ahead); each 32-column chunk
// then reads it back with 8 broadcast LDS.128.  BIAS = false leaves the kernel exactly as without the feature.
template <int KB, int BN, int NS, int MODE, bool MC, bool ATM, bool BIAS>
__global__ void __launch_bounds__(TC_THREADS2, 1) score_tc_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                  const __grid_constant__ CUtensorMap tmB, TcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  constexpr bool KBLK = KB > 4;
  static_assert(!KBLK || ATM, "the K-blocked ring takes the user tile from tensor memory");
  constexpr int A_BYTES = ATM ? 0 : KB * BM * 128;
  // accumulator ring in tensor memory: MMA(t + NACC - 1) may be issued while tile t is still being read out.  The per-tile chain
  // (commit -> barrier -> tcgen05.ld -> filter -> arrive -> next MMA) costs ~2k cycles against ~130 of MMA at H = 64, so the depth of
  // this ring, not the tensor pipe, sets the tile rate: three buffers when they fit beside the A tile (BN 128: 384 + KB*32 <= 512)
  constexpr int NACC = (3 * BN + (ATM ? KB * 32 : 0) <= 512) ? 3 : 2;
  constexpr int TM_COLS = (ATM || NACC * BN > 256) ? 512 : (NACC * BN > 128 ? 256 : 128);   // accumulators NACC x BN (+ KB*32 columns of A behind them)
  constexpr uint32_t A_COL = NACC * BN;
  constexpr int B_STAGE = KBLK ? BN * 128 : KB * BN * 128;
  uint8_t* sA = smem;
  uint8_t* sB = sA + A_BYTES;
  const int KCP = MODE == 0 ? (a.KC <= 32 ? 32 : 64) : 0;     // list slots reserved per user row (the two-pass modes keep no lists on chip)
  uint32_t* lk = reinterpret_cast<uint32_t*>(sB + NS * B_STAGE);  // [KCP][128] order-preserving score keys, slot-major: the
  int* li = reinterpret_cast<int*>(lk + BM * KCP);                // [KCP][128] item ids      thread that owns a row scans it conflict-free
  float* thr_s = reinterpret_cast<float*>(li + BM * KCP);         // [128] (unused scratch)
  float* vsm = thr_s + BM;                                        // [4][32][32] chunk parking area of the epilogue warps
  float* bsm = vsm + 4 * 1024;                                    // BIAS: [8][64] or [4][128] per-warp bias of the current tile
  uint64_t* bars = reinterpret_cast<uint64_t*>(bsm + (BIAS ? 512 : 0));
  uint64_t* full = bars;               // [NS] B stage filled (TMA tx)
  uint64_t* empty = bars + NS;         // [NS] B stage consumed (tcgen05.commit)
  uint64_t* tfull = bars + 2 * NS;     // [NACC] accumulator ready (tcgen05.commit)
  uint64_t* tempty = bars + 2 * NS + NACC;  // [NACC] accumulator drained (epilogue warps)
  uint64_t* abar = bars + 2 * NS + 2 * NACC;  // A tile landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NS + 2 * NACC + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int split = MC ? blockIdx.y : blockIdx.x, u0 = (MC ? blockIdx.x : blockIdx.y) * BM;
  const uint32_t crank = MC ? tc::cluster_ctarank() : 0u;
  int tfirst, tstep, ntiles;
  tc_tile_walk<MODE>(a, BN, split, tfirst, tstep, ntiles);
  const int it0 = min(a.n_items, tfirst * BN), it1 = min(a.n_items, (tfirst + (ntiles > 0 ? (ntiles - 1) * tstep + 1 : 0)) * BN);   // item span touched

  if (threadIdx.x == 0) {
    tc::tma_prefetch_desc(&tmA);
    tc::tma_prefetch_desc(&tmB);
    for (int i = 0; i < NS; ++i) {
      tc::mbar_init(full + i, 1);
      tc::mbar_init(empty + i, MC ? 2 : 1);      // multicast ring: both CTAs of the pair must have consumed a stage
    }
    for (int i = 0; i < NACC; ++i) {
      tc::mbar_init(tfull + i, 1);
      tc::mbar_init(tempty + i, MODE == 0 ? 4 : 8);
    }
    tc::mbar_init(abar, ATM ? 4 : 1);            // A in TMEM: one arrival per epilogue warp after its tcgen05.st completed
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc<TM_COLS>(tmem_slot);
  tc::tc_fence_before();
  __syncthreads();
  if (MC) tc::cluster_sync();                    // the peer's barriers exist before anything is multicast into this CTA
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      if (!ATM) {
        tc::mbar_arrive_expect_tx(abar, A_BYTES);
        for (int kb = 0; kb < KB; ++kb) tc::tma_load_2d(sA + kb * BM * 128, &tmA, kb * 64, u0, abar);
      }
      if constexpr (KBLK) {
        for (int t = 0; t < ntiles; ++t)
          for (int kb = 0; kb < KB; ++kb) {
            const int g = t * KB + kb, st = g % NS;
            tc::mbar_wait(empty + st, ((g / NS) & 1) ^ 1);
            tc::mbar_arrive_expect_tx(full + st, B_STAGE);
            if (MC)
              tc::tma_load_2d_mc(sB + st * B_STAGE + crank * (BN / 2) * 128, &tmB, kb * 64, (tfirst + t * tstep) * BN + (int)crank * (BN / 2),
                                 full + st, (uint16_t)3);
            else
              tc::tma_load_2d(sB + st * B_STAGE, &tmB, kb * 64, (tfirst + t * tstep) * BN, full + st);
          }
      } else
      for (int t = 0; t < ntiles; ++t) {
        const int st = t % NS;
        tc::mbar_wait(empty + st, ((t / NS) & 1) ^ 1);
        tc::mbar_arrive_expect_tx(full + st, B_STAGE);
        if (MC) {
          for (int kb = 0; kb < KB; ++kb)
            tc::tma_load_2d_mc(sB + st * B_STAGE + kb * BN * 128 + crank * (BN / 2) * 128, &tmB, kb * 64,
                               (tfirst + t * tstep) * BN + (int)crank * (BN / 2), full + st, (uint16_t)3);
        } else {
          for (int kb = 0; kb < KB; ++kb) tc::tma_load_2d(sB + st * B_STAGE + kb * BN * 128, &tmB, kb * 64, (tfirst + t * tstep) * BN, full + st);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = tc::idesc_bf16_f32(BM, BN);
      tc::mbar_wait(abar, 0);
      for (int t = 0; t < ntiles; ++t) {
        const int st = t % NS, acc = t % NACC;
        tc::mbar_wait(tempty + acc, ((t / NACC) & 1) ^ 1);
        if constexpr (KBLK) {
          const uint32_t d_tmem = tmem_base + acc * BN;
          for (int kb = 0; kb < KB; ++kb) {
            const int g = t * KB + kb, gs = g % NS;
            tc::mbar_wait(full + gs, (g / NS) & 1);
            tc::tc_fence_after();
            const uint64_t bd = tc::smem_desc_k_sw128(tc::smem_u32(sB + gs * B_STAGE));
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4)
              tc::mma_bf16_ts(d_tmem, tmem_base + A_COL + kb * 32 + k4 * 8, bd + (uint64_t)(k4 * 2), idesc, (kb | k4) != 0);
            if (MC) tc::mma_commit_mc(empty + gs, (uint16_t)3); else tc::mma_commit(empty + gs);
          }
          tc::mma_commit(tfull + acc);
          continue;
        }
        tc::mbar_wait(full + st, (t / NS) & 1);
        tc::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
#pragma unroll
        for (int kb = 0; kb < KB; ++kb) {
          const uint64_t bd = tc::smem_desc_k_sw128(tc::smem_u32(sB + st * B_STAGE + kb * BN * 128));
          if (ATM) {
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4)   // K = 16 per MMA = 8 TMEM columns of A
              tc::mma_bf16_ts(d_tmem, tmem_base + A_COL + kb * 32 + k4 * 8, bd + (uint64_t)(k4 * 2), idesc, (kb | k4) != 0);
          } else {
            const uint64_t ad = tc::smem_desc_k_sw128(tc::smem_u32(sA + kb * BM * 128));
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4)   // 4 x K=16 per 64-wide swizzle atom: +32 bytes on the start address
              tc::mma_bf16_ss(d_tmem, ad + (uint64_t)(k4 * 2), bd + (uint64_t)(k4 * 2), idesc, (kb | k4) != 0);
          }
        }
        if (MC) tc::mma_commit_mc(empty + st, (uint16_t)3); else tc::mma_commit(empty + st);
        tc::mma_commit(tfull + acc);
      }
    }
  } else {
    // epilogue: thread == user row, for the threshold filter AND for the maintenance of that row's candidate list: every lane
    // inserts its own candidates into its own slot-major list (no cross-lane traffic, all 32 rows of a warp progress in parallel)
    const int q = warp & 3;                  // TMEM lane quarter this warp may access (hardware: warp id % 4)
    const int half = (warp - 2) >> 2;        // two-pass kernels: which half of a tile's columns this warp filters (0 in the single pass)
    const int row = 32 * q + lane;
    const int u = u0 + row;
    const int KC = MODE == 0 ? a.KC : a.KC / 2;      // two-pass: every (row, column half) owns KC/2 candidate slots = one virtual split
    const int CB = MODE == 0 ? 0 : half * (BN / 2), CE = MODE == 0 ? BN : CB + BN / 2;
    constexpr int CW = 32;      // columns per tcgen05.ld (64-column loads were measured 2x SLOWER: 0.38 -> 0.82 ms at 512 x 1M x 256)
    if (ATM && half == 0) {     // this thread's feature row (bf16, KB*32 words) -> TMEM columns A_COL.. of its lane
      const uint4* frow = reinterpret_cast<const uint4*>(a.feats_bf16 + (long long)(u < a.U ? u : 0) * (KB * 64));
#pragma unroll 1
      for (int i = 0; i < KB; ++i) {
        uint32_t r[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint4 x = u < a.U ? __ldg(frow + i * 8 + j) : make_uint4(0u, 0u, 0u, 0u);
          r[4 * j] = x.x; r[4 * j + 1] = x.y; r[4 * j + 2] = x.z; r[4 * j + 3] = x.w;
        }
        tc::tmem_st32(tmem_base + ((uint32_t)(32 * q) << 16) + A_COL + 32 * i, r);
      }
      tc::tmem_st_wait();
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(abar);
    }
    if (MODE == 0) {
      for (int k = 0; k < KC; ++k) {
        lk[k * BM + row] = 0u;               // key 0 = "worse than anything"
        li[k * BM + row] = -1;
      }
    }
    int sb = 0, se = 0;                      // this row's seen ids inside the item span this CTA touches
    if (a.seen_indptr && u < a.U) {
      const int hi = a.seen_indptr[u + 1];
      sb = tc_seen_lower_bound(a.seen_idx, a.seen_indptr[u], hi, a.item_offset + it0);
      se = tc_seen_lower_bound(a.seen_idx, sb, hi, a.item_offset + it1);
    }
    // per-tile bias staging (BIAS only): this warp's BW columns of tile t sit in bs[]; the next tile's are already in registers
    constexpr int BW = MODE == 0 ? BN : BN / 2;
    float bnext[BIAS ? BW / 32 : 1];
    auto bias_fetch = [&](int t) {           // global -> registers, one tile ahead of its use (hides the load latency)
      if constexpr (BIAS) {
        const int ib = (tfirst + t * tstep) * BN + CB + lane;
#pragma unroll
        for (int j = 0; j < BW / 32; ++j) bnext[j] = (t < ntiles && ib + 32 * j < a.n_items) ? __ldg(a.bias + ib + 32 * j) : 0.f;
      }
    };
    auto bias_stage = [&](int t) {           // registers -> this warp's smem row, then fetch the next tile's
      if constexpr (BIAS) {
        float* bs = bsm + (warp - 2) * BW;
        __syncwarp();
#pragma unroll
        for (int j = 0; j < BW / 32; ++j) bs[lane + 32 * j] = bnext[j];
        __syncwarp();
        bias_fetch(t + 1);
      }
    };
    auto bias_add = [&](float (&v)[32], int c0) {   // v[c] += bias of column c0 + c (same value in every lane: broadcast loads)
      if constexpr (BIAS) {
        const float4* b4 = reinterpret_cast<const float4*>(bsm + (warp - 2) * BW + (c0 - CB));
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 b = b4[j];
          v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
        }
      }
    };
    bias_fetch(0);
    auto unkey = [](uint32_t k) -> float { return k == 0u ? -INFINITY : __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); };
    auto fkey = [](float f) -> uint32_t {
      const uint32_t b = __float_as_uint(f);
      return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
    };
    float thr;
    if constexpr (MODE == 1) {
      // ---- fixed threshold, append only: no list maintenance in the hot loop at all
      thr = u < a.U ? a.tau[u] : INFINITY;
      int cnt = 0;
      bool overflow = false;
      const long long vsplit = (long long)split * 2 + half;
      const long long obase = (vsplit * a.U + (u < a.U ? u : 0)) * KC;
      for (int t = 0; t < ntiles; ++t) {
        const int st = t % NACC;
        bias_stage(t);
        tc::mbar_wait(tfull + st, (t / NACC) & 1);
        tc::tc_fence_after();
        const int tb = (tfirst + t * tstep) * BN;
#pragma unroll 1
        for (int c0 = CB; c0 < CE; c0 += CW) {
          float v[CW];
          tc::tmem_ldw<CW>(tmem_base + ((uint32_t)(32 * q) << 16) + st * BN + c0, v);
          if (c0 + CW == CE) {               // accumulator fully read: hand it back to the MMA warp
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(tempty + st);
          }
          bias_add(v, c0);
          const int ib = tb + c0;
          const int nvalid = a.n_items - ib;
          if (nvalid < CW) {
#pragma unroll
            for (int c = 0; c < CW; ++c)
              if (c >= nvalid) v[c] = -INFINITY;
          }
          if (a.debug == 1) continue;
          float mx = v[0];
#pragma unroll
          for (int c = 1; c < CW; ++c) mx = fmaxf(mx, v[c]);
          if (a.debug == 2) continue;
          if (mx > thr) {                    // rare (about one row in 75 per chunk): walk the registers, no staging through smem
#pragma unroll
            for (int c = 0; c < CW; ++c) {
              if (v[c] > thr) {
                const int item = a.item_offset + ib + c;
                if (!tc_is_seen(a, sb, se, item)) {       // candidates go straight to HBM, no list on chip
                  if (cnt < KC) { a.part_scores[obase + cnt] = v[c]; a.part_ids[obase + cnt] = item; ++cnt; }
                  else overflow = true;
                }
              }
            }
          }
        }
      }
      if (overflow) thr = INFINITY;          // candidates were dropped: the caller must re-run this user exactly
      if (u < a.U) {
        for (int k = cnt; k < KC; ++k) { a.part_scores[obase + k] = -INFINITY; a.part_ids[obase + k] = -1; }
        a.part_thr[vsplit * a.U + u] = thr;
      }
    } else if constexpr (MODE == 2) {
      // ---- sample pass: only the maximum of every sampled tile is kept, [sample tile][user] in part_scores (tau_select_kernel picks the
      // R-th largest of them): no lists, no shared memory, one store per (row, tile)
      thr = 0.f;
      for (int t = 0; t < ntiles; ++t) {
        const int st = t % NACC;
        bias_stage(t);
        tc::mbar_wait(tfull + st, (t / NACC) & 1);
        tc::tc_fence_after();
        const int tb = (tfirst + t * tstep) * BN;
        float mx = -INFINITY;
#pragma unroll 1
        for (int c0 = CB; c0 < CE; c0 += CW) {
          float v[CW];
          tc::tmem_ldw<CW>(tmem_base + ((uint32_t)(32 * q) << 16) + st * BN + c0, v);
          if (c0 + CW == CE) {
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(tempty + st);
          }
          bias_add(v, c0);
          const int nvalid = a.n_items - (tb + c0);
#pragma unroll
          for (int c = 0; c < CW; ++c) mx = fmaxf(mx, c < nvalid ? v[c] : -INFINITY);
        }
        if (u < a.U) a.part_scores[((long long)(split + t * a.n_splits) * 2 + half) * a.U + u] = mx;
      }
    } else {
    uint32_t mink = 0u;                      // smallest key in the list and its slot
    int minpos = 0;
    // rej: keys <= rej cannot be among the K' best of the WHOLE catalog: max of this split's K'-th best (mink) and the best
    // K'-th best any other split has published so far (K' items of one split beat it, so the global K'-th best does too)
    uint32_t rej = 0u, published = 0u;
    thr = u < a.U ? -INFINITY : INFINITY;    // rej as a float (-inf while nothing is known)
    auto insert = [&](float sc, int itl) {
      const uint32_t key = fkey(sc);
      if (key <= rej) return;
      const int item = a.item_offset + itl;
      if (MODE == 0 && tc_is_seen(a, sb, se, item)) return;    // the sample pass only needs score quantiles: seen items may stay
      lk[minpos * BM + row] = key;
      li[minpos * BM + row] = item;
      uint32_t nm = 0xffffffffu;
      int np = 0;
      for (int k = 0; k < KC; ++k) {
        const uint32_t x = lk[k * BM + row];
        if (x < nm) { nm = x; np = k; }
      }
      mink = nm; minpos = np;
      if (nm > rej) { rej = nm; thr = unkey(nm); }
    };
    for (int t = 0; t < ntiles; ++t) {
      const int st = t % NACC;
      // thresholds of the other splits: issue the (L2) load now, consume it after this tile
      const uint32_t gnext = (MODE == 0 && a.gthr && u < a.U) ? __ldcg(a.gthr + u) : 0u;
      bias_stage(t);
      tc::mbar_wait(tfull + st, (t / NACC) & 1);
      tc::tc_fence_after();
      const int tb = (tfirst + t * tstep) * BN;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        float v[32];
        tc::tmem_ld32(tmem_base + ((uint32_t)(32 * q) << 16) + st * BN + c0, v);
        if (c0 + 32 == BN) {               // accumulator fully read: hand it back to the MMA warp
          tc::tc_fence_before();
          __syncwarp();
          if (lane == 0) tc::mbar_arrive(tempty + st);
        }
        bias_add(v, c0);
        const int ib = tb + c0;
        const int nvalid = a.n_items - ib;
        if (nvalid < 32) {
#pragma unroll
          for (int c = 0; c < 32; ++c)
            if (c >= nvalid) v[c] = -INFINITY;
        }
        if (a.debug == 1) continue;      // pipeline-only timing experiment
        unsigned m = 0u;                    // bit c set <=> this row's score in column c beats the row threshold
#pragma unroll
        for (int c = 0; c < 32; ++c) m |= (v[c] > thr) ? (1u << c) : 0u;
        unsigned bb = __ballot_sync(0xffffffffu, m != 0u);
        if (bb == 0u || a.debug == 2) continue;   // common case once the lists are warm
        // park the 32x32 chunk in smem (lane-contiguous, conflict free); every lane then walks ITS OWN fired columns with one
        // copy of the insert code
        float* vs = vsm + q * 1024;
#pragma unroll
        for (int c = 0; c < 32; ++c) vs[c * 32 + lane] = v[c];
        __syncwarp();
        while (m) {
          const int c = __ffs(m) - 1;
          m &= m - 1;
          insert(vs[c * 32 + lane], ib + c);
        }
        __syncwarp();
      }
      if (MODE == 0 && a.gthr && u < a.U) {
        if (mink > published) { atomicMax(a.gthr + u, mink); published = mink; }   // rare once the list is warm
        if (gnext > rej) { rej = gnext; thr = unkey(gnext); }
      }
    }
    }
    if (MODE == 0 && u < a.U) {
      const long long o = ((long long)split * a.U + u) * KC;
      for (int k = 0; k < KC; ++k) {
        const uint32_t key = lk[k * BM + row];
        const int id = li[k * BM + row];
        a.part_scores[o + k] = id >= 0 ? __uint_as_float((key & 0x80000000u) ? (key & 0x7fffffffu) : ~key) : -INFINITY;
        a.part_ids[o + k] = id;
      }
      a.part_thr[(long long)split * a.U + u] = thr;
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (MC) tc::cluster_sync();                    // nobody leaves while the peer may still multicast into / arrive on this CTA
  if (warp == 1) tc::tmem_dealloc<TM_COLS>(tmem_base);
}

// fp32 -> bf16 rows (round to nearest even) + max squared row norm (atomicMax on the float bits; values >= 0)
__global__ void __launch_bounds__(256) to_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, long long rows, int H,
                                                      float* __restrict__ max_normsq) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  for (long long r = (long long)blockIdx.x * 8 + w; r < rows; r += (long long)gridDim.x * 8) {
    float ns = 0.f;
    for (int c = 2 * l; c < H; c += 64) {
      const float2 v = *reinterpret_cast<const float2*>(x + r * H + c);
      ns = fmaf(v.x, v.x, fmaf(v.y, v.y, ns));
      *reinterpret_cast<__nv_bfloat162*>(y + r * H + c) = __floats2bfloat162_rn(v.x, v.y);
    }
    if (max_normsq) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) ns += __shfl_xor_sync(0xffffffffu, ns, o);
      if (l == 0) atomicMax(reinterpret_cast<unsigned int*>(max_normsq), __float_as_uint(ns));
    }
  }
}

struct RescoreArgs {
  const float* feats; const float* E; const float* part_scores; const int* part_ids; const float* part_thr; const float* max_normsq;
  float* out_scores; int* out_ids; int* flags;
  const int* answers; double* metric_acc;
  int U, H, item_offset, K, KC, n_splits;
  const float* bias; const float* max_abs_bias;   // BIAS: [n_items] per-item bias (local index) and max |bias|
};

constexpr int RS_MAXC = 2048;   // candidate slots per user (n_splits * KC)
constexpr int RS_NT = 256;
constexpr int RS_STAGES = 2, RS_CW = 32, RS_LD = RS_CW + 4;   // re-score ring: stages per warp, columns per stage, floats per staged row (+4: conflict-free float4 reads)
// dynamic shared memory of the re-score kernel for rows of up to HMAX floats: the user vector, then the per-warp rings
constexpr size_t rs_smem(int HMAX) { return (HMAX + (size_t)(RS_NT / 32) * RS_STAGES * 32 * RS_LD) * sizeof(float); }

// One CTA per user: (1) compact the valid candidates of all splits, (2) one THREAD per candidate (rows staged through a per-warp cp.async ring) recomputes its score in fp32 with
// the same sequential fmaf order as the exact kernel (bit-identical scores, so the two paths can be mixed and compared), 16 row
// loads in flight per thread, (3) rank counting under the total order (score desc, id asc) places the K best, (4) the exactness flag
// and the fused get_full_sort_score sums.
// sortable key of a candidate: larger key = better under (score desc, id asc); -0.0 is folded into +0.0 so that equal floats give equal keys
__device__ __forceinline__ unsigned long long rs_key(float s, int id) {
  const unsigned u = __float_as_uint(s + 0.f);
  const unsigned o = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)o << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)id);
}

template <bool BIAS, int HMAX>
__global__ void __launch_bounds__(RS_NT, 2) rescore_select_kernel(RescoreArgs a) {
  __shared__ int cid[RS_MAXC];
  __shared__ float csc[RS_MAXC];
  __shared__ __align__(16) unsigned long long ckey[RS_MAXC];
  __shared__ int cnt_s, first_s;
  __shared__ float red[RS_NT / 32];
  __shared__ float kth_s;
  const int u = blockIdx.x, tid = threadIdx.x, w = tid >> 5, l = tid & 31;
  const int n = a.n_splits * a.KC;
  if (tid == 0) { cnt_s = 0; first_s = -1; kth_s = -INFINITY; }
  const float* f = a.feats + (long long)u * a.H;
  float fn = 0.f;
  for (int c = tid; c < a.H; c += RS_NT) fn = fmaf(f[c], f[c], fn);
  float thr_max = -INFINITY;
  for (int s = tid; s < a.n_splits; s += RS_NT) thr_max = fmaxf(thr_max, a.part_thr[(long long)s * a.U + u]);
  __syncthreads();
  for (int c = tid; c < n; c += RS_NT) {
    const int sp = c / a.KC, k = c - sp * a.KC;
    const int id = a.part_ids[((long long)sp * a.U + u) * a.KC + k];
    if (id >= 0) cid[atomicAdd(&cnt_s, 1)] = id;
  }
  // |f|^2 and max threshold over the CTA
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { fn += __shfl_xor_sync(0xffffffffu, fn, o); thr_max = fmaxf(thr_max, __shfl_xor_sync(0xffffffffu, thr_max, o)); }
  __shared__ float fn_s[RS_NT / 32], tm_s[RS_NT / 32];
  if (l == 0) { fn_s[w] = fn; tm_s[w] = thr_max; }
  __syncthreads();
  const int m = cnt_s;
  fn = 0.f; thr_max = -INFINITY;
  for (int i = 0; i < RS_NT / 32; ++i) { fn += fn_s[i]; thr_max = fmaxf(thr_max, tm_s[i]); }
  // fp32 re-score.  Thread c owns candidate c and keeps the exact kernel's sequential fmaf chain; the rows reach it through a per-warp
  // cp.async ring (32 rows x RS_CW columns per stage, 16-byte pieces, consecutive lanes per row: every 128-byte row segment is one
  // coalesced request and a whole stage is in flight at once -- a thread reading its own 1 KB row directly serialises on DRAM latency).
  {
    extern __shared__ __align__(16) float rs_dyn[];
    float* fs = rs_dyn;                                           // [H] user vector
    float* ring = rs_dyn + HMAX + w * (RS_STAGES * 32 * RS_LD);   // this warp's stages
    for (int c = tid; c < a.H; c += RS_NT) fs[c] = f[c];
    __syncthreads();
    const int nch = a.H / RS_CW;
    for (int base = 0; base < m; base += RS_NT) {
      const int wbase = base + 32 * w;
      if (wbase >= m) break;                                      // warp-uniform
      const int total = nch;
      auto issue = [&](int ch) {
        float* st = ring + (ch % RS_STAGES) * (32 * RS_LD);
#pragma unroll
        for (int i = 0; i < RS_CW / 4; ++i) {
          const int idx = i * 32 + l, row = idx / (RS_CW / 4), seg = idx % (RS_CW / 4);
          const int c = wbase + row;
          const bool ok = c < m;
          const float* src = a.E + (long long)((ok ? cid[c] : cid[wbase]) - a.item_offset) * a.H + ch * RS_CW + seg * 4;
          const uint32_t dst = (uint32_t)__cvta_generic_to_shared(st + row * RS_LD + seg * 4);
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(ok ? 16 : 0));
        }
        asm volatile("cp.async.commit_group;");
      };
      for (int ch = 0; ch < RS_STAGES - 1; ++ch) {
        if (ch < total) issue(ch); else asm volatile("cp.async.commit_group;");
      }
      float acc = 0.f;
      for (int ch = 0; ch < total; ++ch) {
        if (ch + RS_STAGES - 1 < total) issue(ch + RS_STAGES - 1); else asm volatile("cp.async.commit_group;");
        asm volatile("cp.async.wait_group %0;" ::"n"(RS_STAGES - 1));
        __syncwarp();
        const float* st = ring + (ch % RS_STAGES) * (32 * RS_LD) + l * RS_LD;
        const float* fv0 = fs + ch * RS_CW;
#pragma unroll
        for (int j = 0; j < RS_CW / 4; ++j) {
          const float4 ev = *reinterpret_cast<const float4*>(st + 4 * j);
          const float4 fv = *reinterpret_cast<const float4*>(fv0 + 4 * j);
          acc = fmaf(fv.x, ev.x, acc); acc = fmaf(fv.y, ev.y, acc); acc = fmaf(fv.z, ev.z, acc); acc = fmaf(fv.w, ev.w, acc);
        }
        __syncwarp();
      }
      if (wbase + l < m) {
        if constexpr (BIAS) acc += a.bias[cid[wbase + l] - a.item_offset];   // after the whole chain, as in the exact kernel: bit-identical
        csc[wbase + l] = acc; ckey[wbase + l] = rs_key(acc, cid[wbase + l]);
      }
    }
  }
  __syncthreads();
  const int answer = a.answers ? a.answers[u] : -1;
  for (int c = tid; c < m; c += RS_NT) {
    const float s = csc[c];
    const int id = cid[c];
    const unsigned long long key = ckey[c];
    int rank = 0;
    int j = 0;
    for (; j + 4 <= m; j += 4) {                 // branch-free: one 64-bit compare per rival under the total order (score desc, id asc)
      const ulonglong2 k01 = *reinterpret_cast<const ulonglong2*>(ckey + j), k23 = *reinterpret_cast<const ulonglong2*>(ckey + j + 2);
      rank += (k01.x > key) + (k01.y > key) + (k23.x > key) + (k23.y > key);
    }
    for (; j < m; ++j) rank += ckey[j] > key;
    if (rank < a.K) {
      a.out_scores[(long long)u * a.K + rank] = s;
      a.out_ids[(long long)u * a.K + rank] = id;
      if (id == answer) first_s = rank;
      if (rank == a.K - 1) kth_s = s;
    }
  }
  for (int k = m + tid; k < a.K; k += RS_NT) {          // fewer than K candidates: pad (the user is flagged below)
    a.out_scores[(long long)u * a.K + k] = -INFINITY;
    a.out_ids[(long long)u * a.K + k] = -1;
  }
  __syncthreads();
  if (tid == 0) {
    const float kth = m >= a.K ? kth_s : -INFINITY;
    // a non-candidate's exact score exceeds tau by at most eps: the bf16 operand rounding 2^-7 |f| max|e|, plus with a bias the
    // rounding of the two fp32 bias additions (epilogue and re-score), each <= 2^-24 |<f,e> + b| <= 2^-24 (|f| max|e| + max|b|);
    // 2^-22 leaves a factor 2 of margin.  A bias that dwarfs the dot products therefore widens eps until the user is flagged and
    // re-run exactly, rather than returning a list the bound cannot prove.
    float eps = 0.0078125f * sqrtf(fn) * sqrtf(*a.max_normsq);        // 2^-7 |f| max|e|
    if constexpr (BIAS) eps += 2.384185791015625e-07f * (sqrtf(fn) * sqrtf(*a.max_normsq) + *a.max_abs_bias);
    const int flag = (thr_max > -INFINITY && !(kth > thr_max + eps)) ? 1 : 0;
    a.flags[u] = flag;
    // fused get_full_sort_score epilogue (sasrec/utils.py:686-708) for the users whose list is proven exact
    if (!flag && a.answers && a.metric_acc) {
      const int first = first_s;
      atomicAdd(a.metric_acc + 5, 1.0);
      if (first >= 0) {
        const double g = 1.0 / log2((double)first + 2.0);
        if (first < 5) { atomicAdd(a.metric_acc + 0, 1.0); atomicAdd(a.metric_acc + 1, g); }
        if (first < 10) { atomicAdd(a.metric_acc + 2, 1.0); atomicAdd(a.metric_acc + 3, g); }
        atomicAdd(a.metric_acc + 4, 1.0 / ((double)first + 1.0));
      }
    }
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D bf16 row-major [rows][H] tensor, box = [box_rows][64 cols], 128-byte swizzle
int make_map(CUtensorMap* m, const void* base, long long rows, int H, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return ADT_E_CUDA;
  cuuint64_t gdim[2] = {(cuuint64_t)H, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)H * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? ADT_OK : ADT_E_CUDA;
}

static bool tc_atmem() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("ADT_TC_ATMEM"); v = e ? atoi(e) : 1; }
  return v != 0;
}
template <int KB, int BN, int NS, int MODE, bool ATM, bool BIAS>
int launch_tc_ns(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap* tmBh, const TcArgs& k, dim3 grid, cudaStream_t s, size_t smem) {
  if (tmBh) {      // 2-CTA clusters over pairs of user tiles, grid = (user tiles, splits)
    if (MODE == 0) return ADT_E_SHAPE;
    cudaFuncSetAttribute(score_tc_kernel<KB, BN, NS, MODE, true, ATM, BIAS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid.y, grid.x); cfg.blockDim = dim3(MODE == 0 ? TC_THREADS : TC_THREADS2); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, score_tc_kernel<KB, BN, NS, MODE, true, ATM, BIAS>, tmA, *tmBh, k) == cudaSuccess ? ADT_OK : ADT_E_CUDA;
  }
  cudaFuncSetAttribute(score_tc_kernel<KB, BN, NS, MODE, false, ATM, BIAS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  score_tc_kernel<KB, BN, NS, MODE, false, ATM, BIAS><<<grid, MODE == 0 ? TC_THREADS : TC_THREADS2, smem, s>>>(tmA, tmB, k);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}
// deepest catalog-tile ring (2..4 stages) that fits the 227 KB of shared memory next to the user tile and the top-K lists
template <int KB, int BN, int MODE, bool ATM, bool BIAS>
int launch_tc_a(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap* tmBh, const TcArgs& k, dim3 grid, cudaStream_t s) {
  const size_t fixed = 1024 + (ATM ? 0 : (size_t)KB * BM * 128) + (MODE == 0 ? (size_t)(k.KC <= 32 ? 32 : 64) * BM * 8 : 0) + BM * 4 + 4 * 1024 * 4 + 256 +
                       (BIAS ? 512 * 4 : 0);
  const size_t stage = (size_t)KB * BN * 128, cap = 227 * 1024;
  // the ring must hold more than one DRAM round trip (~1 us) of tensor work: a [128 x 128 x 64] tile is only 256 cycles
  if (fixed + 8 * stage <= cap) return launch_tc_ns<KB, BN, 8, MODE, ATM, BIAS>(tmA, tmB, tmBh, k, grid, s, fixed + 8 * stage);
  if (fixed + 6 * stage <= cap) return launch_tc_ns<KB, BN, 6, MODE, ATM, BIAS>(tmA, tmB, tmBh, k, grid, s, fixed + 6 * stage);
  if (fixed + 4 * stage <= cap) return launch_tc_ns<KB, BN, 4, MODE, ATM, BIAS>(tmA, tmB, tmBh, k, grid, s, fixed + 4 * stage);
  if (fixed + 3 * stage <= cap) return launch_tc_ns<KB, BN, 3, MODE, ATM, BIAS>(tmA, tmB, tmBh, k, grid, s, fixed + 3 * stage);
  if (fixed + 2 * stage <= cap) return launch_tc_ns<KB, BN, 2, MODE, ATM, BIAS>(tmA, tmB, tmBh, k, grid, s, fixed + 2 * stage);
  return ADT_E_SHAPE;
}
// the K-blocked ring (KB > 4): 16 KB stages, eight of them (one H = 512 catalog tile, 128 KB in flight), every mode with the user tile in
// tensor memory.  Shared memory: 86 KB of lists, parking area and barriers beside the ring in mode 0 (214 KB), 22 KB in the two-pass modes.
template <int KB, int BN, int MODE, bool BIAS>
int launch_tc_k(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap* tmBh, const TcArgs& k, dim3 grid, cudaStream_t s) {
  constexpr int NS = 8;
  const size_t fixed = 1024 + (MODE == 0 ? (size_t)(k.KC <= 32 ? 32 : 64) * BM * 8 : 0) + BM * 4 + 4 * 1024 * 4 + 256 + (BIAS ? 512 * 4 : 0);
  const size_t smem = fixed + (size_t)NS * BN * 128;
  if (smem > 227 * 1024) return ADT_E_SHAPE;
  return launch_tc_ns<KB, BN, NS, MODE, true, BIAS>(tmA, tmB, tmBh, k, grid, s, smem);
}
// with a bias the two-pass kernels always take the user tile in tensor memory (the default; ADT_TC_ATMEM=0 is a measurement switch
// for the unbiased kernels only), which keeps the number of instantiations down
template <int KB, int BN, int MODE>
int launch_tc(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap* tmBh, const TcArgs& k, dim3 grid, cudaStream_t s) {
  if constexpr (KB > 4) {
    if (k.bias) return launch_tc_k<KB, BN, MODE, true>(tmA, tmB, tmBh, k, grid, s);
    return launch_tc_k<KB, BN, MODE, false>(tmA, tmB, tmBh, k, grid, s);
  } else {
    if (k.bias) {
      if constexpr (MODE != 0) return launch_tc_a<KB, BN, MODE, true, true>(tmA, tmB, tmBh, k, grid, s);
      else return launch_tc_a<KB, BN, MODE, false, true>(tmA, tmB, tmBh, k, grid, s);
    }
    if (MODE != 0 && tc_atmem()) return launch_tc_a<KB, BN, MODE, true, false>(tmA, tmB, tmBh, k, grid, s);
    return launch_tc_a<KB, BN, MODE, false, false>(tmA, tmB, tmBh, k, grid, s);
  }
}
// catalog tile width: 128 items, except that the single-pass H = 256 kernel (user tile 64 KB + lists 32-64 KB on chip) only has room
// for 64-item tiles.  Wider is better there: a [128 x 64 x 16] MMA re-reads its 4 KB A fragment for 2 KB of B, 192 B/clk of a
// 128 B/clk shared-memory port; with 128 columns it is 128 B/clk (measured 512 x 1M x 256: 0.77 -> 0.66 ms).
static int tc_bn(int KB, int two_pass_mode) { return (KB == 4 && !two_pass_mode) ? 64 : 128; }
template <int MODE>
int launch_tc_h(int KB, int BN, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap* tmBh, const TcArgs& k, dim3 grid, cudaStream_t s) {
  if (KB == 1) return launch_tc<1, 128, MODE>(tmA, tmB, tmBh, k, grid, s);
  if (KB == 2) return launch_tc<2, 128, MODE>(tmA, tmB, tmBh, k, grid, s);
  if (KB == 3) return launch_tc<3, 128, MODE>(tmA, tmB, tmBh, k, grid, s);
  if (KB == 4) return BN == 64 ? launch_tc<4, 64, MODE>(tmA, tmB, tmBh, k, grid, s) : launch_tc<4, 128, MODE>(tmA, tmB, tmBh, k, grid, s);
  if (KB == 5) return launch_tc<5, 128, MODE>(tmA, tmB, tmBh, k, grid, s);
  if (KB == 6) return launch_tc<6, 128, MODE>(tmA, tmB, tmBh, k, grid, s);
  if (KB == 7) return launch_tc<7, 128, MODE>(tmA, tmB, tmBh, k, grid, s);
  if (KB == 8) return launch_tc<8, 128, MODE>(tmA, tmB, tmBh, k, grid, s);
  return ADT_E_SHAPE;
}

// tau[u] = the R-th largest of the nst sampled-tile maxima of user u (layout [sample tile][U]; -inf when there are fewer than R).
// The R largest tile maxima are R distinct catalog scores >= tau, so with a sample of 1/sstride of the tiles about R*sstride (or a few
// more) catalog items score above tau.  Warp per user, nst <= 2048.
__global__ void __launch_bounds__(256) tau_select_kernel(const float* __restrict__ tile_max, int nst, int U, int R, float* __restrict__ tau) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int u = blockIdx.x * 8 + w;
  if (u >= U) return;
  float mine[64];                             // lane l owns entries l, l+32, ...
#pragma unroll
  for (int j = 0; j < 64; ++j) {
    const int c = l + 32 * j;
    mine[j] = c < nst ? tile_max[(long long)c * U + u] : -INFINITY;
  }
  float kth = -INFINITY;
  for (int r = 0; r < R; ++r) {
    float bm = -INFINITY;
    int bj = -1;
#pragma unroll
    for (int j = 0; j < 64; ++j)
      if (mine[j] > bm) { bm = mine[j]; bj = j; }
    float wm = bm;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, o));
    const unsigned who = __ballot_sync(0xffffffffu, bj >= 0 && bm == wm);
    if (who == 0u) { kth = -INFINITY; break; }     // fewer than R scores in the sample
    if (l == __ffs(who) - 1) {
#pragma unroll
      for (int j = 0; j < 64; ++j)
        if (j == bj) mine[j] = -INFINITY;
    }
    kth = wm;
  }
  if (l == 0) tau[u] = kth;
}

}  // namespace

extern "C" int adt_to_bf16(const float* x, void* y, int64_t rows, int32_t H, float* max_normsq, adt_stream_t s_) {
  if (H & 1) return ADT_E_SHAPE;
  const long long blocks = (rows + 7) / 8;
  to_bf16_kernel<<<(int)(blocks < 148 * 16 ? (blocks > 0 ? blocks : 1) : 148 * 16), 256, 0, (cudaStream_t)s_>>>(
      x, reinterpret_cast<__nv_bfloat16*>(y), (long long)rows, H, max_normsq);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}

// launch plan of adt_score_topk_tc for (U users, n_items catalog rows, top-K): list capacity KC per (split, user) and the number of
// catalog splits.  Returns 1 when the two-pass (sample threshold + append-only) scheme applies, else 0 (single streaming pass).
static const int TC_TWO_PASS_MIN_ITEMS = 65536, TC_SSTRIDE = 16;

static int tc_target(int K) { return K * 6 > 192 ? K * 6 : 192; }    // catalog items expected above a user's threshold tau
extern "C" int adt_score_tc_plan(int32_t U, int32_t H, int32_t n_items, int32_t K, int32_t* KC_out, int32_t* n_splits_out) {
  static int two_pass = -1;
  if (two_pass < 0) { const char* e = getenv("ADT_TC_TWO_PASS"); two_pass = e ? atoi(e) : 1; }
  const int tiles = (U + BM - 1) / BM;
  const int KBp = (H + 63) / 64;
  int BN = tc_bn(KBp, 1);
  int ntt = (n_items + BN - 1) / BN;
  int S = 148 / tiles > 1 ? 148 / tiles : 1;
  if (S > ntt) S = ntt;
  int KC, mode = 0;
  // two passes pay off while a split is short (few user tiles -> many splits): with >= 8 splits per user tile a streaming list never
  // gets warm (measured: 512 users x 1M items 1.04 -> 0.78 ms at H = 256, 0.74 -> 0.51 ms at H = 64); with 32 user tiles the 4 long
  // splits of the single streaming pass are faster (4096 users: 4.0 ms vs 5.4 ms)
  if (two_pass && n_items >= TC_TWO_PASS_MIN_ITEMS && K <= 48 && S >= 8) {
    // the sample pass parks one maximum per sampled tile in the candidate scratch (n_splits*KC floats per user, <= 2048) and the
    // threshold pass needs >= 4x the expected number of candidates per split (tiles are interleaved over the splits: even spread)
    int sstride = TC_SSTRIDE;
    while (2 * ((ntt + sstride - 1) / sstride) > RS_MAXC) sstride *= 2;
    const int nst = 2 * ((ntt + sstride - 1) / sstride);      // one maximum per sampled half tile
    int R = (tc_target(K) + sstride - 1) / sstride;
    if (R < 6) R = 6;
    const int eff = R * sstride;
    int best_s = 0, best_kc = 0, best_cost = 0;
    for (int kc = 32; kc <= 64; kc *= 2) {      // keep the split count that fills the SMs when a capacity allows it, else the fewest extra splits
      int s2 = S < RS_MAXC / kc ? S : RS_MAXC / kc;
      if (s2 * kc < nst) s2 = (nst + kc - 1) / kc;
      const int per = kc - 8;               // >= 4x the expected candidates overall; each (split, column half) owns kc/2 of the slots
      if (s2 * per < 4 * eff) s2 = (4 * eff + per - 1) / per;
      const int cost = s2 <= S ? S - s2 : 4096 + s2;
      if (s2 * kc <= RS_MAXC && s2 <= ntt && (!best_s || cost < best_cost)) { best_s = s2; best_kc = kc; best_cost = cost; }
    }
    if (best_s) { S = best_s; KC = best_kc; mode = 1; } else KC = 64;
  }
  if (!mode) {
    BN = tc_bn(KBp, 0);
    ntt = (n_items + BN - 1) / BN;
    KC = K + 8 > 2 * K ? K + 8 : 2 * K;
    if (KC > 64) KC = 64;
    if (S * KC > RS_MAXC) S = RS_MAXC / KC;
  }
  if (S < 1) S = 1;
  *KC_out = KC; *n_splits_out = S;
  return mode;
}

extern "C" int adt_score_topk_tc(const adt_score_topk_tc_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (a->H % 64 || a->H > 512 || a->K <= 0 || a->K > a->KC || a->KC > 64 || a->n_splits <= 0 || a->n_splits * a->KC > RS_MAXC || a->U <= 0)
    return ADT_E_SHAPE;
  if (a->item_bias && !a->max_abs_bias) return ADT_E_SHAPE;
  CUtensorMap tmA, tmB;
  const int KB = a->H / 64;
  if (int e = make_map(&tmA, a->feats_bf16, a->U, a->H, BM)) return e;
  TcArgs k;
  k.seen_indptr = a->seen_indptr; k.seen_idx = a->seen_idx; k.part_scores = a->part_scores; k.part_ids = a->part_ids; k.part_thr = a->part_thr;
  k.U = a->U; k.n_items = a->n_items; k.item_offset = a->item_offset; k.KC = a->KC; k.n_splits = a->n_splits;
  k.feats_bf16 = reinterpret_cast<const __nv_bfloat16*>(a->feats_bf16);
  k.bias = a->item_bias;
  k.gthr = nullptr;
  if (a->n_splits > 1 && a->flags) {     // `flags` doubles as the threshold exchange buffer until the re-score kernel overwrites it
    k.gthr = reinterpret_cast<unsigned int*>(a->flags);
    cudaMemsetAsync(a->flags, 0, sizeof(int) * (size_t)a->U, s);
  }
  { const char* dbg = getenv("ADT_TC_DEBUG"); k.debug = dbg ? atoi(dbg) : 0; }
  dim3 grid(a->n_splits, (a->U + BM - 1) / BM);
  int rc;
  bool two = false;
  k.tau = nullptr; k.sstride = 1;
  // Large catalogs: two passes.  (1) a SAMPLE of every 16th catalog tile is scored and only the maximum of each sampled tile is kept
  // per user; the R-th largest of those maxima becomes the user's threshold tau, so about 16 R (>= 6 K) catalog items score above it.
  // (2) the whole catalog is scored against that FIXED threshold: the epilogue is one max-reduction and one compare per 32 scores, the
  // rare candidates are appended straight to HBM (no sorted lists, no warm-up phase per split, no list storage on chip -> a deeper
  // TMA ring).  Everything above tau is a candidate, so the exactness test of the re-score kernel is unchanged (thr = tau, or +inf
  // after an overflow of a split's KC slots).
  static int two_pass = -1;
  if (two_pass < 0) { const char* e = getenv("ADT_TC_TWO_PASS"); two_pass = e ? atoi(e) : 1; }
  // sample stride: every 16th catalog tile, coarser when the tile maxima would not fit the scratch (part_scores holds
  // n_splits*KC floats per user) or the selection kernel (2048 values per user)
  int BN = tc_bn(KB, 1);
  const int ntt = (a->n_items + BN - 1) / BN;
  int cap = a->n_splits * a->KC < 2048 ? a->n_splits * a->KC : 2048;
  cap /= 2;                                  // the sample pass keeps one maximum per sampled HALF tile (two epilogue warps per row)
  int sstride = TC_SSTRIDE;
  while ((ntt + sstride - 1) / sstride > cap) sstride *= 2;
  const int nst = (ntt + sstride - 1) / sstride;
  int R = (tc_target(a->K) + sstride - 1) / sstride;
  if (R < 6) R = 6;
  // two passes only when the caller's scratch follows adt_score_tc_plan: room for 4x the expected candidates of a split
  if (two_pass && a->n_items >= TC_TWO_PASS_MIN_ITEMS && a->K <= 48 && nst >= 4 * R && (long long)a->n_splits * (a->KC - 8) >= 4ll * R * sstride) {
    if (int e = make_map(&tmB, a->item_emb_bf16, a->n_items, a->H, BN)) return e;
    TcArgs ks = k;
    ks.sstride = sstride; ks.gthr = nullptr;
    // pairs of user tiles share every catalog tile through TMA multicast (ADT_TC_MULTICAST=0 disables)
    static int mc = -1;
    if (mc < 0) { const char* e = getenv("ADT_TC_MULTICAST"); mc = e ? atoi(e) : 1; }
    CUtensorMap tmBhalf;
    const CUtensorMap* tmBh = nullptr;
    if (mc && (grid.y % 2) == 0) {
      if (int e = make_map(&tmBhalf, a->item_emb_bf16, a->n_items, a->H, BN / 2)) return e;
      tmBh = &tmBhalf;
    }
    rc = launch_tc_h<2>(KB, BN, tmA, tmB, tmBh, ks, grid, s);
    if (rc) return rc;
    float* tau = a->out_scores;            // U floats of scratch: overwritten by the re-score kernel at the end
    tau_select_kernel<<<(a->U + 7) / 8, 256, 0, s>>>(a->part_scores, 2 * nst, a->U, R, tau);
    two = true;
    k.tau = tau; k.gthr = nullptr;
    rc = launch_tc_h<1>(KB, BN, tmA, tmB, tmBh, k, grid, s);
  } else {
    BN = tc_bn(KB, 0);
    if (int e = make_map(&tmB, a->item_emb_bf16, a->n_items, a->H, BN)) return e;
    rc = launch_tc_h<0>(KB, BN, tmA, tmB, nullptr, k, grid, s);
  }
  if (rc) return rc;
  RescoreArgs r;
  r.feats = a->feats; r.E = a->item_emb; r.part_scores = a->part_scores; r.part_ids = a->part_ids; r.part_thr = a->part_thr;
  r.max_normsq = a->max_normsq; r.out_scores = a->out_scores; r.out_ids = a->out_ids; r.flags = a->flags;
  r.U = a->U; r.H = a->H; r.item_offset = a->item_offset; r.K = a->K; r.KC = a->KC; r.n_splits = a->n_splits;
  if (two) { r.KC = a->KC / 2; r.n_splits = 2 * a->n_splits; }     // every (split, column half) wrote its own list and threshold
  r.answers = a->answers; r.metric_acc = a->metric_acc;
  r.bias = a->item_bias; r.max_abs_bias = a->max_abs_bias;
  const bool wide = a->H > 256;
  void (*rk)(RescoreArgs) = a->item_bias ? (wide ? rescore_select_kernel<true, 512> : rescore_select_kernel<true, 256>)
                                         : (wide ? rescore_select_kernel<false, 512> : rescore_select_kernel<false, 256>);
  const size_t rsm = rs_smem(wide ? 512 : 256);
  cudaFuncSetAttribute(rk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rsm);
  rk<<<a->U, RS_NT, rsm, s>>>(r);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}
