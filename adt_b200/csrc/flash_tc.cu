// Fused attention core for long sequences (up to 2048 positions) on the 5th-generation tensor cores: S = q k^T and P never leave
// the SM.  Same masks, same Philox dropout stream, same lse and the same bf16 rounding of the dropped probabilities as the batched
// tcgen05 path of block_tc.cuh (attn_row_kernel + strided-batch adt_gemm_tc), which writes [B*nh][L][L] scores to HBM instead.
//
// Operands: the bf16 pack [q | k | v] ([M][3H], q pre-scaled) and, backward, bf16 dctx [M][H], read through 4-D TMA maps
// {column in head, row, head, sequence}: a tile never crosses the end of its sequence (TMA zero-fills rows >= L and columns >= hd).
// A [128 x hd] tile is ks = ceil(hd / 64) boxes of [128 rows x 64 bf16] with 128-byte swizzle, one 16 KB box per 64 columns.  The
// same bytes serve as a K-major operand (q, k, dctx, v in the score products) and as an MN-major one (v in P v, dctx and q in the
// key-gradient products, k in dS k): every MMA with N = hd runs at N = 64 ks over the zero-filled columns.
//
// One CTA = 128 threads; thread t owns TMEM lane t = query row t of the tile, so each Philox call serves the 8 keys of one row as in
// attn_row_kernel.  Thread 0 also issues the TMA loads and the MMAs (one issuer, mbarrier hand-offs).
//   forward  : CTA per (sequence*head, 128-query tile), walks key tiles (above the causal diagonal skipped) with a 2-stage k/v ring;
//              S -> TMEM, online max / sum in registers, P~ = bf16(exp(s - m) * mask) -> smem, O += P~ v in TMEM (rescaled in TMEM
//              when the running max moves), ctx = O / l, lse = m + log l.
//   dk / dv  : CTA per (sequence*head, 128-key tile), walks query tiles; S = q k^T and dP~ = dctx v^T -> TMEM, P = exp(s - lse),
//              dS = P (dP~ m - delta) with delta = rowsum(dctx ctx); dv += P~^T dctx, dk += dS^T q with P~ / dS read MN-major.
//   dq       : CTA per (sequence*head, 128-query tile), walks key tiles; the same S, dP~, dS; dq += dS k.
// Every output element is written once with a plain store: no atomics, no memsets, bitwise reproducible.
#include <string.h>

#include "../../include/adt_b200.h"
#include "flash_tc.cuh"

namespace adt {

namespace {

// scores of keys jb .. jb+31 for query row i: keys >= L and (causal) keys > i are excluded; padded keys (mask_mode 1) are REPLACED by
// -1e9 as masked_fill does, so a fully padded row stays uniform over its L keys
__device__ __forceinline__ void mask32(float (&v)[32], int i, int jb, const FlashArgs& a, const int* __restrict__ kid) {
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    const int j = jb + k;
    if (j >= a.L || (a.mask_mode == 0 && j > i)) v[k] = -INFINITY;
    else if (a.mask_mode == 1 && __ldg(kid + j) == 0) v[k] = -1e9f;
  }
}

__global__ void __launch_bounds__(FT, 1) flash_fwd_kernel(const __grid_constant__ CUtensorMap tq, const __grid_constant__ CUtensorMap tk,
                                                          const __grid_constant__ CUtensorMap tv, FlashArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const int ks = a.ks, SB = ks * BOX;
  uint8_t* sQ = align1024(smem_raw);
  uint8_t* sK = sQ + SB;                 // [2] stages
  uint8_t* sV = sK + 2 * SB;             // [2] stages
  uint8_t* sP = sV + 2 * SB;             // [128 queries][128 keys]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * BOX);
  uint64_t *q_full = bars, *kv_full = bars + 1, *s_bar = bars + 3, *pv_bar = bars + 4;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 5);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int z = blockIdx.x, b = z / a.nh, h = z - b * a.nh;
  const int nqt = (a.L + FT - 1) / FT, qt = nqt - 1 - blockIdx.y, q0 = qt * FT;
  const int nkt = a.mask_mode == 0 ? qt + 1 : nqt;
  const int* kid = a.key_ids ? a.key_ids + (long long)b * a.L : nullptr;

  if (tid == 0) {
    tc::tma_prefetch_desc(&tq); tc::tma_prefetch_desc(&tk); tc::tma_prefetch_desc(&tv);
    for (int i = 0; i < 5; ++i) tc::mbar_init(bars + i, 1);
    tc::fence_barrier_init();
  }
  if (warp == 0) tc::tmem_alloc<256>(tslot);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t lane_off = (uint32_t)(32 * warp) << 16;
  const uint32_t tS = *tslot, tO = tS + 128;

  auto load_kv = [&](int t) {
    const int st = t & 1;
    tc::mbar_arrive_expect_tx(kv_full + st, 2 * SB);
    load_tile(sK + st * SB, &tk, ks, t * FT, h, b, kv_full + st);
    load_tile(sV + st * SB, &tv, ks, t * FT, h, b, kv_full + st);
  };
  if (tid == 0) {
    tc::mbar_arrive_expect_tx(q_full, SB);
    load_tile(sQ, &tq, ks, q0, h, b, q_full);
    load_kv(0);
    if (nkt > 1) load_kv(1);
    tc::mbar_wait(q_full, 0);
    tc::mbar_wait(kv_full, 0);
    tc::tc_fence_after();
    mma_kk(tS, sQ, sK, a.hd);
    tc::mma_commit(s_bar);
  }
  __syncwarp();

  const int i = q0 + tid;
  const bool row_ok = i < a.L;
  const unsigned long long drow = a.drop.base + (unsigned long long)z * a.L + i;
  float m_run = -INFINITY, l_run = 0.f;
  for (int t = 0; t < nkt; ++t) {
    const int j0 = t * FT;
    tc::mbar_wait(s_bar, t & 1);
    tc::tc_fence_after();
    float mt = -INFINITY;
    for (int c0 = 0; c0 < FT; c0 += 32) {
      float v[32];
      tc::tmem_ld32(tS + lane_off + c0, v);
      mask32(v, i, j0 + c0, a, kid);
#pragma unroll
      for (int k = 0; k < 32; ++k) mt = fmaxf(mt, v[k]);
    }
    const float m_new = fmaxf(m_run, mt), alpha = exp2f((m_run - m_new) * LOG2E);
    m_run = m_new;
    if (t > 0) {                                  // P~ v of the previous tile done: P~ buffer free, O stable -> rescale O
      tc::mbar_wait(pv_bar, (t - 1) & 1);
      tc::tc_fence_after();
      if (__any_sync(0xffffffffu, alpha != 1.f)) {
        for (int c0 = 0; c0 < 64 * ks; c0 += 32) {
          float v[32];
          tc::tmem_ld32(tO + lane_off + c0, v);
          uint32_t u[32];
#pragma unroll
          for (int k = 0; k < 32; ++k) u[k] = __float_as_uint(v[k] * alpha);
          tc::tmem_st32(tO + lane_off + c0, u);
        }
        tc::tmem_st_wait();
      }
    }
    float ls = 0.f;
    for (int c0 = 0; c0 < FT; c0 += 32) {
      float v[32], mv[32];
      tc::tmem_ld32(tS + lane_off + c0, v);
      mask32(v, i, j0 + c0, a, kid);
      drop32(mv, i, j0 + c0, row_ok, drow, a);
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const float p = v[k] == -INFINITY ? 0.f : exp2f((v[k] - m_new) * LOG2E);
        ls += p;
        v[k] = p * mv[k];
      }
      st_row32(sP, tid, c0, v);
    }
    l_run = l_run * alpha + ls;
    tc::fence_proxy_async();
    tc::tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc::tc_fence_after();
      mma_xn(tO, sP, 0, sV + (t & 1) * SB, ks, t > 0);
      tc::mma_commit(pv_bar);
      if (t + 1 < nkt) {
        tc::mbar_wait(kv_full + ((t + 1) & 1), ((t + 1) >> 1) & 1);
        tc::tc_fence_after();
        mma_kk(tS, sQ, sK + ((t + 1) & 1) * SB, a.hd);
        tc::mma_commit(s_bar);
      }
      if (t + 2 < nkt) {                          // stage t & 1 is free once P~ v of tile t completed
        tc::mbar_wait(pv_bar, t & 1);
        load_kv(t + 2);
      }
    }
    __syncwarp();
  }
  tc::mbar_wait(pv_bar, (nkt - 1) & 1);
  tc::tc_fence_after();
  const long long grow = (long long)b * a.L + i;
  store_acc(tO + lane_off, row_ok ? a.ctx + grow * a.H : nullptr, h * a.hd, a.hd, ks, 1.f / l_run);
  if (row_ok && a.lse) a.lse[(long long)z * a.L + i] = m_run + logf(l_run);
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc<256>(tS);
}

// backward softmax adjoint of one [128 queries x 128 keys] tile from S and dP~ in TMEM: P~ = P m -> sP (nullable), dS = P (dP~ m - delta)
// -> sDS, both bf16 [query][key]
__device__ __forceinline__ void bwd_tile(uint32_t tS, uint32_t tdP, uint8_t* sP, uint8_t* sDS, int i, int j0, bool row_ok, float lse_i,
                                         float delta_i, unsigned long long drow, const FlashArgs& a, const int* kid) {
  const int r = threadIdx.x;
  for (int c0 = 0; c0 < FT; c0 += 32) {
    float v[32], dp[32], mv[32];
    tc::tmem_ld32(tS + c0, v);
    tc::tmem_ld32(tdP + c0, dp);
    mask32(v, i, j0 + c0, a, kid);
    drop32(mv, i, j0 + c0, row_ok, drow, a);
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      const float p = (v[k] == -INFINITY || !row_ok) ? 0.f : exp2f((v[k] - lse_i) * LOG2E);
      v[k] = p * mv[k];
      dp[k] = p * (dp[k] * mv[k] - delta_i);
    }
    if (sP) st_row32(sP, r, c0, v);
    st_row32(sDS, r, c0, dp);
  }
}

__global__ void __launch_bounds__(FT, 1) flash_bwd_dkdv_kernel(const __grid_constant__ CUtensorMap tq, const __grid_constant__ CUtensorMap tk,
                                                               const __grid_constant__ CUtensorMap tv, const __grid_constant__ CUtensorMap tdo,
                                                               FlashArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const int ks = a.ks, SB = ks * BOX, NS = a.nstage;
  uint8_t* sK = align1024(smem_raw);
  uint8_t* sV = sK + SB;
  uint8_t* sQ = sV + SB;                 // [NS] stages of q, then [NS] of dctx
  uint8_t* sD = sQ + NS * SB;
  uint8_t* sP = sD + NS * SB;
  uint8_t* sDS = sP + 2 * BOX;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sDS + 2 * BOX);
  uint64_t *kv_full = bars, *qd_full = bars + 1, *sd_bar = bars + 3, *mm_bar = bars + 4;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 5);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int z = blockIdx.x, b = z / a.nh, h = z - b * a.nh;
  const int nt = (a.L + FT - 1) / FT, kt = nt - 1 - blockIdx.y, k0 = kt * FT;
  const int qbeg = a.mask_mode == 0 ? kt : 0, nq = nt - qbeg;
  const int* kid = a.key_ids ? a.key_ids + (long long)b * a.L : nullptr;

  if (tid == 0) {
    tc::tma_prefetch_desc(&tq); tc::tma_prefetch_desc(&tk); tc::tma_prefetch_desc(&tv); tc::tma_prefetch_desc(&tdo);
    for (int i = 0; i < 5; ++i) tc::mbar_init(bars + i, 1);
    tc::fence_barrier_init();
  }
  if (warp == 0) tc::tmem_alloc<512>(tslot);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t lane_off = (uint32_t)(32 * warp) << 16;
  const uint32_t tS = *tslot, tdP = tS + 128, tdV = tS + 256, tdK = tS + 384;

  auto load_qd = [&](int n) {
    const int st = n % NS;
    tc::mbar_arrive_expect_tx(qd_full + st, 2 * SB);
    load_tile(sQ + st * SB, &tq, ks, (qbeg + n) * FT, h, b, qd_full + st);
    load_tile(sD + st * SB, &tdo, ks, (qbeg + n) * FT, h, b, qd_full + st);
  };
  auto issue_sdp = [&](int n) {
    const int st = n % NS;
    mma_kk(tS, sQ + st * SB, sK, a.hd);
    mma_kk(tdP, sD + st * SB, sV, a.hd);
    tc::mma_commit(sd_bar);
  };
  if (tid == 0) {
    tc::mbar_arrive_expect_tx(kv_full, 2 * SB);
    load_tile(sK, &tk, ks, k0, h, b, kv_full);
    load_tile(sV, &tv, ks, k0, h, b, kv_full);
    for (int n = 0; n < NS && n < nq; ++n) load_qd(n);
    tc::mbar_wait(kv_full, 0);
    tc::mbar_wait(qd_full, 0);
    tc::tc_fence_after();
    issue_sdp(0);
  }
  __syncwarp();

  for (int n = 0; n < nq; ++n) {
    const int i = (qbeg + n) * FT + tid;
    const bool row_ok = i < a.L;
    const long long zi = (long long)z * a.L + i;
    const float lse_i = row_ok ? __ldg(a.lse_in + zi) : 0.f, delta_i = row_ok ? __ldg(a.delta + zi) : 0.f;
    tc::mbar_wait(sd_bar, n & 1);
    tc::tc_fence_after();
    if (n > 0) tc::mbar_wait(mm_bar, (n - 1) & 1);     // the previous dv / dk products have read sP / sDS
    bwd_tile(tS + lane_off, tdP + lane_off, sP, sDS, i, k0, row_ok, lse_i, delta_i, a.drop.base + (unsigned long long)zi, a, kid);
    tc::fence_proxy_async();
    tc::tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc::tc_fence_after();
      const int st = n % NS;
      mma_xn(tdV, sP, 1, sD + st * SB, ks, n > 0);     // dv += P~^T dctx
      mma_xn(tdK, sDS, 1, sQ + st * SB, ks, n > 0);    // dk += dS^T q
      tc::mma_commit(mm_bar);
      if (NS == 1) {
        tc::mbar_wait(mm_bar, n & 1);
        if (n + 1 < nq) load_qd(n + 1);
      }
      if (n + 1 < nq) {
        tc::mbar_wait(qd_full + (n + 1) % NS, ((n + 1) / NS) & 1);
        tc::tc_fence_after();
        issue_sdp(n + 1);
      }
      if (NS == 2) {
        tc::mbar_wait(mm_bar, n & 1);
        if (n + 2 < nq) load_qd(n + 2);
      }
    }
    __syncwarp();
  }
  tc::mbar_wait(mm_bar, (nq - 1) & 1);
  tc::tc_fence_after();
  const int j = k0 + tid;
  const long long grow = (long long)b * a.L + j;
  store_acc(tdV + lane_off, j < a.L ? a.dv + grow * a.H : nullptr, h * a.hd, a.hd, ks, 1.f);
  store_acc(tdK + lane_off, j < a.L ? a.dk + grow * a.H : nullptr, h * a.hd, a.hd, ks, 1.f);
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc<512>(tS);
}

__global__ void __launch_bounds__(FT, 1) flash_bwd_dq_kernel(const __grid_constant__ CUtensorMap tq, const __grid_constant__ CUtensorMap tk,
                                                             const __grid_constant__ CUtensorMap tv, const __grid_constant__ CUtensorMap tdo,
                                                             FlashArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const int ks = a.ks, SB = ks * BOX, NS = a.nstage;
  uint8_t* sQ = align1024(smem_raw);
  uint8_t* sD = sQ + SB;
  uint8_t* sK = sD + SB;                 // [NS] stages of k, then [NS] of v
  uint8_t* sV = sK + NS * SB;
  uint8_t* sDS = sV + NS * SB;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sDS + 2 * BOX);
  uint64_t *qd_full = bars, *kv_full = bars + 1, *sd_bar = bars + 3, *mm_bar = bars + 4;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 5);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int z = blockIdx.x, b = z / a.nh, h = z - b * a.nh;
  const int nt = (a.L + FT - 1) / FT, qt = nt - 1 - blockIdx.y, q0 = qt * FT;
  const int nkt = a.mask_mode == 0 ? qt + 1 : nt;
  const int* kid = a.key_ids ? a.key_ids + (long long)b * a.L : nullptr;

  if (tid == 0) {
    tc::tma_prefetch_desc(&tq); tc::tma_prefetch_desc(&tk); tc::tma_prefetch_desc(&tv); tc::tma_prefetch_desc(&tdo);
    for (int i = 0; i < 5; ++i) tc::mbar_init(bars + i, 1);
    tc::fence_barrier_init();
  }
  if (warp == 0) tc::tmem_alloc<512>(tslot);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t lane_off = (uint32_t)(32 * warp) << 16;
  const uint32_t tS = *tslot, tdP = tS + 128, tdQ = tS + 256;

  auto load_kv = [&](int n) {
    const int st = n % NS;
    tc::mbar_arrive_expect_tx(kv_full + st, 2 * SB);
    load_tile(sK + st * SB, &tk, ks, n * FT, h, b, kv_full + st);
    load_tile(sV + st * SB, &tv, ks, n * FT, h, b, kv_full + st);
  };
  auto issue_sdp = [&](int n) {
    const int st = n % NS;
    mma_kk(tS, sQ, sK + st * SB, a.hd);
    mma_kk(tdP, sD, sV + st * SB, a.hd);
    tc::mma_commit(sd_bar);
  };
  if (tid == 0) {
    tc::mbar_arrive_expect_tx(qd_full, 2 * SB);
    load_tile(sQ, &tq, ks, q0, h, b, qd_full);
    load_tile(sD, &tdo, ks, q0, h, b, qd_full);
    for (int n = 0; n < NS && n < nkt; ++n) load_kv(n);
    tc::mbar_wait(qd_full, 0);
    tc::mbar_wait(kv_full, 0);
    tc::tc_fence_after();
    issue_sdp(0);
  }
  __syncwarp();

  const int i = q0 + tid;
  const bool row_ok = i < a.L;
  const long long zi = (long long)z * a.L + i;
  const float lse_i = row_ok ? __ldg(a.lse_in + zi) : 0.f, delta_i = row_ok ? __ldg(a.delta + zi) : 0.f;
  for (int n = 0; n < nkt; ++n) {
    tc::mbar_wait(sd_bar, n & 1);
    tc::tc_fence_after();
    if (n > 0) tc::mbar_wait(mm_bar, (n - 1) & 1);     // the previous dq product has read sDS
    bwd_tile(tS + lane_off, tdP + lane_off, nullptr, sDS, i, n * FT, row_ok, lse_i, delta_i, a.drop.base + (unsigned long long)zi, a, kid);
    tc::fence_proxy_async();
    tc::tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc::tc_fence_after();
      mma_xn(tdQ, sDS, 0, sK + (n % NS) * SB, ks, n > 0);   // dq += dS k
      tc::mma_commit(mm_bar);
      if (NS == 1) {
        tc::mbar_wait(mm_bar, n & 1);
        if (n + 1 < nkt) load_kv(n + 1);
      }
      if (n + 1 < nkt) {
        tc::mbar_wait(kv_full + (n + 1) % NS, ((n + 1) / NS) & 1);
        tc::tc_fence_after();
        issue_sdp(n + 1);
      }
      if (NS == 2) {
        tc::mbar_wait(mm_bar, n & 1);
        if (n + 2 < nkt) load_kv(n + 2);
      }
    }
    __syncwarp();
  }
  tc::mbar_wait(mm_bar, (nkt - 1) & 1);
  tc::tc_fence_after();
  const long long grow = (long long)b * a.L + i;
  store_acc(tdQ + lane_off, row_ok ? a.dq + grow * a.H : nullptr, h * a.hd, a.hd, ks, 1.f);
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc<512>(tS);
}

// delta[z][i] = sum_c dctx[b, i, head h, c] * ctx[b, i, head h, c]   (one warp per (row, head))
__global__ void __launch_bounds__(256) flash_delta_kernel(const float* __restrict__ ctx, const float* __restrict__ dctx, float* __restrict__ delta,
                                                          int M, int L, int H, int nh) {
  const int lane = threadIdx.x & 31, hd = H / nh;
  const long long n = (long long)M * nh;
  for (long long w = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); w < n; w += (long long)gridDim.x * 8) {
    const long long r = w / nh;
    const int h = (int)(w - r * nh);
    const float* c = ctx + r * H + h * hd;
    const float* d = dctx + r * H + h * hd;
    float s = 0.f;
    for (int k = lane; k < hd; k += 32) s = fmaf(c[k], d[k], s);
    s = warp_sum(s);
    const long long b = r / L, i = r - b * L;
    if (lane == 0) delta[(b * nh + h) * L + i] = s;
  }
}

size_t fwd_smem(int ks) { return 1024 + (size_t)5 * ks * BOX + 2 * BOX + 64; }
size_t dkdv_smem(int ks, int ns) { return 1024 + (size_t)(2 + 2 * ns) * ks * BOX + 4 * BOX + 64; }
size_t dq_smem(int ks, int ns) { return 1024 + (size_t)(2 + 2 * ns) * ks * BOX + 2 * BOX + 64; }

FlashArgs mk_args(int L, int H, int nh, int mask_mode, const int* key_ids, const DropDesc& d) {
  FlashArgs a;
  memset(&a, 0, sizeof(a));
  a.L = L; a.H = H; a.nh = nh; a.hd = H / nh; a.ks = (a.hd + 63) / 64; a.mask_mode = mask_mode; a.key_ids = key_ids; a.drop = d;
  a.nstage = a.ks == 1 ? 2 : 1;
  return a;
}

}  // namespace

// fused forward over the bf16 pack qkv = [q | k | v] ([B*L][3H]); writes ctx [B*L][H] fp32 and lse [B][nh][L] (nullable)
int flash_attn_fwd(const __nv_bfloat16* qkv, float* ctx, float* lse, const int* key_ids, int B, int L, int H, int nh, int mask_mode,
                   const DropDesc& d, cudaStream_t s) {
  FlashArgs a = mk_args(L, H, nh, mask_mode, key_ids, d);
  a.ctx = ctx; a.lse = lse;
  CUtensorMap tq, tk, tv;
  if (head_map(&tq, qkv, B, L, H, nh, 3 * H) || head_map(&tk, qkv + H, B, L, H, nh, 3 * H) || head_map(&tv, qkv + 2 * H, B, L, H, nh, 3 * H))
    return ADT_E_CUDA;
  const size_t sm = fwd_smem(a.ks);
  cudaFuncSetAttribute(flash_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
  flash_fwd_kernel<<<dim3(B * nh, (L + FT - 1) / FT), FT, sm, s>>>(tq, tk, tv, a);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}

// fused backward: delta from ctx and dctx (fp32), then dk / dv and dq from the bf16 packs qkv and dcb = bf16(dctx) [B*L][H]
int flash_attn_bwd(const __nv_bfloat16* qkv, const __nv_bfloat16* dcb, const float* ctx, const float* dctx, float* delta, const float* lse,
                   const int* key_ids, float* dq, float* dk, float* dv, int B, int L, int H, int nh, int mask_mode, const DropDesc& d,
                   cudaStream_t s) {
  const long long M = (long long)B * L, rows = M * nh;
  const long long blocks = (rows + 7) / 8;
  flash_delta_kernel<<<(int)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, s>>>(ctx, dctx, delta, (int)M, L, H, nh);
  FlashArgs a = mk_args(L, H, nh, mask_mode, key_ids, d);
  a.lse_in = lse; a.delta = delta; a.dq = dq; a.dk = dk; a.dv = dv;
  CUtensorMap tq, tk, tv, tdo;
  if (head_map(&tq, qkv, B, L, H, nh, 3 * H) || head_map(&tk, qkv + H, B, L, H, nh, 3 * H) || head_map(&tv, qkv + 2 * H, B, L, H, nh, 3 * H) ||
      head_map(&tdo, dcb, B, L, H, nh, H))
    return ADT_E_CUDA;
  const dim3 grid(B * nh, (L + FT - 1) / FT);
  const size_t s1 = dkdv_smem(a.ks, a.nstage), s2 = dq_smem(a.ks, a.nstage);
  cudaFuncSetAttribute(flash_bwd_dkdv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s1);
  cudaFuncSetAttribute(flash_bwd_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s2);
  flash_bwd_dkdv_kernel<<<grid, FT, s1, s>>>(tq, tk, tv, tdo, a);
  flash_bwd_dq_kernel<<<grid, FT, s2, s>>>(tq, tk, tv, tdo, a);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}

}  // namespace adt
