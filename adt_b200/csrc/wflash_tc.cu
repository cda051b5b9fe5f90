// STOSA-ADT's Wasserstein attention core (kernels_stosa.cuh: wattn_fwd_kernel / wattn_bwd_kernel) for sequences whose keys the
// resident kernels cannot hold in shared memory, up to 2048 positions, on the 5th-generation tensor cores: the scores never leave the SM.
// Same scores, same additive mask (-2^32 + 1), same Philox dropout stream and the same (max, 1/sum) row statistics as the resident
// kernels; bf16 operands, fp32 accumulation.  The tile machinery is flash_tc.cuh's (TMA ring, mbarrier hand-offs, one issuing thread).
//
// Score operands.  The distance |x_i - y_j|^2 of x = [mq | sqrt cq] and y = [mk | sqrt ck] (sqrt after the 1e-24 clamp) is formed as
// n_i + n_j - 2 <x'_i, y'_j> over the centred rows x' = x - mu, y' = y - mu, mu = the fp32 column mean of the sequence's key rows of the
// head.  A shift shared by both sides leaves the distance unchanged; without it bf16 would round the ~1 that every sqrt(elu + 1) carries
// at initialisation, 100x the spread that tells keys apart.  n = |bf16(x')|^2 in fp32: the score is the exact distance of the rounded
// points, never negative.  Gradients are formed the same way, dS Y' - rowsum(dS) x' (fp32 row / column sums of the bf16 dS).
// The values are centred for the same reason (every cv ~ 1 at initialisation): bf16 mv - mu_mv, cv - mu_cv; the forward adds mu back
// with the fp32 row sums of P~ and P~^2, the backward adds dmctx . mu_mv and dcctx . mu_cv to dP_m, dP_c in fp32, where the
// cancellation dP - delta would otherwise amplify the rounding of the shared part.
//
// prep    : CTA per (sequence, head): mu, bf16 X' / Y' [B*L][2H] (head h at columns 2 hd h ..), bf16 mv / cv [B*L][H], fp32 norms
//           [B][nh][L], the value means, the first valid key of each sequence; backward: bf16 dmctx / dcctx and delta = dmctx.mctx + 2 dcctx.cctx
//           (= sum_j P dP of the resident backward, which is why the backward reads the forward's outputs).
// forward : CTA per (sequence*head, 128-query tile), walks key tiles: S = X' Y'^T -> TMEM, s = (2S - n_i - n_j) / sqrt(hd) + mask,
//           online max / sum, P~ = P m and P~^2 -> smem (bf16), O_m += P~ mv and O_c += P~^2 cv in TMEM (rescaled by alpha / alpha^2
//           when the running max moves); mctx = O_m / l, cctx = O_c / l^2.
// dq      : CTA per query tile, walks key tiles: S, dP_m = dmctx mv^T, dP_c = dcctx cv^T -> TMEM; dP = m (dP_m + 2 P~ dP_c),
//           dS = P (dP - delta) / sqrt(hd) -> smem; A += dS Y'; dmq = 2 (A - rs x')_m, dcq = (A - rs x')_s / sqrt(cq) (-rs below the clamp).
// dk      : CTA per key tile, walks query tiles: the same dS; B += dS^T X'; dmk, dck likewise with the column sums cs.
// dv      : CTA per key tile, walks query tiles: S only; dmv += P~^T dmctx, dcv += (P~^2)^T dcctx.
// TMEM: forward S + O_m + O_c = 256 columns; dq / dk S + dP_m + dP_c + a [128 x 2hd] accumulator = 512; dv 256.
// A row before its sequence's first valid key has no valid key: the additive mask absorbs every one of its scores in fp32, so it
// attends uniformly to all L keys, future ones included (max -2^32, 1/sum = 1/L), and gradients still flow through it.  Tiles holding
// such rows therefore walk every tile of the other side instead of stopping at the causal diagonal.
// Every output element is written once with a plain store: no atomics, no memsets, bitwise reproducible.
#include <string.h>

#include "../../include/adt_b200.h"
#include "flash_tc.cuh"

namespace adt {

namespace {

constexpr float WF_MASK = -4294967296.0f;     // float(-2^32 + 1): the additive mask (W_MASK of kernels_stosa.cuh)
constexpr float WF_CLAMP = 1e-24f;            // clamp of the covariances before the square root (W_CLAMP)

struct WFlashArgs {
  FlashArgs f;                                // L, H, nh, hd, key_ids, nstage, drop (mask_mode 1: dropout over all L keys of a row)
  const float *nq, *nk;                       // [B][nh][L] norms of the query / key packs
  const int* first;                           // [B] first valid key of each sequence (L when there is none)
  float* stat;                                // (max, 1/sum) [B][nh][L][2]: written by the forward, read by the backward
  float *mctx, *cctx;                         // forward outputs [B*L][H]
  const float* delta;                         // [B][nh][L]
  const float* vmu;                           // [B][nh][2hd] column means of the value rows [mv | cv] (bf16 values are centred on them)
  const float *vm, *vc;                       // backward [B][nh][L]: dmctx . mu_mv, dcctx . mu_cv (the centring's share of dP_m, dP_c)
  const float *cq, *ck;                       // covariance streams (clamp branch of the backward epilogues)
  const __nv_bfloat16 *xp, *yp;               // the packs X', Y' (backward epilogues)
  float *dmq, *dcq, *dmk, *dck, *dmv, *dcv;
  int ks2;                                    // 64-column boxes of one [128 x 2hd] score operand tile
  float scale;                                // 1 / sqrt(hd)
};

// mu, packs, norms and first valid key of head h of sequence b (one CTA of 256 threads)
__global__ void __launch_bounds__(256) wflash_prep_kernel(const float* __restrict__ mq, const float* __restrict__ cq, const float* __restrict__ mk,
                                                          const float* __restrict__ ck, const float* __restrict__ mv, const float* __restrict__ cv,
                                                          const int* __restrict__ ids, int L, int H, int nh, __nv_bfloat16* __restrict__ xp,
                                                          __nv_bfloat16* __restrict__ yp, __nv_bfloat16* __restrict__ mvb,
                                                          __nv_bfloat16* __restrict__ cvb, float* __restrict__ nq, float* __restrict__ nk,
                                                          int* __restrict__ first, float* __restrict__ vmu) {
  __shared__ float part[256], vpart[256];
  __shared__ float mu[128], nu[128];
  __shared__ int fmin;
  const int z = blockIdx.x, b = z / nh, h = z - b * nh, hd = H / nh, W = 2 * hd, tid = threadIdx.x;
  const int G = 256 / W, c = tid % W, g = tid / W;
  const long long row0 = (long long)b * L;
  float s = 0.f, v = 0.f;                                   // column sums of y = [mk | sqrt ck] and of [mv | cv] over the L keys, fixed order
  if (g < G)
    for (int j = g; j < L; j += G) {
      const long long o = (row0 + j) * H + h * hd;
      s += c < hd ? mk[o + c] : sqrtf(fmaxf(ck[o + c - hd], WF_CLAMP));
      v += c < hd ? mv[o + c] : cv[o + c - hd];
    }
  part[tid] = s;
  vpart[tid] = v;
  if (tid == 0) fmin = L;
  __syncthreads();
  if (tid < W) {
    float t = 0.f, u = 0.f;
    for (int k = 0; k < G; ++k) t += part[k * W + tid], u += vpart[k * W + tid];
    mu[tid] = t / (float)L;
    nu[tid] = u / (float)L;
    vmu[(long long)z * W + tid] = nu[tid];
  }
  for (int j = tid; j < L; j += 256)
    if (ids[row0 + j] > 0) atomicMin(&fmin, j);
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  // warp per row: bf16(x - mu) and its norm
  auto pack_row = [&](const float* __restrict__ m, const float* __restrict__ cc, __nv_bfloat16* __restrict__ pk, float* __restrict__ nrm, int i) {
    const long long o = (row0 + i) * H + h * hd;
    __nv_bfloat16* dst = pk + (row0 + i) * 2 * H + h * W;
    float n = 0.f;
    for (int k = lane; k < W; k += 32) {
      const float x = k < hd ? m[o + k] : sqrtf(fmaxf(cc[o + k - hd], WF_CLAMP));
      const __nv_bfloat16 e = __float2bfloat16(x - mu[k]);
      dst[k] = e;
      const float f = __bfloat162float(e);
      n = fmaf(f, f, n);
    }
    n = warp_sum(n);
    if (lane == 0) nrm[(long long)z * L + i] = n;
  };
  for (int i = warp; i < L; i += 8) pack_row(mq, cq, xp, nq, i);
  for (int j = warp; j < L; j += 8) {
    pack_row(mk, ck, yp, nk, j);
    const long long o = (row0 + j) * H + h * hd;
    for (int k = lane; k < hd; k += 32) {
      mvb[o + k] = __float2bfloat16(mv[o + k] - nu[k]);
      cvb[o + k] = __float2bfloat16(cv[o + k] - nu[hd + k]);
    }
  }
  if (h == 0 && tid == 0) first[b] = fmin;
}

// backward operands: bf16 dmctx / dcctx, delta[z][i] = dmctx . mctx + 2 dcctx . cctx over head h of row i, and the centring's shares
// vm = dmctx . mu_mv, vc = dcctx . mu_cv (one warp per (row, head))
__global__ void __launch_bounds__(256) wflash_delta_kernel(const float* __restrict__ mctx, const float* __restrict__ cctx, const float* __restrict__ dm,
                                                           const float* __restrict__ dc, const float* __restrict__ vmu, __nv_bfloat16* __restrict__ dmb,
                                                           __nv_bfloat16* __restrict__ dcb, float* __restrict__ delta, float* __restrict__ vm,
                                                           float* __restrict__ vc, int M, int L, int H, int nh) {
  const int lane = threadIdx.x & 31, hd = H / nh;
  const long long n = (long long)M * nh;
  for (long long w = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); w < n; w += (long long)gridDim.x * 8) {
    const long long r = w / nh;
    const int h = (int)(w - r * nh);
    const long long o = r * H + h * hd;
    const long long b = r / L, i = r - b * L;
    const float* nu = vmu + (b * nh + h) * 2 * hd;
    float s = 0.f, sm = 0.f, sc = 0.f;
    for (int k = lane; k < hd; k += 32) {
      const float x = dm[o + k], y = dc[o + k];
      s = fmaf(x, mctx[o + k], s);
      s = fmaf(2.f * y, cctx[o + k], s);
      sm = fmaf(x, nu[k], sm);
      sc = fmaf(y, nu[hd + k], sc);
      dmb[o + k] = __float2bfloat16(x);
      dcb[o + k] = __float2bfloat16(y);
    }
    s = warp_sum(s);
    sm = warp_sum(sm);
    sc = warp_sum(sc);
    if (lane == 0) {
      delta[(b * nh + h) * L + i] = s;
      vm[(b * nh + h) * L + i] = sm;
      vc[(b * nh + h) * L + i] = sc;
    }
  }
}

// scores of keys jb .. jb+31 for query row i from the dot products <x'_i, y'_j> in v: keys >= L never count; key j counts when
// key_ids > 0 and j <= i; a row with no valid key (uni) scores 0 at every key < L (float32(s + mask) is the mask for all of them)
__device__ __forceinline__ void wscore32(float (&v)[32], int i, int jb, float ni, bool uni, const float* __restrict__ nk, const int* __restrict__ kid,
                                         const WFlashArgs& a) {
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    const int j = jb + k;
    if (j >= a.f.L) v[k] = -INFINITY;
    else if (uni) v[k] = 0.f;
    else if (j > i || __ldg(kid + j) <= 0) v[k] = -INFINITY;
    else v[k] = (2.f * v[k] - (ni + __ldg(nk + j))) * a.scale;
  }
}

__global__ void __launch_bounds__(FT, 1) wflash_fwd_kernel(const __grid_constant__ CUtensorMap tx, const __grid_constant__ CUtensorMap ty,
                                                           const __grid_constant__ CUtensorMap tmv, const __grid_constant__ CUtensorMap tcv,
                                                           WFlashArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const int ks2 = a.ks2, SX = ks2 * BOX, SS = SX + 2 * BOX;   // one stage: Y', mv, cv tiles
  uint8_t* sX = align1024(smem_raw);
  uint8_t* sS = sX + SX;                 // [2] stages
  uint8_t* sP = sS + 2 * SS;             // P~   [128 queries][128 keys]
  uint8_t* sP2 = sP + 2 * BOX;           // P~^2
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP2 + 2 * BOX);
  uint64_t *q_full = bars, *kv_full = bars + 1, *s_bar = bars + 3, *pv_bar = bars + 4;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 5);
  const int tid = threadIdx.x, warp = tid >> 5, L = a.f.L, hd = a.f.hd;
  const int z = blockIdx.x, b = z / a.f.nh, h = z - b * a.f.nh;
  const int nt = (L + FT - 1) / FT, qt = nt - 1 - blockIdx.y, q0 = qt * FT;
  const int fb = __ldg(a.first + b);
  const int nkt = q0 < fb ? nt : qt + 1;
  const int* kid = a.f.key_ids + (long long)b * L;
  const float* nk = a.nk + (long long)z * L;

  if (tid == 0) {
    tc::tma_prefetch_desc(&tx); tc::tma_prefetch_desc(&ty); tc::tma_prefetch_desc(&tmv); tc::tma_prefetch_desc(&tcv);
    for (int i = 0; i < 5; ++i) tc::mbar_init(bars + i, 1);
    tc::fence_barrier_init();
  }
  if (warp == 0) tc::tmem_alloc<256>(tslot);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t lane_off = (uint32_t)(32 * warp) << 16;
  const uint32_t tS = *tslot, tOm = tS + 128, tOc = tS + 192;

  auto load_kv = [&](int t) {
    uint8_t* st = sS + (t & 1) * SS;
    uint64_t* bar = kv_full + (t & 1);
    tc::mbar_arrive_expect_tx(bar, SS);
    load_tile(st, &ty, ks2, t * FT, h, b, bar);
    load_tile(st + SX, &tmv, 1, t * FT, h, b, bar);
    load_tile(st + SX + BOX, &tcv, 1, t * FT, h, b, bar);
  };
  if (tid == 0) {
    tc::mbar_arrive_expect_tx(q_full, SX);
    load_tile(sX, &tx, ks2, q0, h, b, q_full);
    load_kv(0);
    if (nkt > 1) load_kv(1);
    tc::mbar_wait(q_full, 0);
    tc::mbar_wait(kv_full, 0);
    tc::tc_fence_after();
    mma_kk(tS, sX, sS, 2 * hd);
    tc::mma_commit(s_bar);
  }
  __syncwarp();

  const int i = q0 + tid;
  const bool row_ok = i < L, uni = i < fb;
  const float ni = row_ok ? __ldg(a.nq + (long long)z * L + i) : 0.f;
  const unsigned long long drow = a.f.drop.base + (unsigned long long)z * L + i;
  float m_run = -INFINITY, l_run = 0.f, l1 = 0.f, l2 = 0.f;   // l1 = sum P~, l2 = sum P~^2 (running, unnormalised): the centring's share
  for (int t = 0; t < nkt; ++t) {
    const int j0 = t * FT;
    tc::mbar_wait(s_bar, t & 1);
    tc::tc_fence_after();
    float mt = -INFINITY;
    for (int c0 = 0; c0 < FT; c0 += 32) {
      float v[32];
      tc::tmem_ld32(tS + lane_off + c0, v);
      wscore32(v, i, j0 + c0, ni, uni, nk, kid, a);
#pragma unroll
      for (int k = 0; k < 32; ++k) mt = fmaxf(mt, v[k]);
    }
    const float m_new = fmaxf(m_run, mt), alpha = m_new == -INFINITY ? 1.f : exp2f((m_run - m_new) * LOG2E);
    m_run = m_new;
    if (t > 0) {                                  // the products of the previous tile are done: P~ buffers free, O stable -> rescale O
      tc::mbar_wait(pv_bar, (t - 1) & 1);
      tc::tc_fence_after();
      if (__any_sync(0xffffffffu, alpha != 1.f)) {
        const float a2 = alpha * alpha;
        for (int c0 = 0; c0 < 128; c0 += 32) {    // O_m (64 columns) then O_c
          float v[32];
          tc::tmem_ld32(tOm + lane_off + c0, v);
          const float f = c0 < 64 ? alpha : a2;
          uint32_t u[32];
#pragma unroll
          for (int k = 0; k < 32; ++k) u[k] = __float_as_uint(v[k] * f);
          tc::tmem_st32(tOm + lane_off + c0, u);
        }
        tc::tmem_st_wait();
      }
    }
    float ls = 0.f, s1 = 0.f, s2 = 0.f;
    for (int c0 = 0; c0 < FT; c0 += 32) {
      float v[32], mv[32], w[32];
      tc::tmem_ld32(tS + lane_off + c0, v);
      wscore32(v, i, j0 + c0, ni, uni, nk, kid, a);
      drop32(mv, i, j0 + c0, row_ok, drow, a.f);
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const float p = v[k] == -INFINITY ? 0.f : exp2f((v[k] - m_new) * LOG2E);
        ls += p;
        v[k] = p * mv[k];
        w[k] = v[k] * v[k];
        s1 += v[k];
        s2 += w[k];
      }
      st_row32(sP, tid, c0, v);
      st_row32(sP2, tid, c0, w);
    }
    l_run = l_run * alpha + ls;
    l1 = l1 * alpha + s1;
    l2 = l2 * alpha * alpha + s2;
    tc::fence_proxy_async();
    tc::tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc::tc_fence_after();
      const uint8_t* st = sS + (t & 1) * SS;
      mma_xn(tOm, sP, 0, st + SX, 1, t > 0);
      mma_xn(tOc, sP2, 0, st + SX + BOX, 1, t > 0);
      tc::mma_commit(pv_bar);
      if (t + 1 < nkt) {
        tc::mbar_wait(kv_full + ((t + 1) & 1), ((t + 1) >> 1) & 1);
        tc::tc_fence_after();
        mma_kk(tS, sX, sS + ((t + 1) & 1) * SS, 2 * hd);
        tc::mma_commit(s_bar);
      }
      if (t + 2 < nkt) {                          // stage t & 1 is free once the products of tile t completed
        tc::mbar_wait(pv_bar, t & 1);
        load_kv(t + 2);
      }
    }
    __syncwarp();
  }
  tc::mbar_wait(pv_bar, (nkt - 1) & 1);
  tc::tc_fence_after();
  const long long grow = (long long)b * L + i;
  const float inv = 1.f / l_run;
  // mctx = (O_m + l1 mu_mv) / l, cctx = (O_c + l2 mu_cv) / l^2: the values were centred on mu before rounding to bf16
  const float* nu = a.vmu + (long long)z * 2 * hd;
  for (int c0 = 0; c0 < 128; c0 += 32) {
    float v[32];
    tc::tmem_ld32(tOm + lane_off + c0, v);
    const int cm = c0 & 63;
    if (!row_ok || cm >= hd) continue;
    const bool cov = c0 >= 64;
    float* out = (cov ? a.cctx : a.mctx) + grow * a.f.H + h * hd + cm;
    const float* mu = nu + (cov ? hd : 0) + cm;
    const float ls = cov ? l2 : l1, sc = cov ? inv * inv : inv;
#pragma unroll
    for (int k = 0; k < 32; k += 4)
      if (cm + k < hd)
        *reinterpret_cast<float4*>(out + k) = make_float4((v[k] + ls * mu[k]) * sc, (v[k + 1] + ls * mu[k + 1]) * sc,
                                                          (v[k + 2] + ls * mu[k + 2]) * sc, (v[k + 3] + ls * mu[k + 3]) * sc);
  }
  if (row_ok) {
    a.stat[((long long)z * L + i) * 2] = uni ? WF_MASK : m_run;
    a.stat[((long long)z * L + i) * 2 + 1] = inv;
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc<256>(tS);
}

// MODE 0 (dq): CTA per query tile, walks key tiles.  MODE 1 (dk) / 2 (dv): CTA per key tile, walks query tiles.
template <int MODE>
__global__ void __launch_bounds__(FT, 1) wflash_bwd_kernel(const __grid_constant__ CUtensorMap tx, const __grid_constant__ CUtensorMap ty,
                                                           const __grid_constant__ CUtensorMap tmv, const __grid_constant__ CUtensorMap tcv,
                                                           const __grid_constant__ CUtensorMap tdm, const __grid_constant__ CUtensorMap tdc,
                                                           WFlashArgs a) {
  constexpr uint32_t NCOL = MODE == 2 ? 256 : 512;
  extern __shared__ uint8_t smem_raw[];
  const int ks2 = a.ks2, SX = ks2 * BOX, SS = SX + 2 * BOX, NS = a.f.nstage;
  uint8_t* sO = align1024(smem_raw);     // the CTA's own tiles: {X', dmctx, dcctx} (dq) or {Y', mv, cv} (dk, dv)
  uint8_t* sS = sO + SS;                 // [NS] stages of the walked side: {Y', mv, cv} (dq) or {X', dmctx, dcctx} (dk, dv)
  uint8_t* sW = sS + NS * SS;            // dS (dq, dk) or P~ and P~^2 (dv), bf16 [128 queries][128 keys]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sW + (MODE == 2 ? 4 : 2) * BOX);
  uint64_t *own_full = bars, *st_full = bars + 1, *sd_bar = bars + 3, *mm_bar = bars + 4;
  uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 5);
  const int tid = threadIdx.x, warp = tid >> 5, L = a.f.L, hd = a.f.hd, H = a.f.H;
  const int z = blockIdx.x, b = z / a.f.nh, h = z - b * a.f.nh;
  const int nt = (L + FT - 1) / FT, own = MODE == 0 ? nt - 1 - blockIdx.y : blockIdx.y;
  const int fb = __ldg(a.first + b);
  // walked tiles: dq the causal key tiles (all of them when the query tile holds rows with no valid key); dk / dv the query tiles
  // 0 .. nu-1 that hold such rows, then the causal ones own .. nt-1
  const int nu = MODE == 0 ? 0 : min(own, (fb + FT - 1) / FT);
  const int nw = MODE == 0 ? (own * FT < fb ? nt : own + 1) : nu + nt - own;
  auto walked = [&](int n) { return MODE == 0 ? n : (n < nu ? n : own + n - nu); };
  const int* kid = a.f.key_ids + (long long)b * L;
  const float* nk = a.nk + (long long)z * L;

  if (tid == 0) {
    tc::tma_prefetch_desc(&tx); tc::tma_prefetch_desc(&ty); tc::tma_prefetch_desc(&tmv); tc::tma_prefetch_desc(&tcv);
    tc::tma_prefetch_desc(&tdm); tc::tma_prefetch_desc(&tdc);
    for (int i = 0; i < 5; ++i) tc::mbar_init(bars + i, 1);
    tc::fence_barrier_init();
  }
  if (warp == 0) tc::tmem_alloc<NCOL>(tslot);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t lane_off = (uint32_t)(32 * warp) << 16;
  const uint32_t tS = *tslot, tdPm = tS + 128, tdPc = tS + 256, tAcc = tS + 384, tMV = tS + 128, tCV = tS + 192;

  auto load_set = [&](uint8_t* dst, bool query_side, int tile, uint64_t* bar) {
    tc::mbar_arrive_expect_tx(bar, SS);
    load_tile(dst, query_side ? &tx : &ty, ks2, tile * FT, h, b, bar);
    load_tile(dst + SX, query_side ? &tdm : &tmv, 1, tile * FT, h, b, bar);
    load_tile(dst + SX + BOX, query_side ? &tdc : &tcv, 1, tile * FT, h, b, bar);
  };
  auto load_walk = [&](int n) { load_set(sS + (n % NS) * SS, MODE != 0, walked(n), st_full + n % NS); };
  auto issue_sdp = [&](int n) {
    uint8_t* w = sS + (n % NS) * SS;
    const uint8_t* q = MODE == 0 ? sO : w;
    const uint8_t* k = MODE == 0 ? w : sO;
    mma_kk(tS, q, k, 2 * hd);
    if (MODE != 2) {
      mma_kk(tdPm, q + SX, k + SX, hd);
      mma_kk(tdPc, q + SX + BOX, k + SX + BOX, hd);
    }
    tc::mma_commit(sd_bar);
  };
  if (tid == 0) {
    load_set(sO, MODE == 0, own, own_full);
    for (int n = 0; n < NS && n < nw; ++n) load_walk(n);
    tc::mbar_wait(own_full, 0);
    tc::mbar_wait(st_full, 0);
    tc::tc_fence_after();
    issue_sdp(0);
  }
  __syncwarp();

  float rsum = 0.f;     // dq: row sum of this query row's dS; dk: column sum of this key's dS
  for (int n = 0; n < nw; ++n) {
    const int qtile = MODE == 0 ? own : walked(n), ktile = MODE == 0 ? walked(n) : own;
    const int i = qtile * FT + tid, j0 = ktile * FT;
    const bool row_ok = i < L, uni = i < fb;
    const long long zi = (long long)z * L + i;
    const float ni = row_ok ? __ldg(a.nq + zi) : 0.f;
    const float mx = (uni || !row_ok) ? 0.f : __ldg(a.stat + 2 * zi), inv = row_ok ? __ldg(a.stat + 2 * zi + 1) : 0.f;
    const float dl = (MODE != 2 && row_ok) ? __ldg(a.delta + zi) : 0.f;
    const float vmi = (MODE != 2 && row_ok) ? __ldg(a.vm + zi) : 0.f, vci = (MODE != 2 && row_ok) ? __ldg(a.vc + zi) : 0.f;
    const unsigned long long drow = a.f.drop.base + (unsigned long long)zi;
    tc::mbar_wait(sd_bar, n & 1);
    tc::tc_fence_after();
    if (n > 0) tc::mbar_wait(mm_bar, (n - 1) & 1);     // the previous products have read sW
    if (MODE == 1 && n > 0) __syncthreads();            // and every thread has read its column of the previous dS
    for (int c0 = 0; c0 < FT; c0 += 32) {
      float v[32], mv[32];
      tc::tmem_ld32(tS + lane_off + c0, v);
      wscore32(v, i, j0 + c0, ni, uni, nk, kid, a);
      drop32(mv, i, j0 + c0, row_ok, drow, a.f);
      if (MODE == 2) {
        float w[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          const float p = (v[k] == -INFINITY || !row_ok) ? 0.f : exp2f((v[k] - mx) * LOG2E) * inv;
          v[k] = p * mv[k];
          w[k] = v[k] * v[k];
        }
        st_row32(sW, tid, c0, v);
        st_row32(sW + 2 * BOX, tid, c0, w);
      } else {
        float dm[32], dc[32];
        tc::tmem_ld32(tdPm + lane_off + c0, dm);
        tc::tmem_ld32(tdPc + lane_off + c0, dc);
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          const float p = (v[k] == -INFINITY || !row_ok) ? 0.f : exp2f((v[k] - mx) * LOG2E) * inv;
          const float dp = mv[k] * ((dm[k] + vmi) + 2.f * p * mv[k] * (dc[k] + vci));
          v[k] = p * (dp - dl) * a.scale;
          if (MODE == 0) rsum += __bfloat162float(__float2bfloat16(v[k]));
        }
        st_row32(sW, tid, c0, v);
      }
    }
    tc::fence_proxy_async();
    tc::tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc::tc_fence_after();
      const uint8_t* w = sS + (n % NS) * SS;
      if (MODE == 0) mma_xn(tAcc, sW, 0, w, ks2, n > 0);          // A += dS Y'
      if (MODE == 1) mma_xn(tAcc, sW, 1, w, ks2, n > 0);          // B += dS^T X'
      if (MODE == 2) {
        mma_xn(tMV, sW, 1, w + SX, 1, n > 0);                     // dmv += P~^T dmctx
        mma_xn(tCV, sW + 2 * BOX, 1, w + SX + BOX, 1, n > 0);     // dcv += (P~^2)^T dcctx
      }
      tc::mma_commit(mm_bar);
      if (NS == 1) {
        tc::mbar_wait(mm_bar, n & 1);
        if (n + 1 < nw) load_walk(n + 1);
      }
      if (n + 1 < nw) {
        tc::mbar_wait(st_full + (n + 1) % NS, ((n + 1) / NS) & 1);
        tc::tc_fence_after();
        issue_sdp(n + 1);
      }
      if (NS == 2) {
        tc::mbar_wait(mm_bar, n & 1);
        if (n + 2 < nw) load_walk(n + 2);
      }
    }
    __syncwarp();
    if (MODE == 1) {                                    // column tid of the bf16 dS tile, in row order
      const uint8_t* col = sW + (tid >> 6) * BOX + (tid & 7) * 2;
      const int cc = (tid & 63) >> 3;
      for (int r = 0; r < FT; ++r)
        rsum += __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(col + r * 128 + ((cc ^ (r & 7)) << 4)));
    }
  }
  tc::mbar_wait(mm_bar, (nw - 1) & 1);
  tc::tc_fence_after();
  const int r = own * FT + tid;
  const long long grow = (long long)b * L + r;
  const bool ok = r < L;
  if (MODE == 2) {
    store_acc(tMV + lane_off, ok ? a.dmv + grow * H : nullptr, h * hd, hd, 1, 1.f);
    store_acc(tCV + lane_off, ok ? a.dcv + grow * H : nullptr, h * hd, hd, 1, 1.f);
  } else {
    // dx = 2 sum G (y' - x') split into the mean half (d mean = 2 e) and the sqrt-cov half (d cov = e / sqrt(cov), -rs below the clamp)
    const __nv_bfloat16* pk = (MODE == 0 ? a.xp : a.yp) + grow * 2 * H + h * 2 * hd;
    const float* cov = (MODE == 0 ? a.cq : a.ck) + grow * H + h * hd;
    float* dmean = (MODE == 0 ? a.dmq : a.dmk) + grow * H + h * hd;
    float* dcov = (MODE == 0 ? a.dcq : a.dck) + grow * H + h * hd;
    for (int c0 = 0; c0 < 64 * ks2; c0 += 32) {
      float v[32];
      tc::tmem_ld32(tAcc + lane_off + c0, v);
      if (!ok || c0 >= 2 * hd) continue;
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const int c = c0 + k;
        const float e = v[k] - rsum * __bfloat162float(pk[c]);
        if (c < hd) {
          dmean[c] = 2.f * e;
        } else {
          const float cv = cov[c - hd];
          dcov[c - hd] = cv > WF_CLAMP ? e / sqrtf(cv) : -rsum;
        }
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc<NCOL>(tS);
}

size_t wfwd_smem(int ks2) { return 1024 + (size_t)(3 * ks2 + 8) * BOX + 64; }
size_t wbwd_smem(int ks2, int ns, int mode) { return 1024 + (size_t)(1 + ns) * (ks2 + 2) * BOX + (mode == 2 ? 4 : 2) * BOX + 64; }

}  // namespace

// scratch of adt_wattention_flash_fwd / _bwd: bf16 X', Y' [M][2H], mv, cv [M][H] (+ dmctx, dcctx), fp32 norms [M nh] x 2, value means
// [B nh][2hd] (+ delta, vm, vc [M nh]),
// int first valid key [B].  Every bf16 array is a multiple of 32 bytes, so each one starts 16-byte aligned.
long long wflash_scratch_bytes(int B, int L, int H, int nh, bool bwd) {
  const long long M = (long long)B * L;
  return M * H * 12 + M * nh * 8 + 8LL * B * H + 4LL * B + (bwd ? M * H * 4 + M * nh * 12 : 0);
}

int wattn_flash(const adt_wattention_args* w, const DropDesc& d, bool bwd, cudaStream_t s) {
  const int B = w->B, L = w->L, H = w->H, nh = w->nh, hd = H / nh;
  const long long M = (long long)B * L;
  uint8_t* p = static_cast<uint8_t*>(w->tc_scratch);
  auto take = [&](long long bytes) { uint8_t* r = p; p += bytes; return r; };
  __nv_bfloat16* xp = reinterpret_cast<__nv_bfloat16*>(take(M * H * 4));
  __nv_bfloat16* yp = reinterpret_cast<__nv_bfloat16*>(take(M * H * 4));
  __nv_bfloat16* mvb = reinterpret_cast<__nv_bfloat16*>(take(M * H * 2));
  __nv_bfloat16* cvb = reinterpret_cast<__nv_bfloat16*>(take(M * H * 2));
  __nv_bfloat16* dmb = bwd ? reinterpret_cast<__nv_bfloat16*>(take(M * H * 2)) : nullptr;
  __nv_bfloat16* dcb = bwd ? reinterpret_cast<__nv_bfloat16*>(take(M * H * 2)) : nullptr;
  float* nq = reinterpret_cast<float*>(take(M * nh * 4));
  float* nk = reinterpret_cast<float*>(take(M * nh * 4));
  float* vmu = reinterpret_cast<float*>(take(8LL * B * H));
  float* delta = bwd ? reinterpret_cast<float*>(take(M * nh * 4)) : nullptr;
  float* vm = bwd ? reinterpret_cast<float*>(take(M * nh * 4)) : nullptr;
  float* vc = bwd ? reinterpret_cast<float*>(take(M * nh * 4)) : nullptr;
  int* first = reinterpret_cast<int*>(take(4LL * B));

  wflash_prep_kernel<<<B * nh, 256, 0, s>>>(w->mq, w->cq, w->mk, w->ck, w->mv, w->cv, w->key_ids, L, H, nh, xp, yp, mvb, cvb, nq, nk, first, vmu);
  if (bwd) {
    const long long blocks = (M * nh + 7) / 8;
    wflash_delta_kernel<<<(int)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, s>>>(w->mctx_in, w->cctx_in, w->dmctx, w->dcctx, vmu, dmb, dcb, delta, vm, vc,
                                                                                   (int)M, L, H, nh);
  }
  WFlashArgs a;
  memset(&a, 0, sizeof(a));
  a.f.L = L; a.f.H = H; a.f.nh = nh; a.f.hd = hd; a.f.ks = 1; a.f.mask_mode = 1; a.f.key_ids = w->key_ids; a.f.drop = d;
  a.ks2 = (2 * hd + 63) / 64;
  a.f.nstage = a.ks2 == 1 ? 2 : 1;
  a.nq = nq; a.nk = nk; a.first = first; a.stat = w->lse; a.mctx = w->mctx; a.cctx = w->cctx; a.delta = delta;
  a.vmu = vmu; a.vm = vm; a.vc = vc;
  a.cq = w->cq; a.ck = w->ck; a.xp = xp; a.yp = yp;
  a.dmq = w->dmq; a.dcq = w->dcq; a.dmk = w->dmk; a.dck = w->dck; a.dmv = w->dmv; a.dcv = w->dcv;
  a.scale = 1.0f / sqrtf((float)hd);
  CUtensorMap tx, ty, tmv, tcv, tdm, tdc;
  if (head_map(&tx, xp, B, L, 2 * H, nh, 2 * H) || head_map(&ty, yp, B, L, 2 * H, nh, 2 * H) || head_map(&tmv, mvb, B, L, H, nh, H) ||
      head_map(&tcv, cvb, B, L, H, nh, H))
    return ADT_E_CUDA;
  const dim3 grid(B * nh, (L + FT - 1) / FT);
  if (!bwd) {
    const size_t sm = wfwd_smem(a.ks2);
    cudaFuncSetAttribute(wflash_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    wflash_fwd_kernel<<<grid, FT, sm, s>>>(tx, ty, tmv, tcv, a);
  } else {
    if (head_map(&tdm, dmb, B, L, H, nh, H) || head_map(&tdc, dcb, B, L, H, nh, H)) return ADT_E_CUDA;
    const size_t s0 = wbwd_smem(a.ks2, a.f.nstage, 0), s2 = wbwd_smem(a.ks2, a.f.nstage, 2);
    cudaFuncSetAttribute(wflash_bwd_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s0);
    cudaFuncSetAttribute(wflash_bwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s0);
    cudaFuncSetAttribute(wflash_bwd_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s2);
    wflash_bwd_kernel<0><<<grid, FT, s0, s>>>(tx, ty, tmv, tcv, tdm, tdc, a);
    wflash_bwd_kernel<1><<<grid, FT, s0, s>>>(tx, ty, tmv, tcv, tdm, tdc, a);
    wflash_bwd_kernel<2><<<grid, FT, s2, s>>>(tx, ty, tmv, tcv, tdm, tdc, a);
  }
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}

}  // namespace adt
