// STOSA-ADT kernels (SURVEY 8a row a20): Wasserstein self/cross attention over (mean, covariance) streams and the
// BPR + positive-vs-negative loss on elementwise Wasserstein distances.
//   reference: /root/reference/stosa/modules.py:22-43 (distances), :222-275 / :312-361 (attention), stosa/trainer.py:358-391 (loss)
// One CTA per (sequence, head); the key side (mean/sqrt-cov keys, mean/cov values) stays resident in shared memory while the
// CTA walks the query tiles, so each operand is read from HBM exactly once per head.
#pragma once
#include "common.cuh"
#include "kernels_bwd.cuh"

namespace adt {

constexpr int WQT = 32;                       // query rows per tile
constexpr float W_MASK = -4294967296.0f;      // float(-2**32 + 1): additive mask of models.py:229-233
constexpr float W_CLAMP = 1e-24f;             // torch.clamp(cov, min=1e-24) before sqrt (modules.py:24-25,41)

struct WAttnArgs {
  const float *mq, *cq, *mk, *ck, *mv, *cv;   // projected streams [B*L, H]; cov streams are already ELU+1
  float *mctx, *cctx, *lse;                   // contexts [B*L, H], softmax row statistics (max, 1/sum) [B, nh, L, 2]
  const int* key_ids;                         // [B, L]: key j is valid iff key_ids[b][j] > 0 (and j <= i)
  const float *dmctx, *dcctx;                 // backward
  float *dmq, *dcq, *dmk, *dck, *dmv, *dcv;
  int B, L, H, nh;
  float inv_sqrt_hd;
  DropDesc drop;
};

__host__ __device__ inline int wattn_ldk(int hd) { return hd + 4; }
__host__ __device__ inline size_t wattn_smem_floats(int L, int hd, bool bwd) {
  const int ldk = wattn_ldk(hd), lp = (L + 7) & ~7;
  L = (L + 3) & ~3;                                         // keeps every sub-array 16-byte aligned
  size_t n = (size_t)4 * L * ldk + L                        // mk, sk, mv, cv, nk
             + (size_t)2 * WQT * ldk + WQT                  // mq, sq, nq
             + (size_t)WQT * lp;                            // P
  if (bwd) n += (size_t)4 * L * ldk + L                     // accumulators + column sums
                + (size_t)2 * WQT * ldk                     // dmctx, dcctx tiles
                + (size_t)2 * WQT * lp;                     // dropout multipliers, dS
  return n;
}

// loads the key side of head h of sequence b; sk = sqrt(max(ck, 1e-24)); nk = |mk|^2 + sum(ck)
__device__ __forceinline__ void wattn_load_keys(const WAttnArgs& p, int b, int h, int hd, int ldk, float* mk, float* sk, float* mv, float* cv,
                                                float* nk) {
  const int hd4 = hd >> 2;
  for (int t = threadIdx.x; t < p.L * hd4; t += NT) {
    const int j = t / hd4, c = (t - j * hd4) * 4;
    const long long g = ((long long)b * p.L + j) * p.H + h * hd + c;
    st4(mk + j * ldk + c, ld4(p.mk + g));
    const float4 ck = ld4(p.ck + g);
    st4(sk + j * ldk + c, make_float4(sqrtf(fmaxf(ck.x, W_CLAMP)), sqrtf(fmaxf(ck.y, W_CLAMP)), sqrtf(fmaxf(ck.z, W_CLAMP)),
                                      sqrtf(fmaxf(ck.w, W_CLAMP))));
    st4(mv + j * ldk + c, ld4(p.mv + g));
    st4(cv + j * ldk + c, ld4(p.cv + g));
  }
  __syncthreads();
  for (int j = threadIdx.x; j < p.L; j += NT) {
    const long long g = ((long long)b * p.L + j) * p.H + h * hd;
    float m2 = 0.f, cs = 0.f;
    for (int c = 0; c < hd; ++c) {
      const float m = mk[j * ldk + c];
      m2 += m * m;
      cs += p.ck[g + c];
    }
    nk[j] = m2 + cs;
  }
}

// query tile: mq, sq, nq
__device__ __forceinline__ void wattn_load_queries(const WAttnArgs& p, int b, int h, int hd, int ldk, int q0, int nq_rows, float* mq, float* sq,
                                                   float* nq) {
  const int hd4 = hd >> 2;
  for (int t = threadIdx.x; t < nq_rows * hd4; t += NT) {
    const int i = t / hd4, c = (t - i * hd4) * 4;
    const long long g = ((long long)b * p.L + q0 + i) * p.H + h * hd + c;
    st4(mq + i * ldk + c, ld4(p.mq + g));
    const float4 cq = ld4(p.cq + g);
    st4(sq + i * ldk + c, make_float4(sqrtf(fmaxf(cq.x, W_CLAMP)), sqrtf(fmaxf(cq.y, W_CLAMP)), sqrtf(fmaxf(cq.z, W_CLAMP)),
                                      sqrtf(fmaxf(cq.w, W_CLAMP))));
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nq_rows; i += NT) {
    const long long g = ((long long)b * p.L + q0 + i) * p.H + h * hd;
    float m2 = 0.f, cs = 0.f;
    for (int c = 0; c < hd; ++c) {
      const float m = mq[i * ldk + c];
      m2 += m * m;
      cs += p.cq[g + c];
    }
    nq[i] = m2 + cs;
  }
  __syncthreads();
}

// masked, scaled scores of the tile into P (modules.py:30-43 then :248-249)
__device__ __forceinline__ void wattn_scores(const WAttnArgs& p, int b, int hd, int ldk, int lp, int q0, int nq_rows, const float* mq,
                                             const float* sq, const float* nq, const float* mk, const float* sk, const float* nk, float* P) {
  const int* ids = p.key_ids + (long long)b * p.L;
  for (int t = threadIdx.x; t < nq_rows * p.L; t += NT) {
    const int i = t / p.L, j = t - i * p.L;
    float dm = 0.f, dc = 0.f;
    for (int c = 0; c < hd; c += 4) {
      const float4 a = ld4(mq + i * ldk + c), k = ld4(mk + j * ldk + c), sa = ld4(sq + i * ldk + c), sb = ld4(sk + j * ldk + c);
      dm += a.x * k.x + a.y * k.y + a.z * k.z + a.w * k.w;
      dc += sa.x * sb.x + sa.y * sb.y + sa.z * sb.z + sa.w * sb.w;
    }
    const float dist = (nq[i] + nk[j]) - 2.f * (dm + dc);
    const bool valid = ids[j] > 0 && j <= q0 + i;
    P[i * lp + j] = -dist * p.inv_sqrt_hd + (valid ? 0.f : W_MASK);
  }
  __syncthreads();
}

// row softmax (warp per row).  FWD computes and stores (max, 1/sum) per row; BWD re-uses them.  They are kept apart because a
// fully masked row has max = -2^32, where max + log(sum) would lose the log(sum) term in fp32.
template <bool FWD>
__device__ __forceinline__ void wattn_softmax(const WAttnArgs& p, int b, int h, int lp, int q0, int nq_rows, float* P) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = warp; i < nq_rows; i += NT / 32) {
    float* row = P + i * lp;
    const long long li = (((long long)b * p.nh + h) * p.L + q0 + i) * 2;
    float mx, inv;
    if (FWD) {
      mx = -INFINITY;
      for (int j = lane; j < p.L; j += 32) mx = fmaxf(mx, row[j]);
      mx = warp_max(mx);
      float s = 0.f;
      for (int j = lane; j < p.L; j += 32) s += expf(row[j] - mx);
      s = warp_sum(s);
      inv = 1.f / s;
      if (lane == 0) { p.lse[li] = mx; p.lse[li + 1] = inv; }
    } else {
      mx = p.lse[li];
      inv = p.lse[li + 1];
    }
    for (int j = lane; j < p.L; j += 32) row[j] = expf(row[j] - mx) * inv;
    for (int j = p.L + lane; j < lp; j += 32) row[j] = 0.f;
  }
  __syncthreads();
}

// dropout multipliers of the tile (1/(1-p) or 0) ; identity when disabled
__device__ __forceinline__ void wattn_dropmask(const WAttnArgs& p, int b, int h, int lp, int q0, int nq_rows, float* Mk) {
  const int lp8 = lp >> 3;
  for (int t = threadIdx.x; t < nq_rows * lp8; t += NT) {
    const int i = t / lp8, g = t - i * lp8;
    float m[8];
    if (p.drop.enabled) {
      drop_mul8_attn(p.drop, p.drop.base + ((unsigned long long)b * p.nh + h) * p.L + q0 + i, lp8, g, m);
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) m[k] = 1.f;
    }
    st4(Mk + i * lp + g * 8, make_float4(m[0], m[1], m[2], m[3]));
    st4(Mk + i * lp + g * 8 + 4, make_float4(m[4], m[5], m[6], m[7]));
  }
  __syncthreads();
}

// forward: contexts mean = P~ mv, cov = P~^2 cv  (modules.py:251-254)
__global__ void __launch_bounds__(NT) wattn_fwd_kernel(WAttnArgs p) {
  extern __shared__ __align__(16) float sm[];
  const int hd = p.H / p.nh, ldk = wattn_ldk(hd), lp = (p.L + 7) & ~7, hd4 = hd >> 2;
  float* mk = sm;
  float* sk = mk + p.L * ldk;
  float* mv = sk + p.L * ldk;
  float* cv = mv + p.L * ldk;
  float* nk = cv + p.L * ldk;
  float* mq = nk + ((p.L + 3) & ~3);
  float* sq = mq + WQT * ldk;
  float* nq = sq + WQT * ldk;
  float* P = nq + WQT;
  for (int bh = blockIdx.x; bh < p.B * p.nh; bh += gridDim.x) {
    const int b = bh / p.nh, h = bh - b * p.nh;
    __syncthreads();
    wattn_load_keys(p, b, h, hd, ldk, mk, sk, mv, cv, nk);
    for (int q0 = 0; q0 < p.L; q0 += WQT) {
      const int rows = min(WQT, p.L - q0);
      wattn_load_queries(p, b, h, hd, ldk, q0, rows, mq, sq, nq);
      wattn_scores(p, b, hd, ldk, lp, q0, rows, mq, sq, nq, mk, sk, nk, P);
      wattn_softmax<true>(p, b, h, lp, q0, rows, P);
      if (p.drop.enabled) {
        const int lp8 = lp >> 3;
        for (int t = threadIdx.x; t < rows * lp8; t += NT) {
          const int i = t / lp8, g = t - i * lp8;
          float m[8];
          drop_mul8_attn(p.drop, p.drop.base + ((unsigned long long)b * p.nh + h) * p.L + q0 + i, lp8, g, m);
          float* r = P + i * lp + g * 8;
#pragma unroll
          for (int k = 0; k < 8; ++k) r[k] *= m[k];
        }
        __syncthreads();
      }
      for (int t = threadIdx.x; t < rows * hd4; t += NT) {
        const int i = t / hd4, c = (t - i * hd4) * 4;
        float4 am = make_float4(0.f, 0.f, 0.f, 0.f), ac = am;
        for (int j = 0; j < p.L; ++j) {
          const float w = P[i * lp + j], w2 = w * w;
          const float4 m = ld4(mv + j * ldk + c), v = ld4(cv + j * ldk + c);
          am.x += w * m.x; am.y += w * m.y; am.z += w * m.z; am.w += w * m.w;
          ac.x += w2 * v.x; ac.y += w2 * v.y; ac.z += w2 * v.z; ac.w += w2 * v.w;
        }
        const long long g = ((long long)b * p.L + q0 + i) * p.H + h * hd + c;
        st4(p.mctx + g, am);
        st4(p.cctx + g, ac);
      }
      __syncthreads();
    }
  }
}

// backward of the above w.r.t. all six projected streams
__global__ void __launch_bounds__(NT) wattn_bwd_kernel(WAttnArgs p) {
  extern __shared__ __align__(16) float sm[];
  const int hd = p.H / p.nh, ldk = wattn_ldk(hd), lp = (p.L + 7) & ~7, hd4 = hd >> 2;
  float* mk = sm;
  float* sk = mk + p.L * ldk;
  float* mv = sk + p.L * ldk;
  float* cv = mv + p.L * ldk;
  float* nk = cv + p.L * ldk;
  float* mq = nk + ((p.L + 3) & ~3);
  float* sq = mq + WQT * ldk;
  float* nq = sq + WQT * ldk;
  float* P = nq + WQT;
  float* amk = P + WQT * lp;       // accumulators: sum_i G_ij (mq_i - mk_j), sum_i G_ij (sq_i - sk_j), sum_i P~ dmctx, sum_i P~^2 dcctx
  float* ask = amk + p.L * ldk;
  float* amv = ask + p.L * ldk;
  float* acv = amv + p.L * ldk;
  float* cs = acv + p.L * ldk;     // column sums of G
  float* dm = cs + ((p.L + 3) & ~3);   // dmctx tile
  float* dc = dm + WQT * ldk;      // dcctx tile
  float* Mk = dc + WQT * ldk;      // dropout multipliers
  float* G = Mk + WQT * lp;        // dP then dS * inv_sqrt_hd
  for (int bh = blockIdx.x; bh < p.B * p.nh; bh += gridDim.x) {
    const int b = bh / p.nh, h = bh - b * p.nh;
    __syncthreads();
    wattn_load_keys(p, b, h, hd, ldk, mk, sk, mv, cv, nk);
    for (int t = threadIdx.x; t < 4 * p.L * ldk + p.L; t += NT) amk[t] = 0.f;   // four accumulators + cs (contiguous)
    __syncthreads();
    for (int q0 = 0; q0 < p.L; q0 += WQT) {
      const int rows = min(WQT, p.L - q0);
      for (int t = threadIdx.x; t < rows * hd4; t += NT) {
        const int i = t / hd4, c = (t - i * hd4) * 4;
        const long long g = ((long long)b * p.L + q0 + i) * p.H + h * hd + c;
        st4(dm + i * ldk + c, ld4(p.dmctx + g));
        st4(dc + i * ldk + c, ld4(p.dcctx + g));
      }
      wattn_load_queries(p, b, h, hd, ldk, q0, rows, mq, sq, nq);
      wattn_scores(p, b, hd, ldk, lp, q0, rows, mq, sq, nq, mk, sk, nk, P);
      wattn_softmax<false>(p, b, h, lp, q0, rows, P);
      wattn_dropmask(p, b, h, lp, q0, rows, Mk);
      // dP_ij = (dmctx_i . mv_j + 2 P~_ij dcctx_i . cv_j) * m_ij
      for (int t = threadIdx.x; t < rows * p.L; t += NT) {
        const int i = t / p.L, j = t - i * p.L;
        float a = 0.f, c2 = 0.f;
        for (int c = 0; c < hd; c += 4) {
          const float4 x = ld4(dm + i * ldk + c), m = ld4(mv + j * ldk + c), y = ld4(dc + i * ldk + c), v = ld4(cv + j * ldk + c);
          a += x.x * m.x + x.y * m.y + x.z * m.z + x.w * m.w;
          c2 += y.x * v.x + y.y * v.y + y.z * v.z + y.w * v.w;
        }
        const float mlt = Mk[i * lp + j], pt = P[i * lp + j] * mlt;
        G[i * lp + j] = (a + 2.f * pt * c2) * mlt;
      }
      __syncthreads();
      // dS = P (dP - sum_j dP P) ; G <- dS / sqrt(hd)
      {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        for (int i = warp; i < rows; i += NT / 32) {
          float d = 0.f;
          for (int j = lane; j < p.L; j += 32) d += G[i * lp + j] * P[i * lp + j];
          d = warp_sum(d);
          for (int j = lane; j < p.L; j += 32) G[i * lp + j] = P[i * lp + j] * (G[i * lp + j] - d) * p.inv_sqrt_hd;
        }
      }
      __syncthreads();
      // query-side gradients: d score_ij / d mq_i = 2 (mk_j - mq_i) / sqrt(hd), d score_ij / d cq_i = (sk_j - sq_i) / (sq_i sqrt(hd)).
      // The differences are formed before the sum over j: every stream shares an offset (~1 for sqrt-cov at initialisation) that the
      // expanded form sum_j G_ij k_j - (sum_j G_ij) q_i would cancel only after fp32 rounding, at ~100x the gradient's own size.
      for (int t = threadIdx.x; t < rows * hd4; t += NT) {
        const int i = t / hd4, c = (t - i * hd4) * 4;
        const float4 q = ld4(mq + i * ldk + c), s = ld4(sq + i * ldk + c);
        float4 am = make_float4(0.f, 0.f, 0.f, 0.f), as = am;
        float rs = 0.f;
        for (int j = 0; j < p.L; ++j) {
          const float g = G[i * lp + j];
          const float4 k = ld4(mk + j * ldk + c), sj = ld4(sk + j * ldk + c);
          am.x += g * (k.x - q.x); am.y += g * (k.y - q.y); am.z += g * (k.z - q.z); am.w += g * (k.w - q.w);
          as.x += g * (sj.x - s.x); as.y += g * (sj.y - s.y); as.z += g * (sj.z - s.z); as.w += g * (sj.w - s.w);
          rs += g;
        }
        const long long go = ((long long)b * p.L + q0 + i) * p.H + h * hd + c;
        const float4 cq = ld4(p.cq + go);
        st4(p.dmq + go, make_float4(2.f * am.x, 2.f * am.y, 2.f * am.z, 2.f * am.w));
        st4(p.dcq + go, make_float4(cq.x > W_CLAMP ? as.x / s.x : -rs, cq.y > W_CLAMP ? as.y / s.y : -rs, cq.z > W_CLAMP ? as.z / s.z : -rs,
                                    cq.w > W_CLAMP ? as.w / s.w : -rs));
      }
      // key-side accumulators (each (j, c) owned by one thread across tiles)
      for (int t = threadIdx.x; t < p.L * hd4; t += NT) {
        const int j = t / hd4, c = (t - j * hd4) * 4;
        // a1 = sum_i G_ij (mq_i - mk_j), a2 = sum_i G_ij (sq_i - sk_j): differences before the sum, as on the query side
        const float4 k = ld4(mk + j * ldk + c), sk4 = ld4(sk + j * ldk + c);
        float4 a1 = ld4(amk + j * ldk + c), a2 = ld4(ask + j * ldk + c), a3 = ld4(amv + j * ldk + c), a4 = ld4(acv + j * ldk + c);
        float s = 0.f;
        for (int i = 0; i < rows; ++i) {
          const float g = G[i * lp + j], pt = P[i * lp + j] * Mk[i * lp + j], pt2 = pt * pt;
          const float4 q = ld4(mq + i * ldk + c), sq4 = ld4(sq + i * ldk + c), x = ld4(dm + i * ldk + c), y = ld4(dc + i * ldk + c);
          a1.x += g * (q.x - k.x); a1.y += g * (q.y - k.y); a1.z += g * (q.z - k.z); a1.w += g * (q.w - k.w);
          a2.x += g * (sq4.x - sk4.x); a2.y += g * (sq4.y - sk4.y); a2.z += g * (sq4.z - sk4.z); a2.w += g * (sq4.w - sk4.w);
          a3.x += pt * x.x; a3.y += pt * x.y; a3.z += pt * x.z; a3.w += pt * x.w;
          a4.x += pt2 * y.x; a4.y += pt2 * y.y; a4.z += pt2 * y.z; a4.w += pt2 * y.w;
          s += g;
        }
        st4(amk + j * ldk + c, a1); st4(ask + j * ldk + c, a2); st4(amv + j * ldk + c, a3); st4(acv + j * ldk + c, a4);
        if (c == 0) cs[j] += s;
      }
      __syncthreads();
    }
    for (int t = threadIdx.x; t < p.L * hd4; t += NT) {
      const int j = t / hd4, c = (t - j * hd4) * 4;
      const long long go = ((long long)b * p.L + j) * p.H + h * hd + c;
      const float s = cs[j];
      const float4 a1 = ld4(amk + j * ldk + c), a2 = ld4(ask + j * ldk + c), sk4 = ld4(sk + j * ldk + c), ck = ld4(p.ck + go);
      st4(p.dmk + go, make_float4(2.f * a1.x, 2.f * a1.y, 2.f * a1.z, 2.f * a1.w));
      st4(p.dck + go, make_float4(ck.x > W_CLAMP ? a2.x / sk4.x : -s, ck.y > W_CLAMP ? a2.y / sk4.y : -s, ck.z > W_CLAMP ? a2.z / sk4.z : -s,
                                  ck.w > W_CLAMP ? a2.w / sk4.w : -s));
      st4(p.dmv + go, ld4(amv + j * ldk + c));
      st4(p.dcv + go, ld4(acv + j * ldk + c));
    }
  }
}

// ---------------------------------------------------------------------------------------------
// BPR + pvn loss on elementwise Wasserstein distances (stosa/trainer.py:358-391).  Warp per row.
// acc[0] += sum softplus(-(d_neg - d_pos + 1e-24)) * t ; acc[1] += sum clamp(d_pos - d_pn, 0) * t ; acc[2] += sum auc term ; acc[3] += sum t
// ---------------------------------------------------------------------------------------------
struct WBprArgs {
  const float *sm, *sc;          // sequence mean / cov outputs [M, H]
  const float *Em, *Ec;          // item mean / cov tables [I+1, H] (cov is raw: ELU+1 applied here)
  const int *pos, *neg;          // [M]
  double* acc;                   // [4]
  const float* gcoef;            // backward: [2] = {g_bpr / n, g_pvn * pvn_weight / n} (device scalars)
  float *dsm, *dsc, *gpm, *gpc, *gnm, *gnc;   // backward outputs [M, H]
  int M, H;
};

__device__ __forceinline__ float elu1(float x) { return (x > 0.f ? x : expm1f(x)) + 1.f; }
__device__ __forceinline__ float elu1_g(float x) { return x > 0.f ? 1.f : expf(x); }
__device__ __forceinline__ float wsqrt(float c) { return sqrtf(fmaxf(c, W_CLAMP)); }

__device__ __forceinline__ void wbpr_dists(const WBprArgs& p, int r, int lane, int ip, int in, float& dp, float& dn, float& dpn) {
  const float* m = p.sm + (long long)r * p.H;
  const float* c = p.sc + (long long)r * p.H;
  const float* pm = p.Em + (long long)ip * p.H;
  const float* pc = p.Ec + (long long)ip * p.H;
  const float* nm = p.Em + (long long)in * p.H;
  const float* nc = p.Ec + (long long)in * p.H;
  float a = 0.f, b = 0.f, d = 0.f;
  for (int k = lane; k < p.H; k += 32) {
    const float mu = m[k], s = wsqrt(c[k]), mp = pm[k], sp = wsqrt(elu1(pc[k])), mn = nm[k], sn = wsqrt(elu1(nc[k]));
    a += (mu - mp) * (mu - mp) + (s - sp) * (s - sp);
    b += (mu - mn) * (mu - mn) + (s - sn) * (s - sn);
    d += (mp - mn) * (mp - mn) + (sp - sn) * (sp - sn);
  }
  dp = warp_sum(a); dn = warp_sum(b); dpn = warp_sum(d);
}

__global__ void __launch_bounds__(NT) wbpr_fwd_kernel(WBprArgs p) {
  const int lane = threadIdx.x & 31, wpb = NT / 32;
  double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < p.M; r += gridDim.x * wpb) {
    const int ip = p.pos[r], in = p.neg[r];
    if (ip <= 0) continue;
    float dp, dn, dpn;
    wbpr_dists(p, r, lane, ip, in, dp, dn, dpn);
    const float d = dn - dp, x = d + 1e-24f;
    s0 += (double)(x > 0.f ? log1pf(expf(-x)) : -x + log1pf(expf(x)));
    s1 += (double)fmaxf(dp - dpn, 0.f);
    s2 += (double)(((d > 0.f) - (d < 0.f) + 1) * 0.5f);   // the AUC term takes sign(dn - dp) without the 1e-24: a tie counts 1/2
    s3 += 1.0;
  }
  if (lane == 0 && s3 > 0) {
    atomicAdd(p.acc + 0, s0); atomicAdd(p.acc + 1, s1); atomicAdd(p.acc + 2, s2); atomicAdd(p.acc + 3, s3);
  }
}

__global__ void __launch_bounds__(NT) wbpr_bwd_kernel(WBprArgs p) {
  const int lane = threadIdx.x & 31, wpb = NT / 32;
  const float c_bpr = p.gcoef[0], c_pvn = p.gcoef[1];
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < p.M; r += gridDim.x * wpb) {
    const int ip = p.pos[r], in = p.neg[r];
    const long long o = (long long)r * p.H;
    if (ip <= 0) {
      for (int k = lane; k < p.H; k += 32) {
        p.dsm[o + k] = 0.f; p.dsc[o + k] = 0.f; p.gpm[o + k] = 0.f; p.gpc[o + k] = 0.f; p.gnm[o + k] = 0.f; p.gnc[o + k] = 0.f;
      }
      continue;
    }
    float dp, dn, dpn;
    wbpr_dists(p, r, lane, ip, in, dp, dn, dpn);
    const float x = dn - dp + 1e-24f;
    const float sg = 1.f / (1.f + expf(x));          // sigmoid(-x) = -d softplus(-x)/dx
    float gdp = c_bpr * sg, gdn = -c_bpr * sg, gdpn = 0.f;
    if (dp - dpn > 0.f) { gdp += c_pvn; gdpn = -c_pvn; }
    const float* pm = p.Em + (long long)ip * p.H;
    const float* pc = p.Ec + (long long)ip * p.H;
    const float* nm = p.Em + (long long)in * p.H;
    const float* nc = p.Ec + (long long)in * p.H;
    for (int k = lane; k < p.H; k += 32) {
      const float mu = p.sm[o + k], cs = p.sc[o + k], s = wsqrt(cs);
      const float mp = pm[k], rp = pc[k], cp = elu1(rp), sp = wsqrt(cp);
      const float mn = nm[k], rn = nc[k], cn = elu1(rn), sn = wsqrt(cn);
      // d/dm1 (m1-m2)^2 = 2(m1-m2) ; d/dc1 (sqrt(c1)-s2)^2 = (s1-s2)/s1 (0 below the clamp)
      p.dsm[o + k] = gdp * 2.f * (mu - mp) + gdn * 2.f * (mu - mn);
      p.dsc[o + k] = cs > W_CLAMP ? (gdp * (s - sp) + gdn * (s - sn)) / s : 0.f;
      p.gpm[o + k] = -gdp * 2.f * (mu - mp) + gdpn * 2.f * (mp - mn);
      p.gnm[o + k] = -gdn * 2.f * (mu - mn) - gdpn * 2.f * (mp - mn);
      const float gcp = cp > W_CLAMP ? (-gdp * (s - sp) + gdpn * (sp - sn)) / sp : 0.f;
      const float gcn = cn > W_CLAMP ? (-gdn * (s - sn) - gdpn * (sp - sn)) / sn : 0.f;
      p.gpc[o + k] = gcp * elu1_g(rp);
      p.gnc[o + k] = gcn * elu1_g(rn);
    }
  }
}

// reconstruction term: acc += sum (a - b)^2 ; bwd: da = 2 (a - b) * g[0] * scale, db = -da   (F.mse_loss, trainer.py:519-520)
__global__ void __launch_bounds__(256) sqdiff_fwd_kernel(const float* __restrict__ a, const float* __restrict__ b, long long n4, double* acc) {
  float s = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 x = reinterpret_cast<const float4*>(a)[i], y = reinterpret_cast<const float4*>(b)[i];
    s += (x.x - y.x) * (x.x - y.x) + (x.y - y.y) * (x.y - y.y) + (x.z - y.z) * (x.z - y.z) + (x.w - y.w) * (x.w - y.w);
  }
  s = warp_sum(s);
  __shared__ float red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int w = 0; w < 8; ++w) t += (double)red[w];
    atomicAdd(acc, t);
  }
}
__global__ void __launch_bounds__(256) sqdiff_bwd_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ g,
                                                         float scale, float* __restrict__ da, float* __restrict__ db, long long n4) {
  const float c = 2.f * g[0] * scale;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 x = reinterpret_cast<const float4*>(a)[i], y = reinterpret_cast<const float4*>(b)[i];
    const float4 d = make_float4(c * (x.x - y.x), c * (x.y - y.y), c * (x.z - y.z), c * (x.w - y.w));
    reinterpret_cast<float4*>(da)[i] = d;
    reinterpret_cast<float4*>(db)[i] = make_float4(-d.x, -d.y, -d.z, -d.w);
  }
}

// catalog rows for full-sort evaluation (trainer.py:464-479): A[i] = [ mean_i | sqrt(clamp(elu(cov_i)+1)) | -(|mean_i|^2 + sum(elu(cov_i)+1)) | 0 0 0 ]
// so that  -(distance(u, i)) + const(u) = [2 mean_u | 2 sqrt(cov_u) | 1 | 0 0 0] . A[i]
__global__ void __launch_bounds__(NT) wcatalog_kernel(const float* __restrict__ Em, const float* __restrict__ Ec, float* __restrict__ A, int n,
                                                      int H, int is_user) {
  const int lane = threadIdx.x & 31, wpb = NT / 32, ld = 2 * H + 4;
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < n; r += gridDim.x * wpb) {
    float nrm = 0.f;
    for (int k = lane; k < H; k += 32) {
      const float m = Em[(long long)r * H + k];
      const float c = is_user ? Ec[(long long)r * H + k] : elu1(Ec[(long long)r * H + k]);
      const float s = wsqrt(c);
      A[(long long)r * ld + k] = is_user ? 2.f * m : m;
      A[(long long)r * ld + H + k] = is_user ? 2.f * s : s;
      nrm += m * m + c;
    }
    nrm = warp_sum(nrm);
    if (lane < 4) A[(long long)r * ld + 2 * H + lane] = lane == 0 ? (is_user ? 1.f : -nrm) : 0.f;
  }
}

// centred catalog for K7 (adt_wcatalog_build / adt_wcatalog_user): item row y_i = [ mean_i | sqrt(elu(cov_i)+1) ], user row
// x_u = [ mean_u | sqrt(cov_u) ], mu = column mean of the y_i;  rows e_i = y_i - mu, bias b_i = -|e_i|^2, user features f_u = 2 (x_u - mu).
constexpr int WCAT_PARTS = 296;     // column-sum blocks (2 per SM); fixed, so the summation order depends on n and H only

__device__ __forceinline__ float wcat_col(const float* __restrict__ Em, const float* __restrict__ Ec, long long r, int c, int H) {
  return c < H ? Em[r * H + c] : wsqrt(elu1(Ec[r * H + c - H]));
}

// Deterministic column mean of the 2H-wide item rows in one launch of WCAT_PARTS blocks.  Block b sums the fixed row range
// [b*chunk, (b+1)*chunk): thread t owns column t % 2H of sub-row t / 2H, fp64 accumulation in row order, sub-rows folded in order.
// The last block to arrive (counter in `work`) folds the WCAT_PARTS partials in block order and resets the counter to 0.
__global__ void __launch_bounds__(NT) wcat_mean_kernel(const float* __restrict__ Em, const float* __restrict__ Ec, int n, int H,
                                                       double* __restrict__ part, unsigned int* counter, float* __restrict__ mu) {
  __shared__ double red[NT];
  __shared__ bool last;
  const int W = 2 * H, S = NT / W, c = threadIdx.x % W, s = threadIdx.x / W;
  const long long chunk = ((long long)n + WCAT_PARTS - 1) / WCAT_PARTS;
  const long long lo = blockIdx.x * chunk, hi = min((long long)n, lo + chunk);
  double acc = 0.0;
  if (s < S) {
#pragma unroll 4
    for (long long r = lo + s; r < hi; r += S) acc += (double)wcat_col(Em, Ec, r, c, H);
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.x < W) {
    double t = red[threadIdx.x];
    for (int j = 1; j < S; ++j) t += red[j * W + threadIdx.x];
    part[(long long)blockIdx.x * W + threadIdx.x] = t;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(counter, 1u) == WCAT_PARTS - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (threadIdx.x < W) {
    double t = 0.0;
#pragma unroll 8
    for (int b = 0; b < WCAT_PARTS; ++b) t += __ldcg(part + (long long)b * W + threadIdx.x);
    mu[threadIdx.x] = (float)(t / (double)n);
  }
  if (threadIdx.x == 0) *counter = 0u;
}

// warp per item row: rows[i] = y_i - mu, bias[i] = -|rows[i]|^2 (fp32, from the stored values)
__global__ void __launch_bounds__(NT) wcat_rows_kernel(const float* __restrict__ Em, const float* __restrict__ Ec, const float* __restrict__ mu,
                                                       int n, int H, float* __restrict__ rows, float* __restrict__ bias) {
  const int lane = threadIdx.x & 31, wpb = NT / 32, W = 2 * H;
  for (long long r = blockIdx.x * wpb + (threadIdx.x >> 5); r < n; r += (long long)gridDim.x * wpb) {
    float nrm = 0.f;
    for (int c = lane; c < W; c += 32) {
      const float e = wcat_col(Em, Ec, r, c, H) - mu[c];
      rows[r * W + c] = e;
      nrm = fmaf(e, e, nrm);
    }
    nrm = warp_sum(nrm);
    if (lane == 0) bias[r] = -nrm;
  }
}

// f[u] = 2 (x_u - mu), [U][2H]; cov already ELU+1 (the encoder's output)
__global__ void __launch_bounds__(NT) wcat_user_kernel(const float* __restrict__ m, const float* __restrict__ cv, const float* __restrict__ mu,
                                                       int U, int H, float* __restrict__ f) {
  const int W = 2 * H;
  const long long total = (long long)U * W;
  for (long long i = (long long)blockIdx.x * NT + threadIdx.x; i < total; i += (long long)gridDim.x * NT) {
    const long long u = i / W;
    const int c = (int)(i - u * W);
    const float x = c < H ? m[u * H + c] : wsqrt(cv[u * H + c - H]);
    f[i] = 2.f * (x - mu[c]);
  }
}

}  // namespace adt
