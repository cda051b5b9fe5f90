// Forward kernels of the SASRec-ADT hot path.  Reference semantics: SURVEY.md appendix A
// (/root/reference/sasrec/model.py:32-81, sasrec/modules.py:270-527, :618-677).
#pragma once
#include "common.cuh"

namespace adt {

// -------------------------------------------------------------------------------------------------
// K1  embedding gather:  x = dropout(E[id]*sqrt(H) + P[t]) * (id != 0)       (model.py:34-41)
// One thread per float4; 128-bit coalesced loads/stores.  mul and add are kept as two roundings so that
// the result is bit-identical to torch's `seqs *= H**0.5; seqs += pos_emb(...)`.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) embed_fwd_kernel(const int* __restrict__ ids, const float* __restrict__ E,
                                                        const float* __restrict__ P, float* __restrict__ x, int M, int L, int H,
                                                        float scale, DropDesc drop) {
  // 32-bit index math (M*H/4 < 2^31, checked by the launcher): the kernel is HBM bound only if the per-element integer work stays small
  const unsigned h4 = (unsigned)H >> 2;
  const unsigned n = (unsigned)M * h4;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned row = i / h4, c4 = i - row * h4;
    const int id = __ldg(ids + row);
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (id != 0) {
      const unsigned t = row % (unsigned)L;
      const float4 e = __ldg(reinterpret_cast<const float4*>(E + (long long)id * H) + c4);
      const float4 p = __ldg(reinterpret_cast<const float4*>(P + (long long)t * H) + c4);
      o.x = __fadd_rn(__fmul_rn(e.x, scale), p.x);
      o.y = __fadd_rn(__fmul_rn(e.y, scale), p.y);
      o.z = __fadd_rn(__fmul_rn(e.z, scale), p.z);
      o.w = __fadd_rn(__fmul_rn(e.w, scale), p.w);
      if (drop.enabled) {
        const float4 m = drop_mul4(drop, (drop.base >> 2) + (unsigned long long)i);
        o = f4_mul(o, m);
      }
    }
    __stcs(reinterpret_cast<float4*>(x) + i, o);
  }
}

// -------------------------------------------------------------------------------------------------
// pre_fwd: LayerNorm + packed in-projection.
//   encoder (kv_from_norm=0, modules.py:646-647,124-130): Qn=LN(x); q=(Qn Wq^T+bq)*qscale; k,v = x Wkv^T + bkv
//   decoder (kv_from_norm=1, modules.py:668-670)        : d =LN(x); q,k,v all from d; d is written to norm_out
// -------------------------------------------------------------------------------------------------
template <int TM, bool MMA>
__global__ void __launch_bounds__(NT) pre_fwd_kernel(const float* __restrict__ x, const float* __restrict__ ln_g,
                                                     const float* __restrict__ ln_b, const float* __restrict__ Win,
                                                     const float* __restrict__ bin, float* __restrict__ q, float* __restrict__ k,
                                                     float* __restrict__ v, float* __restrict__ norm_out, int M, int H, float qscale,
                                                     int kv_from_norm) {
  extern __shared__ __align__(16) float smem[];
  const int ld = H + tile_pad<MMA>();
  float* Xs = smem;
  float* Ns = Xs + TM * ld;
  float* Ws = Ns + TM * ld;
  const int row0 = blockIdx.x * TM;
  ADT_STAMP(0);
  prefetch_vec(ln_g, H); prefetch_vec(ln_b, H); prefetch_vec(bin, 3 * H);
  __shared__ WStreamState wst;
  if (threadIdx.x == 0) {
    wst.g[0] = GemmDesc{Win, H, H, H, 0};
    wst.g[1] = GemmDesc{Win + (long long)H * H, H, 2 * H, H, 0};
    wst.ng = 2;
  }
  __syncthreads();
  WStream<WS_NST, MMA> ws;
  ws.start(&wst, Ws);
  ADT_STAMP(1);
  load_tile<TM>(Xs, ld, x, H, 0, H, row0, M);
  tile_sync();
  ADT_STAMP(2);
  ln_tile<TM>(Xs, Ns, ld, H, ln_g, ln_b, 1e-8f, row0, M);
  __syncthreads();
  ADT_STAMP(3);
  if (norm_out) store_tile<TM>(Ns, ld, norm_out, H, 0, H, row0, M);
  gemm_stream<TM, false, WS_NST, MMA>(Ns, ld, ws, 0, [&](int, int r, int col, float4 a) {
    if (row0 + r < M) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(bin + col));
      *reinterpret_cast<float4*>(q + (long long)(row0 + r) * H + col) = f4_scale(f4_add(a, b), qscale);
    }
  });
  ADT_STAMP(4);
  const float* Akv = kv_from_norm ? Ns : Xs;
  gemm_stream<TM, false, WS_NST, MMA>(Akv, ld, ws, 1, [&](int, int r, int col, float4 a) {
    if (row0 + r < M) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(bin + H + col));
      float* dst = col < H ? (k + (long long)(row0 + r) * H + col) : (v + (long long)(row0 + r) * H + (col - H));
      *reinterpret_cast<float4*>(dst) = f4_add(a, b);
    }
  });
  ADT_STAMP(5);
}

// multipliers for 4 consecutive elements starting at an arbitrary (not 4-aligned) linear index
__device__ __forceinline__ float4 drop_mul4_unaligned(const DropDesc& d, unsigned long long idx0) {
  const unsigned off = (unsigned)idx0 & 3u;
  const float4 a = drop_mul4(d, idx0 >> 2);
  if (off == 0) return a;
  const float4 b = drop_mul4(d, (idx0 >> 2) + 1);
  if (off == 1) return make_float4(a.y, a.z, a.w, b.x);
  if (off == 2) return make_float4(a.z, a.w, b.x, b.y);
  return make_float4(a.w, b.x, b.y, b.z);
}

// -------------------------------------------------------------------------------------------------
// attn_fwd: one CTA per (query tile, head, sequence).  S = q k^T (q pre-scaled) -> mask -> softmax (warp per
// row, shuffle reductions) -> dropout -> ctx = P v.  Scores never leave shared memory.
//   mask_mode 0: causal (j <= i)                                   SASRec  (model.py:43-44)
//   mask_mode 1: key padding only (kid[b][j] != 0), bidirectional   Bert4Rec (bert4rec/model/modules.py:88-91)
// lse (optional) = rowmax + log(rowsum) is saved for the backward pass.
// -------------------------------------------------------------------------------------------------
template <int TM, bool MMA>
__global__ void __launch_bounds__(NT) attn_fwd_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                      const float* __restrict__ v, float* __restrict__ ctx, float* __restrict__ lse,
                                                      const int* __restrict__ key_ids, int L, int H, int nh, int mask_mode,
                                                      DropDesc drop) {
  extern __shared__ __align__(16) float smem[];
  const int hd = H / nh;
  const int ldq = hd + tile_pad<MMA>();
  const int lds = ((L + 3) & ~3) + tile_pad<MMA>();
  float* Qs = smem;
  float* Ss = Qs + TM * ldq;
  float* Ws = Ss + TM * lds;
  const int i0 = blockIdx.x * TM, h = blockIdx.y, b = blockIdx.z;
  const long long seq_off = (long long)b * L * H + (long long)h * hd;
  const int Lk = mask_mode == 0 ? min(L, i0 + TM) : L;  // keys this tile can see
  ADT_STAMP(8);
  __shared__ WStreamState wst;
  if (threadIdx.x == 0) {
    wst.g[0] = GemmDesc{k + seq_off, H, Lk, hd, 0};
    wst.g[1] = GemmDesc{v + seq_off, H, hd, Lk, 1};
    wst.ng = 2;
  }
  __syncthreads();
  WStream<WS_NST, MMA> ws;
  ws.start(&wst, Ws);
  ADT_STAMP(9);
  load_tile<TM>(Qs, ldq, q + seq_off, H, 0, hd, i0, L);
  tile_sync();
  ADT_STAMP(10);
  gemm_stream<TM, false, WS_NST, MMA>(Qs, ldq, ws, 0, [&](int, int r, int col, float4 a) {
    *reinterpret_cast<float4*>(Ss + r * lds + col) = a;
  });
  ADT_STAMP(11);

  // softmax + dropout.  A lane owns 8 consecutive keys (one aligned Philox call); a row is handled by LPR lanes
  // (8 when all visible keys fit 64, else 32) so that 32/LPR rows run side by side in every warp -- the per-row chain
  // (max -> exp -> sum -> 1/sum) is latency bound.
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int Lk4 = (Lk + 3) & ~3;
  const int lpr = Lk4 <= 64 ? 8 : 32;
  const int rpw = 32 / lpr;                 // rows per warp per pass
  const int sub = l % lpr;
  for (int r = w * rpw + l / lpr; r < TM; r += (NT / 32) * rpw) {
    const int i = i0 + r;
    float* srow = Ss + r * lds;
    const bool valid = i < L;
    const int nj = !valid ? 0 : (mask_mode == 0 ? i + 1 : L);
    const int j0 = 8 * sub;
    float sv[8];
    {
      float4 s0 = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY), s1 = s0;
      if (j0 < nj) s0 = *reinterpret_cast<const float4*>(srow + j0);
      if (j0 + 4 < nj) s1 = *reinterpret_cast<const float4*>(srow + j0 + 4);
      sv[0] = s0.x; sv[1] = s0.y; sv[2] = s0.z; sv[3] = s0.w; sv[4] = s1.x; sv[5] = s1.y; sv[6] = s1.z; sv[7] = s1.w;
    }
    float mx = -INFINITY;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float sc = (j0 + c < nj) ? sv[c] : -INFINITY;
      if (mask_mode == 1 && j0 + c < nj && key_ids[b * L + j0 + c] == 0) sc = -1e9f;
      sv[c] = sc;
      mx = fmaxf(mx, sc);
    }
    for (int o = lpr >> 1; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float e = sv[c] == -INFINITY ? 0.f : expf(sv[c] - mx);
      sv[c] = e;
      sum += e;
    }
    for (int o = lpr >> 1; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = valid ? 1.0f / sum : 0.f;
    if (lse && valid && sub == 0) lse[((long long)b * nh + h) * L + i] = mx + logf(sum);
    if (drop.enabled && j0 < nj) {
      float m[8];
      drop_mul8_attn(drop, drop.base + ((unsigned long long)b * nh + h) * L + i, ((L + 7) & ~7) >> 3, sub, m);
#pragma unroll
      for (int c = 0; c < 8; ++c) sv[c] *= m[c];
    }
    if (j0 < Lk4) *reinterpret_cast<float4*>(srow + j0) = make_float4(sv[0] * inv, sv[1] * inv, sv[2] * inv, sv[3] * inv);
    if (j0 + 4 < Lk4) *reinterpret_cast<float4*>(srow + j0 + 4) = make_float4(sv[4] * inv, sv[5] * inv, sv[6] * inv, sv[7] * inv);
  }
  __syncthreads();
  ADT_STAMP(12);
  gemm_stream<TM, true, WS_NST, MMA>(Ss, lds, ws, 1, [&](int, int r, int col, float4 a) {
    if (i0 + r < L) *reinterpret_cast<float4*>(ctx + seq_off + (long long)(i0 + r) * H + col) = a;
  });
  ADT_STAMP(13);
}

// -------------------------------------------------------------------------------------------------
// mid_fwd (decoder): a = ctx1 Wo1^T + bo1 ; q2 = (a Wq2^T + bq2)*qscale ; k2,v2 = feats Wkv2^T + bkv2
// (modules.py:669-672: self-attention out-projection followed by the cross-attention in-projection)
// -------------------------------------------------------------------------------------------------
template <int TM, bool MMA>
__global__ void __launch_bounds__(NT) mid_fwd_kernel(const float* __restrict__ ctx1, const float* __restrict__ feats,
                                                     const float* __restrict__ Wo1, const float* __restrict__ bo1,
                                                     const float* __restrict__ Win2, const float* __restrict__ bin2,
                                                     float* __restrict__ a_out, float* __restrict__ q2, float* __restrict__ k2,
                                                     float* __restrict__ v2, int M, int H, float qscale) {
  extern __shared__ __align__(16) float smem[];
  const int ld = H + tile_pad<MMA>();
  float* T0 = smem;
  float* T1 = T0 + TM * ld;
  float* T2 = T1 + TM * ld;
  float* Ws = T2 + TM * ld;
  const int row0 = blockIdx.x * TM;
  prefetch_vec(bo1, H); prefetch_vec(bin2, 3 * H);
  __shared__ WStreamState wst;
  if (threadIdx.x == 0) {
    wst.g[0] = GemmDesc{Wo1, H, H, H, 0};
    wst.g[1] = GemmDesc{Win2, H, H, H, 0};
    wst.g[2] = GemmDesc{Win2 + (long long)H * H, H, 2 * H, H, 0};
    wst.ng = 3;
  }
  __syncthreads();
  WStream<WS_NST, MMA> ws;
  ws.start(&wst, Ws);
  load_tile<TM>(T0, ld, ctx1, H, 0, H, row0, M);
  load_tile<TM>(T2, ld, feats, H, 0, H, row0, M);
  tile_sync();
  gemm_stream<TM, false, WS_NST, MMA>(T0, ld, ws, 0, [&](int, int r, int col, float4 a) {
    const float4 o = f4_add(a, __ldg(reinterpret_cast<const float4*>(bo1 + col)));
    *reinterpret_cast<float4*>(T1 + r * ld + col) = o;
    if (a_out && row0 + r < M) *reinterpret_cast<float4*>(a_out + (long long)(row0 + r) * H + col) = o;
  });
  gemm_stream<TM, false, WS_NST, MMA>(T1, ld, ws, 1, [&](int, int r, int col, float4 a) {
    if (row0 + r < M)
      *reinterpret_cast<float4*>(q2 + (long long)(row0 + r) * H + col) =
          f4_scale(f4_add(a, __ldg(reinterpret_cast<const float4*>(bin2 + col))), qscale);
  });
  gemm_stream<TM, false, WS_NST, MMA>(T2, ld, ws, 2, [&](int, int r, int col, float4 a) {
    if (row0 + r < M) {
      const float4 o = f4_add(a, __ldg(reinterpret_cast<const float4*>(bin2 + H + col)));
      float* dst = col < H ? (k2 + (long long)(row0 + r) * H + col) : (v2 + (long long)(row0 + r) * H + (col - H));
      *reinterpret_cast<float4*>(dst) = o;
    }
  });
}

// -------------------------------------------------------------------------------------------------
// post_fwd: attention out-projection + residual + (LayerNorm) + point-wise FFN + mask, fused.
//   encoder (IS_DEC=false, modules.py:648-654): y = LN1(x) + ctx Wo^T + bo ; z = LN2(y)
//        out = (drop2(relu(drop1(z C1^T + c1)) C2^T + c2) + z) * keep
//        rec[r][c][:] = log_softmax(ctx[r, head c] Ws^T + bs)  (true layout; the reference's mis-view is a pure row
//        permutation applied on the host side, SURVEY.md A.3); nll_acc += -sum_c rec[r][c][c]
//   decoder (IS_DEC=true,  modules.py:671-676): c = ctx Wo^T + bo ; out = (d + drop2(relu(drop1(c C1^T+c1)) C2^T+c2) + c) * keep
//        mse_acc += sum (enc_in - out)^2
// u_save (y or c) and h1_save (pre-dropout FFN hidden) are written for the backward pass when non-null.
// -------------------------------------------------------------------------------------------------
struct PostFwdArgs {
  const float* ctx; const float* resid;  // enc: x (block input, LN1 recomputed) ; dec: d
  const int* ids;                         // keep = ids[row] != 0
  const float* Wo; const float* bo;
  const float* ln1_g; const float* ln1_b; const float* ln2_g; const float* ln2_b;  // enc only
  const float* C1; const float* c1; const float* C2; const float* c2;
  const float* Wsp; const float* bsp;     // enc only: sparse head [nh][hd], [nh]
  const float* enc_in;                    // dec only (nullable): reconstruction target
  float* u_save; float* h1_save; float* out; float* rec;  // rec: [M][nh][nh] (enc only, nullable)
  double* acc;                            // enc: nll sum ; dec: squared-error sum (nullable)
  int M, H, nh;
  DropDesc drop1, drop2;
};

template <int TM, bool IS_DEC, bool MMA>
__global__ void __launch_bounds__(NT) post_fwd_kernel(PostFwdArgs p) {
  extern __shared__ __align__(16) float smem[];
  __shared__ double red[NT / 32];
  const int H = p.H, M = p.M;
  const int ld = H + tile_pad<MMA>();
  float* T0 = smem;
  float* T1 = T0 + TM * ld;
  float* T2 = T1 + TM * ld;
  float* Ws = T2 + TM * ld;
  const int row0 = blockIdx.x * TM;
  prefetch_vec(p.bo, H); prefetch_vec(p.c1, H); prefetch_vec(p.c2, H);
  if (!IS_DEC) { prefetch_vec(p.ln1_g, H); prefetch_vec(p.ln1_b, H); prefetch_vec(p.ln2_g, H); prefetch_vec(p.ln2_b, H); }
  __shared__ WStreamState wst;
  if (threadIdx.x == 0) {
    wst.g[0] = GemmDesc{p.Wo, H, H, H, 0};
    wst.g[1] = GemmDesc{p.C1, H, H, H, 0};
    wst.g[2] = GemmDesc{p.C2, H, H, H, 0};
    wst.ng = 3;
  }
  __syncthreads();
  WStream<WS_NST, MMA> ws;
  ws.start(&wst, Ws);
  load_tile<TM>(T0, ld, p.ctx, H, 0, H, row0, M);
  if (!IS_DEC) {
    load_tile<TM>(T2, ld, p.resid, H, 0, H, row0, M);
    tile_sync();
    ln_tile<TM>(T2, T1, ld, H, p.ln1_g, p.ln1_b, 1e-8f, row0, M);
  }
  tile_sync();
  gemm_stream<TM, false, WS_NST, MMA>(T0, ld, ws, 0, [&](int, int r, int col, float4 a) {
    float4 o = f4_add(a, __ldg(reinterpret_cast<const float4*>(p.bo + col)));
    if (!IS_DEC) o = f4_add(o, *reinterpret_cast<const float4*>(T1 + r * ld + col));
    *reinterpret_cast<float4*>(T1 + r * ld + col) = o;
    if (p.u_save && row0 + r < M) *reinterpret_cast<float4*>(p.u_save + (long long)(row0 + r) * H + col) = o;
  });
  if (!IS_DEC) {
    // independence head on the per-head context slices: one thread per (row, head c, class j) dot product of length
    // hd, logits parked in the (idle) weight staging area, then one thread per (row, c) log-softmax.
    if (p.rec || p.acc) {
      const int nh = p.nh, hd = H / nh, n2 = nh * nh;
      float* lgs = ws.scratch();
      for (int i = threadIdx.x; i < TM * n2; i += NT) {
        const int r = i / n2, cj = i - r * n2, c = cj / nh, j = cj - c * nh;
        const float* xr = T0 + r * ld + c * hd;
        const float* wr = p.Wsp + j * hd;
        float s = 0.f;
        for (int dd = 0; dd < hd; dd += 4) {
          const float4 a = *reinterpret_cast<const float4*>(xr + dd);
          const float4 b = __ldg(reinterpret_cast<const float4*>(wr + dd));
          s = fmaf(a.x, b.x, s); s = fmaf(a.y, b.y, s); s = fmaf(a.z, b.z, s); s = fmaf(a.w, b.w, s);
        }
        lgs[i] = s + p.bsp[j];
      }
      __syncthreads();
      double nll = 0.0;
      for (int i = threadIdx.x; i < TM * nh; i += NT) {
        const int r = i / nh, c = i - r * nh;
        if (row0 + r >= M) continue;
        const float* lg = lgs + r * n2 + c * nh;
        float mx = lg[0];
        for (int j = 1; j < nh; ++j) mx = fmaxf(mx, lg[j]);
        float se = 0.f;
        for (int j = 0; j < nh; ++j) se += expf(lg[j] - mx);
        const float lz = mx + logf(se);
        if (p.rec)
          for (int j = 0; j < nh; ++j) p.rec[((long long)(row0 + r) * nh + c) * nh + j] = lg[j] - lz;
        nll -= (double)(lg[c] - lz);
      }
      if (p.acc) cta_accumulate(nll, p.acc, red);
    }
    __syncthreads();
    ln_tile<TM>(T1, T1, ld, H, p.ln2_g, p.ln2_b, 1e-8f, row0, M);
    __syncthreads();
  }
  gemm_stream<TM, false, WS_NST, MMA>(T1, ld, ws, 1, [&](int, int r, int col, float4 a) {
    float4 h1 = f4_add(a, __ldg(reinterpret_cast<const float4*>(p.c1 + col)));
    if (p.h1_save && row0 + r < M) *reinterpret_cast<float4*>(p.h1_save + (long long)(row0 + r) * H + col) = h1;
    if (p.drop1.enabled) h1 = f4_mul(h1, drop_mul4(p.drop1, (p.drop1.base + (unsigned long long)(row0 + r) * H + col) >> 2));
    *reinterpret_cast<float4*>(T2 + r * ld + col) = make_float4(fmaxf(h1.x, 0.f), fmaxf(h1.y, 0.f), fmaxf(h1.z, 0.f), fmaxf(h1.w, 0.f));
  });
  double sq = 0.0;
  gemm_stream<TM, false, WS_NST, MMA>(T2, ld, ws, 2, [&](int, int r, int col, float4 a) {
    if (row0 + r >= M) return;
    float4 h2 = f4_add(a, __ldg(reinterpret_cast<const float4*>(p.c2 + col)));
    if (p.drop2.enabled) h2 = f4_mul(h2, drop_mul4(p.drop2, (p.drop2.base + (unsigned long long)(row0 + r) * H + col) >> 2));
    float4 o = f4_add(h2, *reinterpret_cast<const float4*>(T1 + r * ld + col));
    const long long g = (long long)(row0 + r) * H + col;
    if (IS_DEC) o = f4_add(o, *reinterpret_cast<const float4*>(p.resid + g));
    if (p.ids[row0 + r] == 0) o = make_float4(0.f, 0.f, 0.f, 0.f);
    *reinterpret_cast<float4*>(p.out + g) = o;
    if (IS_DEC && p.enc_in) {
      const float4 e = *reinterpret_cast<const float4*>(p.enc_in + g);
      const float dx = e.x - o.x, dy = e.y - o.y, dz = e.z - o.z, dw = e.w - o.w;
      sq += (double)(dx * dx + dy * dy) + (double)(dz * dz + dw * dw);
    }
  });
  if (IS_DEC && p.acc) cta_accumulate(sq, p.acc, red);
}

// -------------------------------------------------------------------------------------------------
// final_fwd: feats = LN_last(x) ; pos/neg logits = <feats, E[pos|neg]> ; BCE partial sums over pos != 0
// (model.py:48,72-76 ; main.py:151-153).  Warp per row.  acc[0]+=softplus(-pos) acc[1]+=softplus(neg) acc[2]+=1
// If ln_g == nullptr the LayerNorm is skipped (supernet: supersasrec.py:56-58 has no last_layernorm).
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ float softplusf(float z) { return fmaxf(z, 0.f) + log1pf(expf(-fabsf(z))); }

template <int U>
__global__ void __launch_bounds__(NT) final_fwd_kernel(const float* __restrict__ x, const float* __restrict__ ln_g,
                                                       const float* __restrict__ ln_b, const float* __restrict__ E,
                                                       const int* __restrict__ pos, const int* __restrict__ neg,
                                                       float* __restrict__ feats, float* __restrict__ pos_logits,
                                                       float* __restrict__ neg_logits, double* __restrict__ acc, int M, int H) {
  __shared__ double red[NT / 32];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0;
  for (int row = blockIdx.x * (NT / 32) + w; row < M; row += gridDim.x * (NT / 32)) {
    const float* xr = x + (long long)row * H;
    float xv[U];
    float sum = 0.f;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = l + 32 * u;
      xv[u] = c < H ? xr[c] : 0.f;
      sum += xv[u];
    }
    float mean = 0.f, rstd = 1.f;
    if (ln_g) {
      mean = warp_sum(sum) / (float)H;
      float var = 0.f;
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (l + 32 * u < H) { const float t = xv[u] - mean; var += t * t; }
      rstd = 1.0f / sqrtf(warp_sum(var) / (float)H + 1e-8f);
    }
    const int pi = pos ? pos[row] : 0, ni = neg ? neg[row] : 0;
    float dp = 0.f, dn = 0.f;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = l + 32 * u;
      if (c < H) {
        const float f = ln_g ? (xv[u] - mean) * rstd * ln_g[c] + ln_b[c] : xv[u];
        feats[(long long)row * H + c] = f;
        if (pos) {
          dp = fmaf(f, E[(long long)pi * H + c], dp);
          dn = fmaf(f, E[(long long)ni * H + c], dn);
        }
      }
    }
    if (pos) {
      dp = warp_sum(dp);
      dn = warp_sum(dn);
      if (l == 0) {
        pos_logits[row] = dp;
        neg_logits[row] = dn;
        if (pi != 0) {
          a0 += (double)softplusf(-dp);
          a1 += (double)softplusf(dn);
          a2 += 1.0;
        }
      }
    }
  }
  if (acc) {
    cta_accumulate(a0, acc + 0, red);
    cta_accumulate(a1, acc + 1, red);
    cta_accumulate(a2, acc + 2, red);
  }
}

}  // namespace adt
