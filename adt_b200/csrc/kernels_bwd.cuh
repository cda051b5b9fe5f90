// Backward kernels of the SASRec-ADT hot path (hand-derived adjoints of kernels_fwd.cuh).
// Weight gradients are reduced over the CTA's row tile in registers and added to the global gradient
// buffers with 128-bit vector atomics (red.global.add.v4.f32).
#pragma once
#include "common.cuh"
#include "kernels_fwd.cuh"

namespace adt {

// elementwise helper over a [TM][C] tile (one float4 per thread step): f(row_local, col)
template <int TM, class F>
__device__ __forceinline__ void tile_foreach4(int C, F f) {
  const int c4n = C >> 2;
  for (int s = threadIdx.x; s < TM * c4n; s += NT) {
    const int r = s / c4n, c4 = s - r * c4n;
    f(r, 4 * c4);
  }
}

// like tile_foreach4, but the global loads of up to UNR elements (LOAD fills a V) are issued before the first USE consumes
// them: one memory round trip per batch instead of one per element
template <int TM, int UNR, class V, class LD, class USE>
__device__ __forceinline__ void tile_foreach4_ld(int C, LD ldf, USE usef) {
  const int c4n = C >> 2, n = TM * c4n;
  for (int s0 = threadIdx.x; s0 < n; s0 += UNR * NT) {
    V v[UNR];
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      const int s = s0 + u * NT;
      if (s < n) { const int r = s / c4n; ldf(r, 4 * (s - r * c4n), v[u]); }
    }
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      const int s = s0 + u * NT;
      if (s < n) { const int r = s / c4n; usef(r, 4 * (s - r * c4n), v[u]); }
    }
  }
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }

// -------------------------------------------------------------------------------------------------
// post_bwd: adjoint of post_fwd.
// -------------------------------------------------------------------------------------------------
struct PostBwdArgs {
  const float* dout;      // upstream grad wrt block output (nullable == 0)
  const float* out;       // dec: saved block output (for the MSE term)
  const float* enc_in;    // dec: reconstruction target (nullable)
  float mse_coef;         // dec: lambda1 * 2 / (M_total*H)
  float* denc;            // dec: grad wrt enc_in written here (nullable)
  const int* ids;
  const float* ctx; const float* u; const float* h1;   // saved: attention context, y (enc) / c (dec), FFN hidden
  const float* Wo; const float* ln2_g; const float* ln2_b; const float* C1; const float* C2; const float* Wsp; const float* bsp;
  float nll_coef;         // enc: lambda2 / (M_total*nh)   (0 -> no fused NLL grad)
  const float* drec;      // enc: external grad wrt rec [M][nh][nh] (compat mode, nullable)
  float* dctx;            // out: grad wrt attention context
  float* dres;            // out: enc -> dy (grad reaching Qn through the residual) ; dec -> dd (grad wrt d)
  float* gWo; float* gbo; float* gln2_g; float* gln2_b; float* gC1; float* gc1; float* gC2; float* gc2; float* gWsp; float* gbsp;
  int M, H, nh;
  DropDesc drop1, drop2;
  __nv_bfloat16* hoist;   // nullable: [6][M][H] bf16 operand copies (dh2, a, dh1, z, dy|dc, ctx) for the hoisted weight gradients
};

template <int TM, bool IS_DEC, bool MMA>
__global__ void __launch_bounds__(NT) post_bwd_kernel(PostBwdArgs p) {
  extern __shared__ __align__(16) float smem[];
  const int H = p.H, M = p.M;
  const int ld = H + tile_pad<MMA>();
  float* G = smem;            // dO -> (enc) dy
  float* A = G + TM * ld;     // a = relu(h1*m1) -> dh1 -> ctx
  float* Bt = A + TM * ld;    // dh2 -> z -> dz/dc -> dctx
  float* Y = Bt + TM * ld;    // enc: y ; dec: c
  float* Ws = Y + TM * ld;    // weight staging; reused as LN-bwd / sparse-head scratch
  const int row0 = blockIdx.x * TM;
  const int rows = min(TM, M - row0);
  const long long hu = (long long)M * H;                                        // one hoisted operand
  __nv_bfloat16* hz = p.hoist ? p.hoist + (long long)row0 * H : nullptr;        // this tile's rows of operand 0
  __shared__ WStreamState wst;
  if (threadIdx.x == 0) {
    wst.g[0] = GemmDesc{p.C2, H, H, H, 1};
    wst.g[1] = GemmDesc{p.C1, H, H, H, 1};
    wst.g[2] = GemmDesc{p.Wo, H, H, H, 1};
    wst.ng = 3;
  }
  __syncthreads();
  WStream<WS_NST, MMA> ws;
  ws.start(&wst, Ws);

  // 1./2. dO = (dout + mse_coef*(out-enc_in)) * keep ; y/c ; a = relu(h1*m1) ; dh2 = dO*m2
  struct PostLd { float4 g, o, e, y, h; int id; };
  tile_foreach4_ld<TM, 2, PostLd>(H, [&](int r, int c, PostLd& v) {
    v.g = v.o = v.e = v.y = v.h = zero4();
    v.id = 0;
    if (row0 + r < M) {
      const long long gi = (long long)(row0 + r) * H + c;
      if (p.dout) v.g = ld4(p.dout + gi);
      if (IS_DEC && p.enc_in) { v.o = ld4(p.out + gi); v.e = ld4(p.enc_in + gi); }
      v.id = p.ids[row0 + r];
      v.y = ld4(p.u + gi);
      v.h = ld4(p.h1 + gi);
    }
  }, [&](int r, int c, const PostLd& v) {
    float4 g = zero4(), a = zero4(), d2 = zero4();
    if (row0 + r < M) {
      const long long gi = (long long)(row0 + r) * H + c;
      g = v.g;
      if (IS_DEC && p.enc_in) {
        const float4 d = make_float4(p.mse_coef * (v.o.x - v.e.x), p.mse_coef * (v.o.y - v.e.y), p.mse_coef * (v.o.z - v.e.z),
                                     p.mse_coef * (v.o.w - v.e.w));
        g = f4_add(g, d);
        if (p.denc) st4(p.denc + gi, make_float4(-d.x, -d.y, -d.z, -d.w));
      }
      if (v.id == 0) g = zero4();
      float4 h = v.h;
      if (p.drop1.enabled) h = f4_mul(h, drop_mul4(p.drop1, (p.drop1.base + (unsigned long long)gi) >> 2));
      a = make_float4(fmaxf(h.x, 0.f), fmaxf(h.y, 0.f), fmaxf(h.z, 0.f), fmaxf(h.w, 0.f));
      d2 = g;
      if (p.drop2.enabled) d2 = f4_mul(d2, drop_mul4(p.drop2, (p.drop2.base + (unsigned long long)gi) >> 2));
    }
    st4(G + r * ld + c, g);
    st4(A + r * ld + c, a);
    st4(Y + r * ld + c, v.y);
    st4(Bt + r * ld + c, d2);
  });
  __syncthreads();
  // 3. dC2 += dh2^T a ; dc2 += colsum(dh2)
  if (hz) { emit_bf16_tile(Bt, ld, H, rows, hz, H); emit_bf16_tile(A, ld, H, rows, hz + hu, H); }
  else wgrad_any<MMA, true, TM>(Bt, ld, H, A, ld, H, rows, p.gC2, H);
  colsum_atomic(Bt, ld, H, rows, p.gc2);
  // 4. da = dh2 C2 ; dh1 = da * [a>0] * m1   (element-wise overwrite of A; A is not this GEMM's operand)
  gemm_stream<TM, true, WS_NST, MMA>(Bt, ld, ws, 0, [&](int, int r, int col, float4 acc) {
    const float4 a = ld4(A + r * ld + col);
    float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
    if (p.drop1.enabled) m = drop_mul4(p.drop1, (p.drop1.base + (unsigned long long)(row0 + r) * H + col) >> 2);
    st4(A + r * ld + col, make_float4(a.x > 0.f ? acc.x * m.x : 0.f, a.y > 0.f ? acc.y * m.y : 0.f,
                                      a.z > 0.f ? acc.z * m.z : 0.f, a.w > 0.f ? acc.w * m.w : 0.f));
  });
  // 5. z = FFN input (enc: LN2(y) -> Bt ; dec: c == Y) ; dC1 += dh1^T z ; dc1 += colsum(dh1)
  const float* Z = Y;
  if (!IS_DEC) {
    ln_tile<TM>(Y, Bt, ld, H, p.ln2_g, p.ln2_b, 1e-8f, row0, M);
    __syncthreads();
    Z = Bt;
  }
  if (hz) { emit_bf16_tile(A, ld, H, rows, hz + 2 * hu, H); emit_bf16_tile(Z, ld, H, rows, hz + 3 * hu, H); }
  else wgrad_any<MMA, true, TM>(A, ld, H, Z, ld, H, rows, p.gC1, H);
  colsum_atomic(A, ld, H, rows, p.gc1);
  // 6. dz (enc) / dc (dec) = dO + dh1 C1  -> Bt
  gemm_stream<TM, true, WS_NST, MMA>(A, ld, ws, 1, [&](int, int r, int col, float4 acc) {
    st4(Bt + r * ld + col, f4_add(acc, ld4(G + r * ld + col)));
  });
  if (!IS_DEC) {
    // 7. dy = LN2^T(dz) -> G
    ln_bwd_tile<TM, false>(Y, Bt, G, ld, H, p.ln2_g, 1e-8f, row0, M, p.gln2_g, p.gln2_b, ws.scratch());
    // 8. dres = dy ; dWo += dy^T ctx
    store_tile<TM>(G, ld, p.dres, H, 0, H, row0, M);
    load_tile<TM>(A, ld, p.ctx, H, 0, H, row0, M);
    tile_sync();
    if (hz) { emit_bf16_tile(G, ld, H, rows, hz + 4 * hu, H); emit_bf16_tile(A, ld, H, rows, hz + 5 * hu, H); }
    else wgrad_any<MMA, true, TM>(G, ld, H, A, ld, H, rows, p.gWo, H);
    colsum_atomic(G, ld, H, rows, p.gbo);
    // 9. dctx = dy Wo (+ independence-head adjoint) -> Bt -> global
    gemm_stream<TM, true, WS_NST, MMA>(G, ld, ws, 2, [&](int, int r, int col, float4 acc) { st4(Bt + r * ld + col, acc); });
    if (p.nll_coef != 0.f || p.drec) {
      const int nh = p.nh, hd = H / nh, n2 = nh * nh;
      float* lgs = ws.scratch();       // [TM][nh*nh] logits -> dlogits
      float* dbs = lgs + TM * n2;      // [nh] bias-grad partial
      for (int i = threadIdx.x; i < nh; i += NT) dbs[i] = 0.f;
      for (int i = threadIdx.x; i < TM * n2; i += NT) {
        const int r = i / n2, cj = i - r * n2, c = cj / nh, j = cj - c * nh;
        const float* xr = A + r * ld + c * hd;
        const float* wr = p.Wsp + j * hd;
        float sacc = 0.f;
        for (int dd = 0; dd < hd; dd += 4) {
          const float4 x4 = ld4(xr + dd);
          const float4 w4 = __ldg(reinterpret_cast<const float4*>(wr + dd));
          sacc = fmaf(x4.x, w4.x, sacc); sacc = fmaf(x4.y, w4.y, sacc); sacc = fmaf(x4.z, w4.z, sacc); sacc = fmaf(x4.w, w4.w, sacc);
        }
        lgs[i] = sacc + p.bsp[j];
      }
      __syncthreads();
      for (int i = threadIdx.x; i < TM * nh; i += NT) {
        const int r = i / nh, c = i - r * nh;
        float* lg = lgs + r * n2 + c * nh;
        if (r >= rows) {
          for (int j = 0; j < nh; ++j) lg[j] = 0.f;
          continue;
        }
        float mx = lg[0];
        for (int j = 1; j < nh; ++j) mx = fmaxf(mx, lg[j]);
        float se = 0.f;
        for (int j = 0; j < nh; ++j) se += expf(lg[j] - mx);
        const float* dr = p.drec ? p.drec + ((long long)(row0 + r) * nh + c) * nh : nullptr;
        float gsum = 0.f;
        if (dr) for (int j = 0; j < nh; ++j) gsum += dr[j];
        for (int j = 0; j < nh; ++j) {
          const float pj = expf(lg[j] - mx) / se;
          float dl = p.nll_coef * (pj - (j == c ? 1.f : 0.f));
          if (dr) dl += dr[j] - pj * gsum;
          lg[j] = dl;
          atomicAdd(dbs + j, dl);
        }
      }
      __syncthreads();
      // dctx[r][c*hd+d] += sum_j dl[r][c][j] * Wsp[j][d]
      for (int i = threadIdx.x; i < TM * H; i += NT) {
        const int r = i / H, col = i - r * H, c = col / hd, dd = col - c * hd;
        const float* dl = lgs + r * n2 + c * nh;
        float add = 0.f;
        for (int j = 0; j < nh; ++j) add = fmaf(dl[j], p.Wsp[j * hd + dd], add);
        Bt[r * ld + col] += add;
      }
      // dWsp[j][d] += sum_{r,c} dl[r][c][j] * ctx[r][c*hd+d]
      for (int i = threadIdx.x; i < nh * hd; i += NT) {
        const int j = i / hd, dd = i - j * hd;
        float accw = 0.f;
        for (int r = 0; r < rows; ++r)
          for (int c = 0; c < nh; ++c) accw = fmaf(lgs[r * n2 + c * nh + j], A[r * ld + c * hd + dd], accw);
        atomicAdd(p.gWsp + i, accw);
      }
      for (int i = threadIdx.x; i < nh; i += NT) atomicAdd(p.gbsp + i, dbs[i]);
      __syncthreads();
    }
    store_tile<TM>(Bt, ld, p.dctx, H, 0, H, row0, M);
  } else {
    // 7. dres = dd = dO ; dWo += dc^T ctx ; dctx = dc Wo
    store_tile<TM>(G, ld, p.dres, H, 0, H, row0, M);
    load_tile<TM>(A, ld, p.ctx, H, 0, H, row0, M);
    tile_sync();
    if (hz) { emit_bf16_tile(Bt, ld, H, rows, hz + 4 * hu, H); emit_bf16_tile(A, ld, H, rows, hz + 5 * hu, H); }
    else wgrad_any<MMA, true, TM>(Bt, ld, H, A, ld, H, rows, p.gWo, H);
    colsum_atomic(Bt, ld, H, rows, p.gbo);
    gemm_stream<TM, true, WS_NST, MMA>(Bt, ld, ws, 2, [&](int, int r, int col, float4 acc) {
      if (row0 + r < M) st4(p.dctx + (long long)(row0 + r) * H + col, acc);
    });
  }
}

// -------------------------------------------------------------------------------------------------
// attn_bwd: adjoint of attn_fwd for one (query tile, head, sequence).  Recomputes P from q,k and the saved
// log-sum-exp; dq is owned by the CTA (plain stores), dk/dv are accumulated with vector atomics because
// several query tiles of a sequence contribute to the same keys.
// -------------------------------------------------------------------------------------------------
template <int TM, bool MMA>
__global__ void __launch_bounds__(NT) attn_bwd_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                      const float* __restrict__ v, const float* __restrict__ dctx,
                                                      const float* __restrict__ lse, const int* __restrict__ key_ids,
                                                      float* __restrict__ dq, float* __restrict__ dk, float* __restrict__ dv, int L,
                                                      int H, int nh, int mask_mode, DropDesc drop) {
  extern __shared__ __align__(16) float smem[];
  const int hd = H / nh;
  const int ldq = hd + tile_pad<MMA>();
  const int lds = ((L + 3) & ~3) + tile_pad<MMA>();
  float* Qs = smem;
  float* dCs = Qs + TM * ldq;
  float* Ps = dCs + TM * ldq;
  float* dPs = Ps + TM * lds;
  float* Ws = dPs + TM * lds;
  const int i0 = blockIdx.x * TM, h = blockIdx.y, b = blockIdx.z;
  const long long seq_off = (long long)b * L * H + (long long)h * hd;
  const int Lk = mask_mode == 0 ? min(L, i0 + TM) : L;
  const int Lk4 = (Lk + 3) & ~3;
  const int rows = min(TM, L - i0);

  __shared__ WStreamState wst;
  if (threadIdx.x == 0) {
    wst.g[0] = GemmDesc{k + seq_off, H, Lk, hd, 0};
    wst.g[1] = GemmDesc{v + seq_off, H, Lk, hd, 0};
    wst.g[2] = GemmDesc{k + seq_off, H, hd, Lk, 1};
    wst.ng = 3;
  }
  __syncthreads();
  WStream<WS_NST, MMA> ws;
  ADT_STAMP(36);
  ws.start(&wst, Ws);
  load_tile<TM>(Qs, ldq, q + seq_off, H, 0, hd, i0, L);
  load_tile<TM>(dCs, ldq, dctx + seq_off, H, 0, hd, i0, L);
  tile_sync();
  ADT_STAMP(37);
  gemm_stream<TM, false, WS_NST, MMA>(Qs, ldq, ws, 0, [&](int, int r, int col, float4 a) { st4(Ps + r * lds + col, a); });
  ADT_STAMP(38);
  gemm_stream<TM, false, WS_NST, MMA>(dCs, ldq, ws, 1, [&](int, int r, int col, float4 a) { st4(dPs + r * lds + col, a); });
  ADT_STAMP(39);

  // per-row part, LPR lanes per row / 32/LPR rows side by side per warp (see attn_fwd)
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int lpr = Lk4 <= 64 ? 8 : 32;
  const int rpw = 32 / lpr;
  const int sub = l % lpr;
  for (int r = w * rpw + l / lpr; r < TM; r += (NT / 32) * rpw) {
    const int i = i0 + r;
    float* prow = Ps + r * lds;
    float* drow = dPs + r * lds;
    const bool valid = i < L;
    const int nj = !valid ? 0 : (mask_mode == 0 ? i + 1 : L);
    const float ls = valid ? lse[((long long)b * nh + h) * L + i] : 0.f;
    const int j0 = 8 * sub;
    float sv[8], dv8[8], mv[8];
    {
      float4 s0 = zero4(), s1 = zero4(), d0 = zero4(), d1 = zero4();
      if (j0 < nj) { s0 = ld4(prow + j0); d0 = ld4(drow + j0); }
      if (j0 + 4 < nj) { s1 = ld4(prow + j0 + 4); d1 = ld4(drow + j0 + 4); }
      sv[0] = s0.x; sv[1] = s0.y; sv[2] = s0.z; sv[3] = s0.w; sv[4] = s1.x; sv[5] = s1.y; sv[6] = s1.z; sv[7] = s1.w;
      dv8[0] = d0.x; dv8[1] = d0.y; dv8[2] = d0.z; dv8[3] = d0.w; dv8[4] = d1.x; dv8[5] = d1.y; dv8[6] = d1.z; dv8[7] = d1.w;
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) mv[c] = 1.f;
    if (drop.enabled && j0 < nj) drop_mul8_attn(drop, drop.base + ((unsigned long long)b * nh + h) * L + i, ((L + 7) & ~7) >> 3, sub, mv);
    float delta = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float pj = 0.f, dp = 0.f;
      if (j0 + c < nj) {
        float sc = sv[c];
        if (mask_mode == 1 && key_ids[b * L + j0 + c] == 0) sc = -1e9f;
        pj = expf(sc - ls);
        dp = dv8[c] * mv[c];
        delta = fmaf(dp, pj, delta);
      }
      sv[c] = pj; dv8[c] = dp;
    }
    for (int o = lpr >> 1; o > 0; o >>= 1) delta += __shfl_xor_sync(0xffffffffu, delta, o);
    if (j0 < Lk4) {
      st4(prow + j0, make_float4(sv[0] * mv[0], sv[1] * mv[1], sv[2] * mv[2], sv[3] * mv[3]));
      st4(drow + j0, make_float4(sv[0] * (dv8[0] - delta), sv[1] * (dv8[1] - delta), sv[2] * (dv8[2] - delta), sv[3] * (dv8[3] - delta)));
    }
    if (j0 + 4 < Lk4) {
      st4(prow + j0 + 4, make_float4(sv[4] * mv[4], sv[5] * mv[5], sv[6] * mv[6], sv[7] * mv[7]));
      st4(drow + j0 + 4, make_float4(sv[4] * (dv8[4] - delta), sv[5] * (dv8[5] - delta), sv[6] * (dv8[6] - delta), sv[7] * (dv8[7] - delta)));
    }
  }
  __syncthreads();
  ADT_STAMP(40);
  // dq = dS k
  gemm_stream<TM, true, WS_NST, MMA>(dPs, lds, ws, 2, [&](int, int r, int col, float4 a) {
    if (i0 + r < L) st4(dq + seq_off + (long long)(i0 + r) * H + col, a);
  });
  ADT_STAMP(41);
  // dk += dS^T q ; dv += Pd^T dctx   (plain stores when this CTA is the only query tile of the sequence)
  if (gridDim.x == 1) {
    wgrad_any<MMA, false, TM>(dPs, lds, Lk, Qs, ldq, hd, rows, dk + seq_off, H);
    wgrad_any<MMA, false, TM>(Ps, lds, Lk, dCs, ldq, hd, rows, dv + seq_off, H);
  } else {
    wgrad_any<MMA, true, TM>(dPs, lds, Lk, Qs, ldq, hd, rows, dk + seq_off, H);
    wgrad_any<MMA, true, TM>(Ps, lds, Lk, dCs, ldq, hd, rows, dv + seq_off, H);
  }
  ADT_STAMP(42);
}

// -------------------------------------------------------------------------------------------------
// mid_bwd (decoder): adjoint of mid_fwd.
// -------------------------------------------------------------------------------------------------
struct MidBwdArgs {
  const float* dq2; const float* dk2; const float* dv2;
  const float* a; const float* feats; const float* ctx1;
  const float* Wo1; const float* Win2;
  float* dfeats;   // accumulated (+=) : several decoder layers and the logits feed the same encoder features
  float* dctx1;
  float* gWo1; float* gbo1; float* gWin2; float* gbin2;
  int M, H; float qscale;
  __nv_bfloat16* hoist;   // nullable: [7][M][H] bf16: dq2*s, a, [dk2|dv2] as one [M][2H], feats, da, ctx1
};

template <int TM, bool MMA>
__global__ void __launch_bounds__(NT) mid_bwd_kernel(MidBwdArgs p) {
  extern __shared__ __align__(16) float smem[];
  const int H = p.H, M = p.M;
  const int ld = H + tile_pad<MMA>(), ld2 = 2 * H + tile_pad<MMA>();
  float* T0 = smem;              // dq2*scale
  float* T1 = T0 + TM * ld;      // a -> feats -> ctx1
  float* DA = T1 + TM * ld;      // grad wrt a
  float* KV = DA + TM * ld;      // [dk2 | dv2]
  float* Ws = KV + TM * ld2;
  const int row0 = blockIdx.x * TM;
  const int rows = min(TM, M - row0);
  __shared__ WStreamState wst;
  if (threadIdx.x == 0) {
    wst.g[0] = GemmDesc{p.Win2, H, H, H, 1};
    wst.g[1] = GemmDesc{p.Win2 + (long long)H * H, H, H, 2 * H, 1};
    wst.g[2] = GemmDesc{p.Wo1, H, H, H, 1};
    wst.ng = 3;
  }
  __syncthreads();
  WStream<WS_NST, MMA> ws;
  ws.start(&wst, Ws);
  struct Ld2 { float4 a, b; };
  tile_foreach4_ld<TM, 4, Ld2>(H, [&](int r, int c, Ld2& v) {
    v.a = v.b = zero4();
    if (row0 + r < M) {
      const long long gi = (long long)(row0 + r) * H + c;
      v.a = ld4(p.dq2 + gi);
      v.b = ld4(p.a + gi);
    }
  }, [&](int r, int c, const Ld2& v) {
    st4(T0 + r * ld + c, f4_scale(v.a, p.qscale));
    st4(T1 + r * ld + c, v.b);
  });
  __syncthreads();
  const long long hu = (long long)M * H;
  __nv_bfloat16* hz = p.hoist ? p.hoist + (long long)row0 * H : nullptr;
  if (hz) { emit_bf16_tile(T0, ld, H, rows, hz, H); emit_bf16_tile(T1, ld, H, rows, hz + hu, H); }
  else wgrad_any<MMA, true, TM>(T0, ld, H, T1, ld, H, rows, p.gWin2, H);
  colsum_atomic(T0, ld, H, rows, p.gbin2);
  gemm_stream<TM, true, WS_NST, MMA>(T0, ld, ws, 0, [&](int, int r, int col, float4 acc) { st4(DA + r * ld + col, acc); });
  load_tile<TM>(KV, ld2, p.dk2, H, 0, H, row0, M);
  load_tile<TM>(KV + H, ld2, p.dv2, H, 0, H, row0, M);
  load_tile<TM>(T1, ld, p.feats, H, 0, H, row0, M);
  tile_sync();
  if (hz) { emit_bf16_tile(KV, ld2, 2 * H, rows, p.hoist + 2 * hu + (long long)row0 * 2 * H, 2 * H); emit_bf16_tile(T1, ld, H, rows, hz + 4 * hu, H); }
  else wgrad_any<MMA, true, TM>(KV, ld2, 2 * H, T1, ld, H, rows, p.gWin2 + (long long)H * H, H);
  colsum_atomic(KV, ld2, 2 * H, rows, p.gbin2 + H);
  gemm_stream<TM, true, WS_NST, MMA>(KV, ld2, ws, 1, [&](int, int r, int col, float4 acc) {
    if (row0 + r < M) {
      float* d = p.dfeats + (long long)(row0 + r) * H + col;
      st4(d, f4_add(ld4(d), acc));
    }
  });
  load_tile<TM>(T1, ld, p.ctx1, H, 0, H, row0, M);
  tile_sync();
  if (hz) { emit_bf16_tile(DA, ld, H, rows, hz + 5 * hu, H); emit_bf16_tile(T1, ld, H, rows, hz + 6 * hu, H); }
  else wgrad_any<MMA, true, TM>(DA, ld, H, T1, ld, H, rows, p.gWo1, H);
  colsum_atomic(DA, ld, H, rows, p.gbo1);
  gemm_stream<TM, true, WS_NST, MMA>(DA, ld, ws, 2, [&](int, int r, int col, float4 acc) {
    if (row0 + r < M) st4(p.dctx1 + (long long)(row0 + r) * H + col, acc);
  });
}

// -------------------------------------------------------------------------------------------------
// pre_bwd: adjoint of pre_fwd.
//   dx = LN^T( dnorm_extra + dq*s Wq [+ dk Wk + dv Wv if kv_from_norm] ) [+ dk Wk + dv Wv if !kv_from_norm] + dx_extra
// -------------------------------------------------------------------------------------------------
struct PreBwdArgs {
  const float* dq; const float* dk; const float* dv;
  const float* x;
  const float* dnorm_extra;   // enc: dy from post_bwd ; dec: dd from post_bwd (nullable)
  const float* dx_extra;      // extra grad added to dx (enc: MSE grad wrt enc_in), nullable
  const float* ln_g; const float* ln_b; const float* Win;
  float* dx;
  float* gWin; float* gbin; float* gln_g; float* gln_b;
  int M, H; float qscale; int kv_from_norm;
  __nv_bfloat16* hoist;   // nullable: [5][M][H] bf16: [dq*s | dk | dv] as one [M][3H], LN(x), x
};

template <int TM, bool MMA>
__global__ void __launch_bounds__(NT) pre_bwd_kernel(PreBwdArgs p) {
  extern __shared__ __align__(16) float smem[];
  const int H = p.H, M = p.M;
  const int ld = H + tile_pad<MMA>();
  float* X = smem;
  float* N = X + TM * ld;
  float* T = N + TM * ld;
  float* D = T + TM * ld;
  float* Ws = D + TM * ld;
  const int row0 = blockIdx.x * TM;
  const int rows = min(TM, M - row0);
  __shared__ WStreamState wst;
  if (threadIdx.x == 0) {
    wst.g[0] = GemmDesc{p.Win, H, H, H, 1};
    wst.g[1] = GemmDesc{p.Win + (long long)H * H, H, H, H, 1};
    wst.g[2] = GemmDesc{p.Win + 2ll * H * H, H, H, H, 1};
    wst.ng = 3;
  }
  __syncthreads();
  WStream<WS_NST, MMA> ws;
  ws.start(&wst, Ws);
  ADT_STAMP(24);
  struct Ld2 { float4 a, b; };
  tile_foreach4_ld<TM, 4, Ld2>(H, [&](int r, int c, Ld2& v) {
    v.a = v.b = zero4();
    if (row0 + r < M) {
      const long long gi = (long long)(row0 + r) * H + c;
      v.a = ld4(p.x + gi);
      v.b = ld4(p.dq + gi);
    }
  }, [&](int r, int c, const Ld2& v) {
    st4(X + r * ld + c, v.a);
    st4(T + r * ld + c, f4_scale(v.b, p.qscale));
  });
  __syncthreads();
  ADT_STAMP(25);
  ln_tile<TM>(X, N, ld, H, p.ln_g, p.ln_b, 1e-8f, row0, M);
  __syncthreads();
  ADT_STAMP(26);
  const long long hu = (long long)M * H;
  __nv_bfloat16* hq = p.hoist ? p.hoist + (long long)row0 * 3 * H : nullptr;    // [M][3H] row of this tile
  if (hq) {
    emit_bf16_tile(T, ld, H, rows, hq, 3 * H);
    emit_bf16_tile(N, ld, H, rows, p.hoist + 3 * hu + (long long)row0 * H, H);
    if (!p.kv_from_norm) emit_bf16_tile(X, ld, H, rows, p.hoist + 4 * hu + (long long)row0 * H, H);
  } else wgrad_any<MMA, true, TM>(T, ld, H, N, ld, H, rows, p.gWin, H);
  ADT_STAMP(27);
  colsum_atomic(T, ld, H, rows, p.gbin);
  ADT_STAMP(28);
  gemm_stream<TM, true, WS_NST, MMA>(T, ld, ws, 0, [&](int, int r, int col, float4 acc) {
    if (p.dnorm_extra && row0 + r < M) acc = f4_add(acc, ld4(p.dnorm_extra + (long long)(row0 + r) * H + col));
    st4(D + r * ld + col, acc);
  });
  ADT_STAMP(29);
  if (!p.kv_from_norm) ln_bwd_tile<TM, false>(X, D, D, ld, H, p.ln_g, 1e-8f, row0, M, p.gln_g, p.gln_b, ws.scratch());
  ADT_STAMP(30);
  const float* Xkv = p.kv_from_norm ? N : X;
  for (int which = 0; which < 2; ++which) {
    load_tile<TM>(T, ld, which == 0 ? p.dk : p.dv, H, 0, H, row0, M);
    tile_sync();
    if (hq) emit_bf16_tile(T, ld, H, rows, hq + (1 + which) * H, 3 * H);
    else wgrad_any<MMA, true, TM>(T, ld, H, Xkv, ld, H, rows, p.gWin + (long long)(1 + which) * H * H, H);
    colsum_atomic(T, ld, H, rows, p.gbin + (1 + which) * H);
    gemm_stream<TM, true, WS_NST, MMA>(T, ld, ws, 1 + which, [&](int, int r, int col, float4 acc) {
      st4(D + r * ld + col, f4_add(acc, ld4(D + r * ld + col)));
    });
  }
  ADT_STAMP(31);
  if (p.kv_from_norm) ln_bwd_tile<TM, false>(X, D, D, ld, H, p.ln_g, 1e-8f, row0, M, p.gln_g, p.gln_b, ws.scratch());
  ADT_STAMP(32);
  struct Ld1 { float4 a; };
  tile_foreach4_ld<TM, 4, Ld1>(H, [&](int r, int c, Ld1& v) {
    v.a = zero4();
    if (p.dx_extra && row0 + r < M) v.a = ld4(p.dx_extra + (long long)(row0 + r) * H + c);
  }, [&](int r, int c, const Ld1& v) {
    if (row0 + r < M) st4(p.dx + (long long)(row0 + r) * H + c, f4_add(ld4(D + r * ld + c), v.a));
  });
  ADT_STAMP(33);
}

// -------------------------------------------------------------------------------------------------
// final_bwd: adjoint of final_fwd (+ BCE).  Warp per row.
//   dpl = -sigmoid(-pl)/n * [pos!=0] (+ ext) ; dnl = sigmoid(nl)/n * [pos!=0] (+ ext)
//   dfeats = dfeats_in + dpl*E[pos] + dnl*E[neg] ; dx = LN^T(dfeats)
//   cpos/cneg (the per-row coefficients of the item-table gradient rows dpl*feats, dnl*feats) are written for
//   the scatter-add kernel.
// -------------------------------------------------------------------------------------------------
struct FinalBwdArgs {
  const float* x; const float* ln_g; const float* E; const int* pos; const int* neg;
  const float* pos_logits; const float* neg_logits;
  const float* dfeats_in;      // nullable
  const double* n_valid;       // device scalar: number of valid (pos != 0) positions of the GLOBAL batch
  float bce_weight;            // 1 for the fused loss, 0 when only external grads are given
  const float* dpl_ext; const float* dnl_ext;   // compat-mode external grads (nullable)
  float* dx; float* cpos; float* cneg; float* gln_g; float* gln_b;
  int M, H;
};

template <int U>
__global__ void __launch_bounds__(NT) final_bwd_kernel(FinalBwdArgs p) {
  __shared__ float red[2 * (NT / 32) * 32 * U];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int H = p.H;
  constexpr int NW = NT / 32;
  float dg[U], db[U];
#pragma unroll
  for (int u = 0; u < U; ++u) dg[u] = db[u] = 0.f;
  const float inv_n = p.bce_weight != 0.f ? (float)(1.0 / fmax(*p.n_valid, 1.0)) * p.bce_weight : 0.f;
  for (int row = blockIdx.x * NW + w; row < p.M; row += gridDim.x * NW) {
    const int pi = p.pos[row], ni = p.neg[row];
    float dpl = 0.f, dnl = 0.f;
    if (pi != 0) {
      const float pl = p.pos_logits[row], nl = p.neg_logits[row];
      dpl = -inv_n / (1.f + expf(pl));
      dnl = inv_n / (1.f + expf(-nl));
    }
    if (p.dpl_ext) dpl += p.dpl_ext[row];
    if (p.dnl_ext) dnl += p.dnl_ext[row];
    if (l == 0) { p.cpos[row] = dpl; p.cneg[row] = dnl; }
    const float* xr = p.x + (long long)row * H;
    float xv[U], gv[U];
    float sum = 0.f;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = l + 32 * u;
      xv[u] = c < H ? xr[c] : 0.f;
      sum += xv[u];
      float g = 0.f;
      if (c < H) {
        if (p.dfeats_in) g = p.dfeats_in[(long long)row * H + c];
        g = fmaf(dpl, p.E[(long long)pi * H + c], g);
        g = fmaf(dnl, p.E[(long long)ni * H + c], g);
      }
      gv[u] = g;
    }
    if (!p.ln_g) {
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (l + 32 * u < H) p.dx[(long long)row * H + l + 32 * u] = gv[u];
      continue;
    }
    const float mean = warp_sum(sum) / (float)H;
    float var = 0.f;
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (l + 32 * u < H) { const float t = xv[u] - mean; var += t * t; }
    const float rstd = 1.0f / sqrtf(warp_sum(var) / (float)H + 1e-8f);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = l + 32 * u;
      if (c < H) {
        const float xh = (xv[u] - mean) * rstd;
        const float gg = gv[u] * p.ln_g[c];
        s1 += gg; s2 += gg * xh;
        dg[u] += gv[u] * xh; db[u] += gv[u];
      }
    }
    s1 = warp_sum(s1) / (float)H;
    s2 = warp_sum(s2) / (float)H;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = l + 32 * u;
      if (c < H) {
        const float xh = (xv[u] - mean) * rstd;
        p.dx[(long long)row * H + c] = rstd * (gv[u] * p.ln_g[c] - s1 - xh * s2);
      }
    }
  }
  if (p.ln_g) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = l + 32 * u;
      if (c < H) { red[w * H + c] = dg[u]; red[(NW + w) * H + c] = db[u]; }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < H; c += NT) {
      float a = 0.f, b = 0.f;
      for (int i = 0; i < NW; ++i) { a += red[i * H + c]; b += red[(NW + i) * H + c]; }
      atomicAdd(p.gln_g + c, a);
      atomicAdd(p.gln_b + c, b);
    }
  }
}

// -------------------------------------------------------------------------------------------------
// pos_emb gradient: dP[t][c] += sum_b dx[b][t][c] * m(b,t,c) * [id != 0]    (adjoint of K1 wrt pos_emb)
// One CTA per group of BS sequences: every thread walks the contiguous [L, H] slab of a sequence (fully coalesced 128-bit
// reads), sums its (t, c4) position over the group in registers, then one vector atomic per position.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT) posgrad_kernel(const float* __restrict__ dx0, const int* __restrict__ ids0, DropDesc drop0,
                                                     const float* __restrict__ dx1, const int* __restrict__ ids1, DropDesc drop1,
                                                     float* __restrict__ gP, int B, int L, int H, int BS) {
  // blockIdx.y selects the lookup (0: encoder sequence, 1: decoder sequence); a null dx skips it
  const float* dx = blockIdx.y == 0 ? dx0 : dx1;
  if (!dx) return;
  const int* ids = blockIdx.y == 0 ? ids0 : ids1;
  const DropDesc drop = blockIdx.y == 0 ? drop0 : drop1;
  const int h4 = H >> 2, n = L * h4;
  const int b0 = blockIdx.x * BS, b1 = min(B, b0 + BS);
  for (int s = threadIdx.x; s < n; s += NT) {
    const int t = s / h4, c4 = s - t * h4;
    float4 acc = zero4();
    for (int b = b0; b < b1; ++b) {
      const int row = b * L + t;
      if (__ldg(ids + row) == 0) continue;
      const long long gi = (long long)row * H + 4 * c4;
      float4 g = ld4(dx + gi);
      if (drop.enabled) g = f4_mul(g, drop_mul4(drop, (drop.base + (unsigned long long)gi) >> 2));
      acc = f4_add(acc, g);
    }
    atomicAdd(reinterpret_cast<float4*>(gP + (long long)t * H) + c4, acc);
  }
}

}  // namespace adt
