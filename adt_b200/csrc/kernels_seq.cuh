// Sequence-resident encoder block for evaluation: short sequences (L <= 64) of narrow models (H == 64) in the bf16 tensor-core mode.
// ONE 128-thread CTA owns ONE whole sequence and runs a complete encoder block on it -- LayerNorm -> packed QKV projection -> causal
// softmax attention (all heads) -> out-projection -> LayerNorm -> FFN -> residual / pad mask (+ the independence head's log-probs) --
// with the sequence's q, k, v, probabilities and context living in shared memory / MMA fragments.  Nothing but the block input and
// the block output touches HBM, and a block is ONE launch instead of three.  Training runs the row-tile kernels: they overlap
// across the two streams of the step graph, and a CTA that pins 83 KB of shared memory per SM would not
// (profiles/r02_seq_kernel_variants.md).
// Reference semantics: EncoderLayer.forward sasrec/modules.py:644-655, MultiheadAttentionADT :270-527, PointWiseFeedForward
// :629-633, SparseInputLinear :696-703 (SURVEY.md appendix A).
//
// Weights: the kernel takes the fp32 parameters (converted on the fly) or, when the caller keeps a bf16 mirror of the flat
// parameter buffer (written by the Adam kernel), cp.asyncs them straight into the padded shared-memory tiles.
// Shared-memory budget: 83 KB per CTA so that two CTAs (two sequences) are resident per SM: 256 sequences = one wave.
#pragma once
#include "kernels_rowtile_small.cuh"

namespace adt {

constexpr int SQ_NT = AS_NT;      // 128 threads = 4 warps x 16 rows = the 64-row sequence tile

struct SeqW {                     // bf16 mirror of the flat fp32 parameter buffer (base16 == nullptr: convert from fp32)
  const float* base32; const __nv_bfloat16* base16;
};

// N weight matrices [64][64] (row-major, nn.Linear layout [out][in]) -> bf16 tiles [64][72].  Mirror present: 16-byte cp.async
// pieces, completed by the caller's sq_weights_wait(); otherwise fp32 loads + conversion in registers.
template <int N>
__device__ __forceinline__ void sq_load_weights(const float* const (&w)[N], const SeqW& s, __nv_bfloat16* tiles) {
  if (s.base16) {
#pragma unroll
    for (int n = 0; n < N; ++n) {
      const __nv_bfloat16* src = s.base16 + (w[n] - s.base32);
      __nv_bfloat16* dst = tiles + n * RS_TILE;
#pragma unroll
      for (int it = 0; it < 512 / SQ_NT; ++it) {
        const int i = threadIdx.x + it * SQ_NT, r = i >> 3, c = i & 7;
        cp_async16(dst + r * RS_LD + 8 * c, src + r * RS_H + 8 * c, true);
      }
    }
    cp_async_commit();
  } else {
    long long lds[N]; int nr[N]; float sc[N]; __nv_bfloat16* d[N]; __nv_bfloat16* dT[N]; float* dF[N];
#pragma unroll
    for (int n = 0; n < N; ++n) { lds[n] = RS_H; nr[n] = 64; sc[n] = 1.f; d[n] = tiles + n * RS_TILE; dT[n] = nullptr; dF[n] = nullptr; }
    rs_load<N>(w, lds, nr, sc, d, dT, dF);
  }
}
__device__ __forceinline__ void sq_weights_wait() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// warp-level double sum -> one atomicAdd per warp
__device__ __forceinline__ void warp_accumulate(double v, double* dst) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(dst, v);
}

__device__ __forceinline__ void frag_zero(float (&v)[8][4]) {
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) v[nb][0] = v[nb][1] = v[nb][2] = v[nb][3] = 0.f;
}
__device__ __forceinline__ void frag_mask_rows(float (&v)[8][4], bool v0, bool v1) {
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    if (!v0) { v[nb][0] = 0.f; v[nb][1] = 0.f; }
    if (!v1) { v[nb][2] = 0.f; v[nb][3] = 0.f; }
  }
}
// v = (v + bias[col]) * scale at the fragment positions
__device__ __forceinline__ void frag_bias_scale(float (&v)[8][4], const float* __restrict__ bias, float scale, int t) {
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const float2 b = __ldg(reinterpret_cast<const float2*>(bias + 8 * nb + 2 * t));
    v[nb][0] = (v[nb][0] + b.x) * scale; v[nb][1] = (v[nb][1] + b.y) * scale;
    v[nb][2] = (v[nb][2] + b.x) * scale; v[nb][3] = (v[nb][3] + b.y) * scale;
  }
}

// ---------------------------------------------------------------------------------------------------------------------------------
// causal / key-padding softmax attention of ONE sequence, all heads, operands in full-width bf16 tiles [64][72] (heads are column
// slices).  Returns the context in fragments (rows i0 / i1 of this thread, all 64 columns).  Same arithmetic and masks as
// attn_small_fwd_kernel without dropout.
// ---------------------------------------------------------------------------------------------------------------------------------
template <int HD>
__device__ __forceinline__ void sq_attn_fwd(float (&ctxf)[8][4], const __nv_bfloat16* __restrict__ Qs, const __nv_bfloat16* __restrict__ Ks,
                                            const __nv_bfloat16* __restrict__ Vs, int L, int mask_mode, const int* __restrict__ kid) {
  constexpr int NH = RS_H / HD;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * w + g, i1 = i0 + 8;
  const bool v0 = i0 < L, v1 = i1 < L;
  const int nbr = (L + 7) >> 3, nks = (L + 15) >> 4;
#pragma unroll
  for (int h = 0; h < NH; ++h) {
    float s[8][4];
    frag_zero(s);
#pragma unroll
    for (int ks = 0; ks < HD / 16; ++ks) {
      uint32_t a[4];
      lm_a<RS_LD>(a, Qs + h * HD, 16 * w, 16 * ks);
#pragma unroll
      for (int nb = 0; nb < 8; ++nb) {
        if (nb < nbr) {
          uint32_t b0, b1;
          lm_b<RS_LD>(b0, b1, Ks + h * HD, 8 * nb, 16 * ks);
          mma16816(s[nb], a, b0, b1);
        }
      }
    }
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int j = 8 * nb + 2 * t + e;
        s[nb][e] = as_masked(s[nb][e], i0, j, L, mask_mode, kid);
        s[nb][2 + e] = as_masked(s[nb][2 + e], i1, j, L, mask_mode, kid);
        mx0 = fmaxf(mx0, s[nb][e]);
        mx1 = fmaxf(mx1, s[nb][2 + e]);
      }
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const float e0 = s[nb][e] == -INFINITY ? 0.f : expf(s[nb][e] - mx0);
        const float e1 = s[nb][2 + e] == -INFINITY ? 0.f : expf(s[nb][2 + e] - mx1);
        s[nb][e] = e0; s[nb][2 + e] = e1;
        sum0 += e0; sum1 += e1;
      }
    }
    sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1); sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
    sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1); sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
    const float inv0 = v0 ? 1.0f / sum0 : 0.f, inv1 = v1 ? 1.0f / sum1 : 0.f;
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) { s[nb][0] *= inv0; s[nb][1] *= inv0; s[nb][2] *= inv1; s[nb][3] *= inv1; }
    float o[HD / 8][4];
#pragma unroll
    for (int db = 0; db < HD / 8; ++db) o[db][0] = o[db][1] = o[db][2] = o[db][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      if (ks < nks) {
        uint32_t a[4];
        a[0] = pack_bf16(s[2 * ks][0], s[2 * ks][1]);
        a[1] = pack_bf16(s[2 * ks][2], s[2 * ks][3]);
        a[2] = pack_bf16(s[2 * ks + 1][0], s[2 * ks + 1][1]);
        a[3] = pack_bf16(s[2 * ks + 1][2], s[2 * ks + 1][3]);
#pragma unroll
        for (int db = 0; db < HD / 8; ++db) {
          uint32_t b0, b1;
          lm_b_t<RS_LD>(b0, b1, Vs + h * HD, 16 * ks, 8 * db);
          mma16816(o[db], a, b0, b1);
        }
      }
    }
#pragma unroll
    for (int db = 0; db < HD / 8; ++db) {
      ctxf[h * (HD / 8) + db][0] = o[db][0]; ctxf[h * (HD / 8) + db][1] = o[db][1];
      ctxf[h * (HD / 8) + db][2] = o[db][2]; ctxf[h * (HD / 8) + db][3] = o[db][3];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------------------
// FFN tail: u = z in fragments -> out = relu(u C1^T + c1) C2^T + c2 + u
// ---------------------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void sq_ffn_fwd(float (&y)[8][4], const float (&u)[8][4], const __nv_bfloat16* __restrict__ C1t,
                                           const __nv_bfloat16* __restrict__ C2t, const float* __restrict__ c1, const float* __restrict__ c2,
                                           int t) {
  float h[8][4];
  frag_zero(h);
  rs_fgemm_frag(h, u, C1t);
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    const float2 b = __ldg(reinterpret_cast<const float2*>(c1 + c));
    h[nb][0] += b.x; h[nb][1] += b.y; h[nb][2] += b.x; h[nb][3] += b.y;
#pragma unroll
    for (int e = 0; e < 4; ++e) h[nb][e] = fmaxf(h[nb][e], 0.f);
  }
  frag_zero(y);
  rs_fgemm_frag(y, h, C2t);
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    const float2 b = __ldg(reinterpret_cast<const float2*>(c2 + c));
    y[nb][0] += b.x; y[nb][1] += b.y; y[nb][2] += b.x; y[nb][3] += b.y;
#pragma unroll
    for (int e = 0; e < 4; ++e) y[nb][e] += u[nb][e];
  }
}

// ---------------------------------------------------------------------------------------------------------------------------------
// Encoder block forward in evaluation mode, one sequence per CTA.
// ---------------------------------------------------------------------------------------------------------------------------------
struct EncSeqFwdArgs {
  const float* x; const int* ids;
  const float* ln1_g; const float* ln1_b; const float* Win; const float* bin; const float* Wo; const float* bo;
  const float* ln2_g; const float* ln2_b; const float* C1; const float* c1; const float* C2; const float* c2;
  const float* Wsp; const float* bsp;
  float* out;                                                                  // [M][64] (nullable when out_last is given)
  float* out_last;                                                             // optional [B][64]: the block output of position L-1 only
  float* rec; double* nll_acc;
  int B, L, mask_mode; float qscale;
  SeqW w;
};

struct EncSeqFwdSmem {
  static constexpr int W = 0, Q = 6 * RS_TILE, K = Q + RS_TILE, V = K + RS_TILE;     // Wq Wk Wv Wo C1 C2 | Q (later ctx) | K | V
  static constexpr size_t TOTAL_BYTES = (size_t)(V + RS_TILE) * 2;
};

template <int HD>
__global__ void __launch_bounds__(SQ_NT, 2) enc_seq_fwd_kernel(EncSeqFwdArgs p) {
  using SM = EncSeqFwdSmem;
  constexpr int NH = RS_H / HD;
  extern __shared__ __align__(16) uint8_t rs_raw[];
  __nv_bfloat16* hb = reinterpret_cast<__nv_bfloat16*>(rs_raw);
  __nv_bfloat16* Wt = hb + SM::W;
  __nv_bfloat16* Qs = hb + SM::Q;
  __nv_bfloat16* Ks = hb + SM::K;
  __nv_bfloat16* Vs = hb + SM::V;
  const int b = blockIdx.x, L = p.L;
  const long long grow0 = (long long)b * L;           // first global row of this sequence
  const long long g0 = grow0 * RS_H;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * w + g, i1 = i0 + 8;
  const bool v0 = i0 < L, v1 = i1 < L;
  ADT_STAMP(48);
  {
    const float* const w6a[3] = {p.Win, p.Win + RS_H * RS_H, p.Win + 2 * RS_H * RS_H};
    const float* const w6b[3] = {p.Wo, p.C1, p.C2};
    sq_load_weights<3>(w6a, p.w, Wt);
    sq_load_weights<3>(w6b, p.w, Wt + 3 * RS_TILE);
  }
  float Xf[8][4], Nf[8][4];
  frag_load(Xf, p.x + g0, i0, i1, v0, v1, t);
  const int keep0 = v0 ? p.ids[grow0 + i0] : 0, keep1 = v1 ? p.ids[grow0 + i1] : 0;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) { Nf[nb][0] = Xf[nb][0]; Nf[nb][1] = Xf[nb][1]; Nf[nb][2] = Xf[nb][2]; Nf[nb][3] = Xf[nb][3]; }
  frag_ln(Nf, p.ln1_g, p.ln1_b, t);                   // Qn = LN1(x)
  frag_mask_rows(Nf, v0, v1);
  ADT_STAMP(49);
  sq_weights_wait();
  __syncthreads();
  ADT_STAMP(50);
  // ---- packed in-projection: q from Qn, k / v from the un-normalised x (modules.py:124-130)
  {
    float o[8][4];
    frag_zero(o);
    rs_fgemm_frag(o, Nf, Wt);
    frag_bias_scale(o, p.bin, p.qscale, t);
    frag_store_tile(Qs, o, i0, i1, t);
    frag_zero(o);
    rs_fgemm_frag(o, Xf, Wt + RS_TILE);
    frag_bias_scale(o, p.bin + RS_H, 1.f, t);
    frag_store_tile(Ks, o, i0, i1, t);
    frag_zero(o);
    rs_fgemm_frag(o, Xf, Wt + 2 * RS_TILE);
    frag_bias_scale(o, p.bin + 2 * RS_H, 1.f, t);
    frag_store_tile(Vs, o, i0, i1, t);
  }
  ADT_STAMP(51);
  __syncthreads();
  ADT_STAMP(52);
  // ---- attention, all heads
  float Cf[8][4];
  sq_attn_fwd<HD>(Cf, Qs, Ks, Vs, L, p.mask_mode, p.ids + grow0);
  ADT_STAMP(53);
  // ---- y = ctx Wo^T + bo + Qn ; independence head on the per-head context slices
  float u[8][4];
  frag_zero(u);
  rs_fgemm_frag(u, Cf, Wt + 3 * RS_TILE);
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const float2 bb = __ldg(reinterpret_cast<const float2*>(p.bo + 8 * nb + 2 * t));
    u[nb][0] += bb.x + Nf[nb][0]; u[nb][1] += bb.y + Nf[nb][1]; u[nb][2] += bb.x + Nf[nb][2]; u[nb][3] += bb.y + Nf[nb][3];
  }
  ADT_STAMP(54);
  if (p.rec || p.nll_acc) {
    __syncthreads();                                  // every warp is done with Q as the attention operand
    frag_store_tile(Qs, Cf, i0, i1, t);               // context tile (bf16, as the row-tile kernels see it)
    __syncthreads();
    double nll = 0.0;
    for (int i = threadIdx.x; i < 64 * NH; i += SQ_NT) {
      const int r = i / NH, c = i - r * NH;
      if (r >= L) continue;
      float lg[NH];
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < NH; ++j) {
        float sacc = 0.f;
        for (int dd = 0; dd < HD; ++dd) sacc = fmaf(__bfloat162float(Qs[r * RS_LD + c * HD + dd]), __ldg(p.Wsp + j * HD + dd), sacc);
        lg[j] = sacc + __ldg(p.bsp + j);
        mx = fmaxf(mx, lg[j]);
      }
      float se = 0.f;
#pragma unroll
      for (int j = 0; j < NH; ++j) se += expf(lg[j] - mx);
      const float lz = mx + logf(se);
      if (p.rec) {
#pragma unroll
        for (int j = 0; j < NH; ++j) p.rec[((grow0 + r) * NH + c) * NH + j] = lg[j] - lz;
      }
#pragma unroll
      for (int j = 0; j < NH; ++j) if (j == c) nll -= (double)(lg[j] - lz);
    }
    if (p.nll_acc) warp_accumulate(nll, p.nll_acc);
  }
  ADT_STAMP(55);
  frag_ln(u, p.ln2_g, p.ln2_b, t);                    // z = LN2(y)
  float o[8][4];
  sq_ffn_fwd(o, u, Wt + 4 * RS_TILE, Wt + 5 * RS_TILE, p.c1, p.c2, t);
  ADT_STAMP(56);
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    if (keep0 == 0) { o[nb][0] = 0.f; o[nb][1] = 0.f; }
    if (keep1 == 0) { o[nb][2] = 0.f; o[nb][3] = 0.f; }
  }
  if (p.out) frag_store(p.out + g0, o, i0, i1, v0, v1, t);
  ADT_STAMP(57);
  if (p.out_last) frag_store(p.out_last + (long long)b * RS_H - (long long)(L - 1) * RS_H, o, i0, i1, i0 == L - 1, i1 == L - 1, t);
}

}  // namespace adt
