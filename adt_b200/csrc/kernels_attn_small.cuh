// Short-sequence attention (L <= 64, head dim 16/32/64) for the bf16 tensor-core mode: ONE 128-thread CTA per (sequence, head),
// whole K/V of the head in shared memory as bf16, scores / probabilities / their adjoints never leave registers
// (mma.sync.m16n8k16 accumulator fragments are re-used as the A fragments of the next product).  Footprint: 15 KB (fwd) /
// 52 KB (bwd) of shared memory, so every (sequence, head) of a 256 x 2 batch is resident in ONE wave (the generic row-tile
// attention kernel needs 62-87 KB and 256 threads per problem: 1.7 waves at the C2 shape).
// Same semantics as attn_fwd_kernel / attn_bwd_kernel (sasrec/modules.py:488-516; bert4rec/model/modules.py:88-96):
// q is pre-scaled, mask_mode 0 = causal, 1 = key padding (-1e9), dropout on the probabilities from the attention-site Philox stream.
#pragma once
#include "common.cuh"
#include "kernels_bwd.cuh"

namespace adt {

constexpr int AS_NT = 128;        // threads per CTA
constexpr int AS_LT = 72;         // row stride (halfwords) of the transposed [HD][64] tiles: conflict-free fragment loads

__device__ __forceinline__ uint32_t ld_u32(const __nv_bfloat16* p) { return *reinterpret_cast<const uint32_t*>(p); }

// ldmatrix fragment loaders on row-major bf16 tiles with row stride LDT halfwords (LDT*2 bytes must be a multiple of 16; 40 and 72
// halfwords give conflict-free 8x8 block loads)
template <int LDT>
__device__ __forceinline__ void lm_a(uint32_t (&a)[4], const __nv_bfloat16* A, int m0, int k0) {            // A[m][k]
  const int l = threadIdx.x & 31;
  const unsigned ad = (unsigned)__cvta_generic_to_shared(A + (m0 + (l & 7) + 8 * ((l >> 3) & 1)) * LDT + k0 + 8 * (l >> 4));
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]) : "r"(ad));
}
template <int LDT>
__device__ __forceinline__ void lm_a_t(uint32_t (&a)[4], const __nv_bfloat16* S, int m0, int k0) {          // A[m][k] = S[k][m]
  const int l = threadIdx.x & 31;
  const unsigned ad = (unsigned)__cvta_generic_to_shared(S + (k0 + (l & 7) + 8 * (l >> 4)) * LDT + m0 + 8 * ((l >> 3) & 1));
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]) : "r"(ad));
}
template <int LDT>
__device__ __forceinline__ void lm_b(uint32_t& b0, uint32_t& b1, const __nv_bfloat16* Bn, int n0, int k0) {  // B[k][n] = Bn[n][k]
  const int l = threadIdx.x & 15;
  const unsigned ad = (unsigned)__cvta_generic_to_shared(Bn + (n0 + (l & 7)) * LDT + k0 + 8 * (l >> 3));
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(b0), "=r"(b1) : "r"(ad));
}
template <int LDT>
__device__ __forceinline__ void lm_b_t(uint32_t& b0, uint32_t& b1, const __nv_bfloat16* Bk, int k0, int n0) {  // B[k][n] = Bk[k][n]
  const int l = threadIdx.x & 15;
  const unsigned ad = (unsigned)__cvta_generic_to_shared(Bk + (k0 + (l & 7) + 8 * (l >> 3)) * LDT + n0);
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(b0), "=r"(b1) : "r"(ad));
}

// rows [0, L) x HD columns of N head slices (global row stride H) -> bf16 tiles [64][HD + 8] and/or transposed copies [HD][72].
// All global loads of all N tensors are issued before the first conversion/store: one memory round trip for the whole prologue.
template <int HD, int N>
__device__ __forceinline__ void as_load(const float* const (&src)[N], int H, int L, __nv_bfloat16* const (&dst)[N],
                                        __nv_bfloat16* const (&dstT)[N]) {
  constexpr int LD = HD + 8, C4 = HD / 4, NIT = 64 * C4 / AS_NT;
  float4 v[N][NIT];
#pragma unroll
  for (int n = 0; n < N; ++n) {
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int idx = threadIdx.x + it * AS_NT;
      const int r = idx / C4, c = (idx - r * C4) * 4;
      v[n][it] = r < L ? __ldg(reinterpret_cast<const float4*>(src[n] + (long long)r * H + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
#pragma unroll
  for (int n = 0; n < N; ++n) {
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int idx = threadIdx.x + it * AS_NT;
      const int r = idx / C4, c = (idx - r * C4) * 4;
      const float4 x = v[n][it];
      if (dst[n]) {
        uint32_t* d = reinterpret_cast<uint32_t*>(dst[n] + r * LD + c);
        d[0] = pack_bf16(x.x, x.y);
        d[1] = pack_bf16(x.z, x.w);
      }
      if (dstT[n]) {
        dstT[n][(c + 0) * AS_LT + r] = __float2bfloat16_rn(x.x);
        dstT[n][(c + 1) * AS_LT + r] = __float2bfloat16_rn(x.y);
        dstT[n][(c + 2) * AS_LT + r] = __float2bfloat16_rn(x.z);
        dstT[n][(c + 3) * AS_LT + r] = __float2bfloat16_rn(x.w);
      }
    }
  }
}

// acc[nb] (16 rows of this warp x 8 columns) += A[rows][0..HD) * B[8nb+g][0..HD)^T, A and B row-major bf16 tiles (stride HD+8)
template <int HD>
__device__ __forceinline__ void as_mma_rows(float (&acc)[8][4], const __nv_bfloat16* __restrict__ A, const __nv_bfloat16* __restrict__ B,
                                            int r0, int nbr) {
  constexpr int LD = HD + 8;
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int ks = 0; ks < HD / 16; ++ks) {
    uint32_t a[4];
    a[0] = ld_u32(A + (r0 + g) * LD + 16 * ks + 2 * t);
    a[1] = ld_u32(A + (r0 + g + 8) * LD + 16 * ks + 2 * t);
    a[2] = ld_u32(A + (r0 + g) * LD + 16 * ks + 2 * t + 8);
    a[3] = ld_u32(A + (r0 + g + 8) * LD + 16 * ks + 2 * t + 8);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      if (nb < nbr) {
        const __nv_bfloat16* bp = B + (8 * nb + g) * LD + 16 * ks + 2 * t;
        mma16816(acc[nb], a, ld_u32(bp), ld_u32(bp + 8));
      }
    }
  }
}

// out[db] (16 rows x 8 head columns) += P[16 rows][0..64) * Bt[8db+g][0..64)^T with P given as accumulator fragments p[nb][4]
// (columns 8nb+2t, +1 of rows g / g+8) and Bt a transposed tile [HD][72]
template <int HD>
__device__ __forceinline__ void as_mma_frag(float (&out)[HD / 8][4], const float (&p)[8][4], const __nv_bfloat16* __restrict__ Bt, int nks) {
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    if (ks < nks) {
      uint32_t a[4];
      a[0] = pack_bf16(p[2 * ks][0], p[2 * ks][1]);
      a[1] = pack_bf16(p[2 * ks][2], p[2 * ks][3]);
      a[2] = pack_bf16(p[2 * ks + 1][0], p[2 * ks + 1][1]);
      a[3] = pack_bf16(p[2 * ks + 1][2], p[2 * ks + 1][3]);
#pragma unroll
      for (int db = 0; db < HD / 8; ++db) {
        const __nv_bfloat16* bp = Bt + (8 * db + g) * AS_LT + 16 * ks + 2 * t;
        mma16816(out[db], a, ld_u32(bp), ld_u32(bp + 8));
      }
    }
  }
}

// acc[nb] += A[16 rows r0..][0..HD) * Bn[8nb..][0..HD)^T with ldmatrix fragments (tiles [64][HD+8])
template <int HD, int LD = HD + 8>
__device__ __forceinline__ void as_mma_rows_lm(float (&acc)[8][4], const __nv_bfloat16* __restrict__ A, const __nv_bfloat16* __restrict__ Bn,
                                               int r0, int nbr) {
#pragma unroll
  for (int ks = 0; ks < HD / 16; ++ks) {
    uint32_t a[4];
    lm_a<LD>(a, A, r0, 16 * ks);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      if (nb < nbr) {
        uint32_t b0, b1;
        lm_b<LD>(b0, b1, Bn, 8 * nb, 16 * ks);
        mma16816(acc[nb], a, b0, b1);
      }
    }
  }
}
// out[db] += P (fragments, k = key index j) * Bk[j][8db..]   with Bk a row-major [64][LD] tile (V or K), via transposing loads
template <int HD, int LD = HD + 8>
__device__ __forceinline__ void as_mma_frag_lm(float (&out)[HD / 8][4], const float (&p)[8][4], const __nv_bfloat16* __restrict__ Bk, int nks) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    if (ks < nks) {
      uint32_t a[4];
      a[0] = pack_bf16(p[2 * ks][0], p[2 * ks][1]);
      a[1] = pack_bf16(p[2 * ks][2], p[2 * ks][3]);
      a[2] = pack_bf16(p[2 * ks + 1][0], p[2 * ks + 1][1]);
      a[3] = pack_bf16(p[2 * ks + 1][2], p[2 * ks + 1][3]);
#pragma unroll
      for (int db = 0; db < HD / 8; ++db) {
        uint32_t b0, b1;
        lm_b_t<LD>(b0, b1, Bk, 16 * ks, 8 * db);
        mma16816(out[db], a, b0, b1);
      }
    }
  }
}

// masked scores -> (unnormalised) exponentials relative to `ref` (row max in fwd, log-sum-exp in bwd); returns nothing, updates s
__device__ __forceinline__ float as_masked(float s, int i, int j, int L, int mask_mode, const int* __restrict__ kid) {
  if (i >= L || j >= L || (mask_mode == 0 && j > i)) return -INFINITY;
  if (mask_mode == 1 && kid[j] == 0) return -1e9f;
  return s;
}

// Dropout multipliers of this thread's 2 x 2 elements of every 8-key block nb: block nb of row r draws ONE Philox call
// (ctr = r*lp8 + nb) whose 32-bit word t holds the 16-bit lanes of columns 8nb+2t, 8nb+2t+1.  The four threads of a quad need the
// four words of the same call, so quad thread t' evaluates the calls of blocks nb = t' (mod 4) for both rows and the words travel
// by shuffle: 4 calls per thread instead of 16.
struct AsDrop { float2 m0[8], m1[8]; };
__device__ __forceinline__ void as_drop_all(AsDrop& o, const DropDesc& d, unsigned long long r0, unsigned long long r1, bool v0, bool v1,
                                            int lp8, int nbr, int t) {
  uint4 x0[2], x1[2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int nb = t + 4 * u;
    x0[u] = x1[u] = make_uint4(0u, 0u, 0u, 0u);
    if (nb < nbr) {
      const unsigned long long c0 = r0 * (unsigned long long)lp8 + (unsigned long long)nb, c1 = r1 * (unsigned long long)lp8 + (unsigned long long)nb;
      if (v0) x0[u] = philox4x32_10((uint32_t)c0, (uint32_t)(c0 >> 32), d.site, drop_step(d), d.seed_lo, d.seed_hi);
      if (v1) x1[u] = philox4x32_10((uint32_t)c1, (uint32_t)(c1 >> 32), d.site, drop_step(d), d.seed_lo, d.seed_hi);
    }
  }
  const int qbase = (threadIdx.x & 31) & ~3;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int src = qbase | (nb & 3), u = nb >> 2;
    const uint4 a = x0[u], b = x1[u];
    // every thread fetches word t of the owner's call: the owner publishes all four words, the reader picks its own
    const uint32_t ax = __shfl_sync(0xffffffffu, a.x, src), ay = __shfl_sync(0xffffffffu, a.y, src), az = __shfl_sync(0xffffffffu, a.z, src),
                   aw = __shfl_sync(0xffffffffu, a.w, src);
    const uint32_t bx = __shfl_sync(0xffffffffu, b.x, src), by = __shfl_sync(0xffffffffu, b.y, src), bz = __shfl_sync(0xffffffffu, b.z, src),
                   bw = __shfl_sync(0xffffffffu, b.w, src);
    const uint32_t w0 = t == 0 ? ax : t == 1 ? ay : t == 2 ? az : aw;
    const uint32_t w1 = t == 0 ? bx : t == 1 ? by : t == 2 ? bz : bw;
    o.m0[nb] = make_float2((w0 & 0xffffu) >= d.thr16 ? d.scale : 0.f, (w0 >> 16) >= d.thr16 ? d.scale : 0.f);
    o.m1[nb] = make_float2((w1 & 0xffffu) >= d.thr16 ? d.scale : 0.f, (w1 >> 16) >= d.thr16 ? d.scale : 0.f);
  }
}

// Forward of one head for the 16 query rows 16w .. 16w+15 of the sequence (w = 0..3: the warp's index in its group of four).  Qs, Ks,
// Vs: bf16 tiles of all 64 rows with row stride LD halfwords, offset to the head's first column; rows >= L hold zeros.  ctx points at
// the head's first column of the sequence's first row (row stride H), lse (nullable) at the (sequence, head) slice of [B][nh][L], and
// rb = drop.base + (b nh + h) L is the Philox row counter of query row 0.
template <int HD, int LD>
__device__ __forceinline__ void as_fwd_head(const __nv_bfloat16* Qs, const __nv_bfloat16* Ks, const __nv_bfloat16* Vs, int w, int L, int H,
                                            int mask_mode, const int* __restrict__ kid, float* __restrict__ ctx, float* __restrict__ lse,
                                            const DropDesc& drop, unsigned long long rb) {
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * w + g, i1 = i0 + 8;
  const int nbr = (L + 7) >> 3, nks = (L + 15) >> 4;
  float s[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) s[nb][0] = s[nb][1] = s[nb][2] = s[nb][3] = 0.f;
  as_mma_rows_lm<HD, LD>(s, Qs, Ks, 16 * w, nbr);
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
  const bool v0 = i0 < L, v1 = i1 < L;
  const float inv0 = v0 ? 1.0f / sum0 : 0.f, inv1 = v1 ? 1.0f / sum1 : 0.f;
  if (lse && t == 0) {
    if (v0) lse[i0] = mx0 + logf(sum0);
    if (v1) lse[i1] = mx1 + logf(sum1);
  }
  const int lp8 = ((L + 7) & ~7) >> 3;
  if (drop.enabled) {
    AsDrop dm;
    as_drop_all(dm, drop, rb + i0, rb + i1, v0, v1, lp8, nbr, t);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      s[nb][0] *= dm.m0[nb].x * inv0; s[nb][1] *= dm.m0[nb].y * inv0;
      s[nb][2] *= dm.m1[nb].x * inv1; s[nb][3] *= dm.m1[nb].y * inv1;
    }
  } else {
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      s[nb][0] *= inv0; s[nb][1] *= inv0; s[nb][2] *= inv1; s[nb][3] *= inv1;
    }
  }
  float o[HD / 8][4];
#pragma unroll
  for (int db = 0; db < HD / 8; ++db) o[db][0] = o[db][1] = o[db][2] = o[db][3] = 0.f;
  as_mma_frag_lm<HD, LD>(o, s, Vs, nks);
#pragma unroll
  for (int db = 0; db < HD / 8; ++db) {
    if (v0) *reinterpret_cast<float2*>(ctx + (long long)i0 * H + 8 * db + 2 * t) = make_float2(o[db][0], o[db][1]);
    if (v1) *reinterpret_cast<float2*>(ctx + (long long)i1 * H + 8 * db + 2 * t) = make_float2(o[db][2], o[db][3]);
  }
}

template <int HD>
__global__ void __launch_bounds__(AS_NT) attn_small_fwd_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                               const float* __restrict__ v, float* __restrict__ ctx,
                                                               float* __restrict__ lse, const int* __restrict__ key_ids, int L, int H,
                                                               int nh, int mask_mode, DropDesc drop) {
  constexpr int LD = HD + 8;
  __shared__ __align__(16) __nv_bfloat16 Qs[64 * LD], Ks[64 * LD], Vs[64 * LD];
  const int bh = blockIdx.x, b = bh / nh, h = bh - b * nh;
  const long long seq_off = (long long)b * L * H + (long long)h * HD;
  {   // rows >= L are written as zeros by the loader (every row of the 64-row tiles is covered)
    const float* const src[3] = {q + seq_off, k + seq_off, v + seq_off};
    __nv_bfloat16* const dst[3] = {Qs, Ks, Vs};
    __nv_bfloat16* const dstT[3] = {nullptr, nullptr, nullptr};
    as_load<HD, 3>(src, H, L, dst, dstT);
  }
  __syncthreads();
  as_fwd_head<HD, LD>(Qs, Ks, Vs, threadIdx.x >> 5, L, H, mask_mode, key_ids + (long long)b * L, ctx + seq_off,
                      lse ? lse + ((long long)b * nh + h) * L : nullptr, drop, drop.base + ((unsigned long long)b * nh + h) * L);
}

// shared memory of the backward kernel (halfwords)
template <int HD>
struct AsBwdSmem {
  static constexpr int LD = HD + 8;
  static constexpr int ROW = 64 * LD, SQ = 64 * AS_LT;
  static constexpr int TOTAL = 4 * ROW + 2 * SQ;              // Q, K, V, dC [64][HD+8] | dS, P~ [64][72]   (all row-major)
};

// Backward of one head for the warp's 16 rows 16w .. 16w+15 (w = 0..3 within its group of four warps): query rows for dq, key rows
// for dk and dv.  Qs, Ks, Vs, dCs: bf16 tiles with row stride LD, offset to the head's columns, zero in rows >= L; dSt, Pt: the group's
// [64][72] scratch tiles.  ls0 / ls1: lse of query rows i0 / i1.  store(which, o) receives dq (0), dk (1), dv (2) of the warp's rows on
// accumulator fragments; sync() is a barrier over the group's warps, between the query-side and the key-side products (the key-side
// products read dS and P~ rows of every warp; after it Ks and Vs are no longer read).
template <int HD, int LD, class Store, class Sync>
__device__ __forceinline__ void as_bwd_head(const __nv_bfloat16* Qs, const __nv_bfloat16* Ks, const __nv_bfloat16* Vs, const __nv_bfloat16* dCs,
                                            __nv_bfloat16* dSt, __nv_bfloat16* Pt, int w, int L, int mask_mode, const int* __restrict__ kid,
                                            float ls0, float ls1, const DropDesc& drop, unsigned long long rb, Store&& store, Sync&& sync) {
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * w + g, i1 = i0 + 8;
  const bool v0 = i0 < L, v1 = i1 < L;
  const int nbr = (L + 7) >> 3, nks = (L + 15) >> 4;
  float p[8][4], dp[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    p[nb][0] = p[nb][1] = p[nb][2] = p[nb][3] = 0.f;
    dp[nb][0] = dp[nb][1] = dp[nb][2] = dp[nb][3] = 0.f;
  }
  as_mma_rows_lm<HD, LD>(p, Qs, Ks, 16 * w, nbr);       // S = q k^T
  as_mma_rows_lm<HD, LD>(dp, dCs, Vs, 16 * w, nbr);     // dP~ = dctx v^T
  const int lp8 = ((L + 7) & ~7) >> 3;
  float dl0 = 0.f, dl1 = 0.f;
  float pt[8][4];                                // P~ = dropout(P)
  AsDrop dm;
  if (drop.enabled) {
    as_drop_all(dm, drop, rb + i0, rb + i1, v0, v1, lp8, nbr, t);
  } else {
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) dm.m0[nb] = dm.m1[nb] = make_float2(1.f, 1.f);
  }
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const float2 m0 = dm.m0[nb], m1 = dm.m1[nb];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int j = 8 * nb + 2 * t + e;
      const float s0 = as_masked(p[nb][e], i0, j, L, mask_mode, kid), s1 = as_masked(p[nb][2 + e], i1, j, L, mask_mode, kid);
      const float p0 = s0 == -INFINITY ? 0.f : expf(s0 - ls0), p1 = s1 == -INFINITY ? 0.f : expf(s1 - ls1);
      const float mm0 = e ? m0.y : m0.x, mm1 = e ? m1.y : m1.x;
      const float d0 = dp[nb][e] * mm0, d1 = dp[nb][2 + e] * mm1;       // dP = dP~ * mask
      dl0 = fmaf(d0, p0, dl0); dl1 = fmaf(d1, p1, dl1);
      p[nb][e] = p0; p[nb][2 + e] = p1;
      dp[nb][e] = d0; dp[nb][2 + e] = d1;
      pt[nb][e] = p0 * mm0; pt[nb][2 + e] = p1 * mm1;
    }
  }
  dl0 += __shfl_xor_sync(0xffffffffu, dl0, 1); dl0 += __shfl_xor_sync(0xffffffffu, dl0, 2);
  dl1 += __shfl_xor_sync(0xffffffffu, dl1, 1); dl1 += __shfl_xor_sync(0xffffffffu, dl1, 2);
  // dS = P (dP - delta) ; transposed bf16 copies of dS and P~ for the key-side products
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const float ds0 = p[nb][e] * (dp[nb][e] - dl0), ds1 = p[nb][2 + e] * (dp[nb][2 + e] - dl1);
      dp[nb][e] = ds0; dp[nb][2 + e] = ds1;
    }
    if (nb < nbr) {
      const int j = 8 * nb + 2 * t;
      *reinterpret_cast<uint32_t*>(dSt + i0 * AS_LT + j) = pack_bf16(dp[nb][0], dp[nb][1]);
      *reinterpret_cast<uint32_t*>(dSt + i1 * AS_LT + j) = pack_bf16(dp[nb][2], dp[nb][3]);
      *reinterpret_cast<uint32_t*>(Pt + i0 * AS_LT + j) = pack_bf16(pt[nb][0], pt[nb][1]);
      *reinterpret_cast<uint32_t*>(Pt + i1 * AS_LT + j) = pack_bf16(pt[nb][2], pt[nb][3]);
    }
  }
  // dq = dS k
  {
    float o[HD / 8][4];
#pragma unroll
    for (int db = 0; db < HD / 8; ++db) o[db][0] = o[db][1] = o[db][2] = o[db][3] = 0.f;
    as_mma_frag_lm<HD, LD>(o, dp, Ks, nks);
    store(0, o);
  }
  sync();
  // dk = dS^T q ; dv = P~^T dctx   (this warp owns key rows 16w .. 16w+15)
#pragma unroll
  for (int which = 0; which < 2; ++which) {
    const __nv_bfloat16* A = which == 0 ? dSt : Pt;       // [i][j]: used transposed, A[m = j][k = i]
    const __nv_bfloat16* Bk = which == 0 ? Qs : dCs;      // [i][d]: B[k = i][n = d]
    float o[HD / 8][4];
#pragma unroll
    for (int db = 0; db < HD / 8; ++db) o[db][0] = o[db][1] = o[db][2] = o[db][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      if (ks < nks) {
        uint32_t a[4];
        lm_a_t<AS_LT>(a, A, 16 * w, 16 * ks);
#pragma unroll
        for (int db = 0; db < HD / 8; ++db) {
          uint32_t b0, b1;
          lm_b_t<LD>(b0, b1, Bk, 16 * ks, 8 * db);
          mma16816(o[db], a, b0, b1);
        }
      }
    }
    store(1 + which, o);
  }
}

template <int HD>
__global__ void __launch_bounds__(AS_NT) attn_small_bwd_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                               const float* __restrict__ v, const float* __restrict__ dctx,
                                                               const float* __restrict__ lse, const int* __restrict__ key_ids,
                                                               float* __restrict__ dq, float* __restrict__ dk, float* __restrict__ dv,
                                                               int L, int H, int nh, int mask_mode, DropDesc drop) {
  using SM = AsBwdSmem<HD>;
  constexpr int LD = SM::LD;
  extern __shared__ __align__(16) uint8_t as_raw[];
  __nv_bfloat16* Qs = reinterpret_cast<__nv_bfloat16*>(as_raw);
  __nv_bfloat16* Ks = Qs + SM::ROW;
  __nv_bfloat16* Vs = Ks + SM::ROW;
  __nv_bfloat16* dCs = Vs + SM::ROW;
  __nv_bfloat16* dSt = dCs + SM::ROW;        // dS[i][j], row-major
  __nv_bfloat16* Pt = dSt + SM::SQ;          // P~[i][j], row-major
  const int bh = blockIdx.x, b = bh / nh, h = bh - b * nh;
  const long long seq_off = (long long)b * L * H + (long long)h * HD;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * w + g, i1 = i0 + 8;
  const bool v0 = i0 < L, v1 = i1 < L;
  const float ls0 = v0 ? lse[((long long)b * nh + h) * L + i0] : 0.f;     // issued early: consumed after the first product
  const float ls1 = v1 ? lse[((long long)b * nh + h) * L + i1] : 0.f;
  {
    const float* const src[4] = {q + seq_off, k + seq_off, v + seq_off, dctx + seq_off};
    __nv_bfloat16* const dst[4] = {Qs, Ks, Vs, dCs};
    __nv_bfloat16* const dstT[4] = {nullptr, nullptr, nullptr, nullptr};
    as_load<HD, 4>(src, H, L, dst, dstT);
  }
  __syncthreads();
  // plain stores: the CTA owns the whole head
  as_bwd_head<HD, LD>(Qs, Ks, Vs, dCs, dSt, Pt, w, L, mask_mode, key_ids + (long long)b * L, ls0, ls1, drop,
                      drop.base + ((unsigned long long)b * nh + h) * L,
                      [&](int which, const float (&o)[HD / 8][4]) {
                        float* out = which == 0 ? dq : which == 1 ? dk : dv;
#pragma unroll
                        for (int db = 0; db < HD / 8; ++db) {
                          if (v0) *reinterpret_cast<float2*>(out + seq_off + (long long)i0 * H + 8 * db + 2 * t) = make_float2(o[db][0], o[db][1]);
                          if (v1) *reinterpret_cast<float2*>(out + seq_off + (long long)i1 * H + 8 * db + 2 * t) = make_float2(o[db][2], o[db][3]);
                        }
                      },
                      [] { __syncthreads(); });
}

}  // namespace adt
