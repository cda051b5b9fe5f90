// Shared device building blocks for the ADT hot-path kernels (sm_100a).
//
// Every transformer-block kernel in this library is a "row-tile" kernel: one CTA
// (256 threads) owns TM rows of the flattened [B*L, H] activation matrix, keeps
// them in shared memory across a chain of fused ops (LayerNorm -> GEMM -> bias
// -> dropout -> ReLU -> residual -> mask), and streams weight matrices through a
// double-buffered cp.async staging area.  All arithmetic is fp32 (the reference
// is fp32 end to end; SURVEY.md section 8a) with fp32 FFMA register tiles.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace adt {

// phase timestamps of CTA (0,0,0) for latency debugging (read back with adt_debug_read)
__device__ long long g_dbg_clock[64];
#define ADT_STAMP(i) do { if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 0) g_dbg_clock[i] = clock64(); } while (0)

constexpr int NT = 256;        // threads per CTA for all row-tile kernels
constexpr int CH = 64;         // weight chunk edge (rows and cols)
constexpr int CHP = CH + 4;    // padded chunk row stride in floats (272 B: 16B aligned, LDS.128 conflict free)
constexpr int CHPB = CH + 8;   // chunk row stride of K-major chunks in bf16-MMA mode (288 B: LDS.64 fragment loads conflict free)
constexpr int WS_NST = 2;                // depth of the weight-chunk ring
constexpr int WS_SLOT = CH * CHPB;       // floats per ring slot (large enough for both strides)
constexpr int WS_FLOATS = WS_NST * WS_SLOT;  // staging area

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 dropout (must match oracle/philox.py bit for bit)
// ---------------------------------------------------------------------------------------------
struct DropDesc {
  uint32_t enabled;   // 0: identity
  uint32_t thr;       // keep iff rnd >= thr
  uint32_t thr16;     // 16-bit threshold of the attention-probability sites
  float scale;        // 1/(1-p)
  uint32_t seed_lo, seed_hi, step, site;
  unsigned long long base;  // element offset added to every index (batch offset b0 * per-sample elements)
  const uint32_t* step_dev; // optional device-side counter added to step
};
__device__ __forceinline__ uint32_t drop_step(const DropDesc& d) { return d.step_dev ? d.step + *d.step_dev : d.step; }

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

// multipliers (0 or scale) for the 4 consecutive elements idx4*4 .. idx4*4+3
__device__ __forceinline__ float4 drop_mul4(const DropDesc& d, unsigned long long idx4) {
  const uint4 r = philox4x32_10((uint32_t)idx4, (uint32_t)(idx4 >> 32), d.site, drop_step(d), d.seed_lo, d.seed_hi);
  return make_float4(r.x >= d.thr ? d.scale : 0.f, r.y >= d.thr ? d.scale : 0.f, r.z >= d.thr ? d.scale : 0.f,
                     r.w >= d.thr ? d.scale : 0.f);
}
__device__ __forceinline__ float drop_mul1(const DropDesc& d, unsigned long long idx) {
  const uint4 r = philox4x32_10((uint32_t)(idx >> 2), (uint32_t)(idx >> 34), d.site, drop_step(d), d.seed_lo, d.seed_hi);
  const uint32_t lane = (uint32_t)idx & 3u;
  const uint32_t v = lane == 0 ? r.x : lane == 1 ? r.y : lane == 2 ? r.z : r.w;
  return v >= d.thr ? d.scale : 0.f;
}

// attention-probability sites: multipliers for keys 8*c8 .. 8*c8+7 of row r (padded row stride lp8 = ceil8(L)/8 calls):
// 16-bit lane k of philox(ctr = r*lp8 + c8); d.base holds the ROW offset of this rank.
__device__ __forceinline__ void drop_mul8_attn(const DropDesc& d, unsigned long long r, int lp8, int c8, float (&m)[8]) {
  const unsigned long long c = r * (unsigned long long)lp8 + (unsigned long long)c8;
  const uint4 x = philox4x32_10((uint32_t)c, (uint32_t)(c >> 32), d.site, drop_step(d), d.seed_lo, d.seed_hi);
  const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
  for (int k = 0; k < 8; ++k) m[k] = ((w[k >> 1] >> (16 * (k & 1))) & 0xffffu) >= d.thr16 ? d.scale : 0.f;
}

// ---------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool valid) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  const int sz = valid ? 16 : 0;  // src-size 0 => 16 bytes of zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

// CTA-wide sum of one double per thread -> atomicAdd into *dst (thread 0). scratch: >= 8 doubles of smem.
__device__ __forceinline__ void cta_accumulate(double v, double* dst, double* scratch) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) scratch[w] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < NT / 32; ++i) s += scratch[i];
    atomicAdd(dst, s);
  }
}

// ---------------------------------------------------------------------------------------------
// Activation tiles: smem [TM][ld] fp32, ld = C + 4 (C multiple of 4).
// ---------------------------------------------------------------------------------------------
// Load rows row0..row0+TM-1 (rows >= M are zero filled) of a row-major [M, ldg] matrix, columns c0..c0+C-1.
// ASYNCHRONOUS: the rows are fetched with cp.async (all 16-byte pieces of the tile in flight at once instead of one dependent
// round trip per loop iteration); the tile is only valid after tile_sync().
template <int TM>
__device__ __forceinline__ void load_tile(float* __restrict__ T, int ld, const float* __restrict__ G, long long ldg, int c0,
                                          int C, int row0, int M) {
  const int c4n = C >> 2;
  for (int s = threadIdx.x; s < TM * c4n; s += NT) {
    const int r = s / c4n, c4 = s - r * c4n;
    const bool ok = row0 + r < M;
    cp_async16(T + r * ld + 4 * c4, G + (ok ? (long long)(row0 + r) * ldg + c0 + 4 * c4 : 0ll), ok);
  }
}
// completes every outstanding cp.async of this thread (tile loads and weight-ring chunks alike), then the CTA barrier
__device__ __forceinline__ void tile_sync() {
  asm volatile("cp.async.wait_all;\n" ::: "memory");
  __syncthreads();
}
template <int TM>
__device__ __forceinline__ void store_tile(const float* __restrict__ T, int ld, float* __restrict__ G, long long ldg, int c0,
                                           int C, int row0, int M) {
  const int c4n = C >> 2;
  for (int s = threadIdx.x; s < TM * c4n; s += NT) {
    const int r = s / c4n, c4 = s - r * c4n;
    if (row0 + r < M)
      *reinterpret_cast<float4*>(G + (long long)(row0 + r) * ldg + c0 + 4 * c4) = *reinterpret_cast<const float4*>(T + r * ld + 4 * c4);
  }
}

// LayerNorm of every row of a tile, biased variance, eps inside the sqrt (torch.nn.LayerNorm; reference eps=1e-8,
// sasrec/modules.py:638,640,660 and model.py:29).  FOUR lanes per row (64 rows in flight per pass, two shuffle steps
// per reduction) instead of a warp per row: the per-row dependent chain (sum -> mean -> var -> rsqrt) is latency
// bound, so rows must run side by side.  dst may alias src.  Rows with row0+r >= M are written as zeros.
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v;
}
template <int TM>
__device__ __forceinline__ void ln_tile(const float* __restrict__ S, float* __restrict__ D, int ld, int C,
                                        const float* __restrict__ gamma, const float* __restrict__ beta, float eps, int row0, int M,
                                        float* __restrict__ stats = nullptr) {
  const int q = threadIdx.x & 3, n4 = C >> 2;
  for (int r = threadIdx.x >> 2; r < ((TM + 63) & ~63); r += NT / 4) {
    const bool in_tile = r < TM;
    const bool valid = in_tile && (row0 + r < M);
    const float* s = S + (in_tile ? r : 0) * ld;
    float sum = 0.f;
    if (valid)
      for (int g = q; g < n4; g += 4) {
        const float4 v = *reinterpret_cast<const float4*>(s + 4 * g);
        sum += (v.x + v.y) + (v.z + v.w);
      }
    const float mean = quad_sum(sum) / (float)C;
    float var = 0.f;
    if (valid)
      for (int g = q; g < n4; g += 4) {
        const float4 v = *reinterpret_cast<const float4*>(s + 4 * g);
        const float a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
        var += (a * a + b * b) + (c * c + d * d);
      }
    const float rstd = 1.0f / sqrtf(quad_sum(var) / (float)C + eps);
    if (stats && in_tile && q == 0) { stats[2 * r] = valid ? mean : 0.f; stats[2 * r + 1] = valid ? rstd : 0.f; }
    if (!in_tile) continue;
    float* d = D + r * ld;
    for (int g = q; g < n4; g += 4) {
      float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
      if (valid) {
        const float4 v = *reinterpret_cast<const float4*>(s + 4 * g);
        const float4 ga = __ldg(reinterpret_cast<const float4*>(gamma) + g), be = __ldg(reinterpret_cast<const float4*>(beta) + g);
        o = make_float4((v.x - mean) * rstd * ga.x + be.x, (v.y - mean) * rstd * ga.y + be.y, (v.z - mean) * rstd * ga.z + be.z,
                        (v.w - mean) * rstd * ga.w + be.w);
      }
      *reinterpret_cast<float4*>(d + 4 * g) = o;
    }
  }
}

// LayerNorm backward on a tile. X: LN input rows, G: upstream grad rows (dL/d out). Writes dX into DX (may alias G,
// must not alias X) -- if ACCUM, adds to DX instead.  Four lanes per row for the row statistics; dgamma/dbeta are
// column sums over the tile done by (column, row-group) threads and added with atomics.
// red: smem scratch of >= 4*TM floats (mean, rstd per row).
template <int TM, bool ACCUM>
__device__ __forceinline__ void ln_bwd_tile(const float* __restrict__ X, const float* __restrict__ G, float* __restrict__ DX, int ld,
                                            int C, const float* __restrict__ gamma, float eps, int row0, int M,
                                            float* __restrict__ dgamma, float* __restrict__ dbeta, float* __restrict__ red) {
  const int q = threadIdx.x & 3, n4 = C >> 2;
  // column sums first (they need the un-overwritten G when DX aliases G): dgamma[c] = sum_r g*xhat, dbeta[c] = sum_r g
  for (int r = threadIdx.x >> 2; r < ((TM + 63) & ~63); r += NT / 4) {
    const bool in_tile = r < TM;
    const bool valid = in_tile && (row0 + r < M);
    const float* x = X + (in_tile ? r : 0) * ld;
    float sum = 0.f;
    if (valid)
      for (int g = q; g < n4; g += 4) {
        const float4 v = *reinterpret_cast<const float4*>(x + 4 * g);
        sum += (v.x + v.y) + (v.z + v.w);
      }
    const float mean = quad_sum(sum) / (float)C;
    float var = 0.f;
    if (valid)
      for (int g = q; g < n4; g += 4) {
        const float4 v = *reinterpret_cast<const float4*>(x + 4 * g);
        const float a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
        var += (a * a + b * b) + (c * c + d * d);
      }
    const float rstd = 1.0f / sqrtf(quad_sum(var) / (float)C + eps);
    if (in_tile && q == 0) { red[2 * r] = mean; red[2 * r + 1] = valid ? rstd : 0.f; }
  }
  __syncthreads();
  {
    const int groups = NT / C > 0 ? NT / C : 1;
    const int col = threadIdx.x % C, grp = threadIdx.x / C;
    if (grp < groups) {
      for (int c = col; c < C; c += NT) {   // (only iterates once unless C > NT)
        float dg = 0.f, db = 0.f;
        for (int r = grp; r < TM; r += groups) {
          const float rs = red[2 * r + 1];
          if (rs != 0.f) {
            const float g = G[r * ld + c];
            dg = fmaf(g, (X[r * ld + c] - red[2 * r]) * rs, dg);
            db += g;
          }
        }
        atomicAdd(dgamma + c, dg);
        atomicAdd(dbeta + c, db);
      }
    }
  }
  __syncthreads();
  for (int r = threadIdx.x >> 2; r < ((TM + 63) & ~63); r += NT / 4) {
    const bool in_tile = r < TM;
    const float mean = in_tile ? red[2 * r] : 0.f, rstd = in_tile ? red[2 * r + 1] : 0.f;
    const bool valid = in_tile && rstd != 0.f;
    const float* x = X + (in_tile ? r : 0) * ld;
    const float* gr = G + (in_tile ? r : 0) * ld;
    float s1 = 0.f, s2 = 0.f;
    if (valid)
      for (int g = q; g < n4; g += 4) {
        const float4 xv = *reinterpret_cast<const float4*>(x + 4 * g), gv = *reinterpret_cast<const float4*>(gr + 4 * g);
        const float4 ga = __ldg(reinterpret_cast<const float4*>(gamma) + g);
        const float g0 = gv.x * ga.x, g1 = gv.y * ga.y, g2 = gv.z * ga.z, g3 = gv.w * ga.w;
        s1 += (g0 + g1) + (g2 + g3);
        s2 += (g0 * (xv.x - mean) + g1 * (xv.y - mean)) * rstd + (g2 * (xv.z - mean) + g3 * (xv.w - mean)) * rstd;
      }
    s1 = quad_sum(s1) / (float)C;
    s2 = quad_sum(s2) / (float)C;
    if (!in_tile) continue;
    float* dx = DX + r * ld;
    for (int g = q; g < n4; g += 4) {
      float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
      if (valid) {
        const float4 xv = *reinterpret_cast<const float4*>(x + 4 * g), gv = *reinterpret_cast<const float4*>(gr + 4 * g);
        const float4 ga = __ldg(reinterpret_cast<const float4*>(gamma) + g);
        o = make_float4(rstd * (gv.x * ga.x - s1 - (xv.x - mean) * rstd * s2), rstd * (gv.y * ga.y - s1 - (xv.y - mean) * rstd * s2),
                        rstd * (gv.z * ga.z - s1 - (xv.z - mean) * rstd * s2), rstd * (gv.w * ga.w - s1 - (xv.w - mean) * rstd * s2));
      }
      float4* dst = reinterpret_cast<float4*>(dx + 4 * g);
      if (ACCUM) { const float4 old = *dst; o = make_float4(o.x + old.x, o.y + old.y, o.z + old.z, o.w + old.w); }
      *dst = o;
    }
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// Weight staging: one [64][64] chunk of a row-major matrix -> smem [64][CHP] (zero filled outside).
// PERM: store global chunk row n at smem row (n>>2) + 16*(n&3) so that the NT micro-kernel's thread tx
//       reads rows tx+16j (conflict free) while owning the 4 CONTIGUOUS output columns 4tx..4tx+3.
// ---------------------------------------------------------------------------------------------
template <bool PERM, int STRIDE = CHP>
__device__ __forceinline__ void stage_chunk(float* __restrict__ buf, const float* __restrict__ G, long long ldg, int r0, int c0,
                                            int nr, int nc) {
#pragma unroll
  for (int it = 0; it < (CH * CH / 4) / NT; ++it) {
    const int s = threadIdx.x + it * NT;
    const int r = s >> 4, c4 = s & 15;
    const bool ok = (r < nr) && (4 * c4 < nc);
    const int rs = PERM ? ((r >> 2) + 16 * (r & 3)) : r;
    const float* src = ok ? (G + (long long)(r0 + r) * ldg + c0 + 4 * c4) : G;
    cp_async16(buf + rs * STRIDE + 4 * c4, src, ok);
  }
}

// acc[i][j] += sum_k A[ty+16i][k0+k] * W[n0+4tx+j][k]      (chunk staged with PERM=true)
template <int RM>
__device__ __forceinline__ void mma_nt(float (&acc)[RM][4], const float* __restrict__ A, int lda, int k0,
                                       const float* __restrict__ Wc, int klen) {
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const float* a0 = A + ty * lda + k0;
  const float* w0 = Wc + tx * CHP;
#pragma unroll 2
  for (int kk = 0; kk < klen; kk += 4) {
    float4 a[RM], w[4];
#pragma unroll
    for (int i = 0; i < RM; ++i) a[i] = *reinterpret_cast<const float4*>(a0 + 16 * i * lda + kk);
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = *reinterpret_cast<const float4*>(w0 + 16 * j * CHP + kk);
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        acc[i][j] = fmaf(a[i].x, w[j].x, acc[i][j]);
        acc[i][j] = fmaf(a[i].y, w[j].y, acc[i][j]);
        acc[i][j] = fmaf(a[i].z, w[j].z, acc[i][j]);
        acc[i][j] = fmaf(a[i].w, w[j].w, acc[i][j]);
      }
  }
}

// acc[i][c] += sum_n A[ty+16i][n0+n] * W[n][c0+4tx+c]       (chunk staged with PERM=false)
template <int RM>
__device__ __forceinline__ void mma_nn(float (&acc)[RM][4], const float* __restrict__ A, int lda, int n0,
                                       const float* __restrict__ Wc, int nlen) {
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const float* a0 = A + ty * lda + n0;
  const float* w0 = Wc + 4 * tx;
#pragma unroll 2
  for (int nn = 0; nn < nlen; nn += 4) {
    float4 a[RM], w[4];
#pragma unroll
    for (int i = 0; i < RM; ++i) a[i] = *reinterpret_cast<const float4*>(a0 + 16 * i * lda + nn);
#pragma unroll
    for (int u = 0; u < 4; ++u) w[u] = *reinterpret_cast<const float4*>(w0 + (nn + u) * CHP);
#pragma unroll
    for (int i = 0; i < RM; ++i) {
      acc[i][0] = fmaf(a[i].x, w[0].x, acc[i][0]); acc[i][1] = fmaf(a[i].x, w[0].y, acc[i][1]);
      acc[i][2] = fmaf(a[i].x, w[0].z, acc[i][2]); acc[i][3] = fmaf(a[i].x, w[0].w, acc[i][3]);
      acc[i][0] = fmaf(a[i].y, w[1].x, acc[i][0]); acc[i][1] = fmaf(a[i].y, w[1].y, acc[i][1]);
      acc[i][2] = fmaf(a[i].y, w[1].z, acc[i][2]); acc[i][3] = fmaf(a[i].y, w[1].w, acc[i][3]);
      acc[i][0] = fmaf(a[i].z, w[2].x, acc[i][0]); acc[i][1] = fmaf(a[i].z, w[2].y, acc[i][1]);
      acc[i][2] = fmaf(a[i].z, w[2].z, acc[i][2]); acc[i][3] = fmaf(a[i].z, w[2].w, acc[i][3]);
      acc[i][0] = fmaf(a[i].w, w[3].x, acc[i][0]); acc[i][1] = fmaf(a[i].w, w[3].y, acc[i][1]);
      acc[i][2] = fmaf(a[i].w, w[3].z, acc[i][2]); acc[i][3] = fmaf(a[i].w, w[3].w, acc[i][3]);
    }
  }
}

// Row-tile GEMM driver.
//   NN == false:  Y[r][n] = sum_k A[r][k] * W[n][k]     W is [Nout][Kred] row-major (nn.Linear weight), ld = ldw
//   NN == true :  Y[r][c] = sum_n A[r][n] * W[n][c]     W is [Kred][Nout] row-major, ld = ldw
// A is an smem tile [TM][lda] whose reduction extent is Kred (columns beyond Kred are never read because the staged
// chunk is zero there -- but they must be finite, so tiles are allocated with zeroed padding).
// epi(i, row_local, col, float4 v) is called once per thread per (row ty+16i, columns col..col+3); col < Nout guaranteed
// (Nout is a multiple of 4).  Ends with a __syncthreads(): tile writes made by epi are visible on return.
template <int TM, bool NN, class Epi>
__device__ __forceinline__ void gemm_tile(const float* __restrict__ A, int lda, int Kred, const float* __restrict__ W, long long ldw,
                                          int Nout, float* __restrict__ Ws, Epi epi) {
  constexpr int RM = TM / 16;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int noc = (Nout + CH - 1) / CH, nrc = (Kred + CH - 1) / CH;
  const int total = noc * nrc;
  auto stage = [&](int t) {
    const int oc = t / nrc, rc = t - oc * nrc;
    float* buf = Ws + (t & 1) * CH * CHP;
    if (!NN)
      stage_chunk<true>(buf, W, ldw, oc * CH, rc * CH, min(CH, Nout - oc * CH), min(CH, Kred - rc * CH));
    else
      stage_chunk<false>(buf, W, ldw, rc * CH, oc * CH, min(CH, Kred - rc * CH), min(CH, Nout - oc * CH));
    cp_async_commit();
  };
  stage(0);
  float acc[RM][4];
  for (int t = 0; t < total; ++t) {
    const int oc = t / nrc, rc = t - oc * nrc;
    if (rc == 0) {
#pragma unroll
      for (int i = 0; i < RM; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
    }
    if (t + 1 < total) {
      stage(t + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* buf = Ws + (t & 1) * CH * CHP;
    // round the reduction length up to 4 (staged zeros make the tail harmless)
    const int rlen = min(CH, Kred - rc * CH);
    if (!NN) mma_nt<RM>(acc, A, lda, rc * CH, buf, rlen);
    else mma_nn<RM>(acc, A, lda, rc * CH, buf, rlen);
    if (rc == nrc - 1) {
      const int col = oc * CH + 4 * tx;
      if (col < Nout) {
#pragma unroll
        for (int i = 0; i < RM; ++i) epi(i, ty + 16 * i, col, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// Weight stream: all GEMMs of a kernel are declared up-front; their [64x64] chunks flow through an NST-deep cp.async
// ring that keeps prefetching ACROSS GEMM boundaries, so a GEMM phase never starts with an exposed global->smem
// round trip (at H=64 every GEMM is a single chunk: without this each phase would wait for its own load).
// One (possibly empty) cp.async group is committed per issue() so that wait_group<NST-1> is always the right count.
// ---------------------------------------------------------------------------------------------
struct GemmDesc {
  const float* W; long long ldw; int Nout, Kred, nn;   // nn = 0: Y = A W^T (W [Nout][Kred]) ; nn = 1: Y = A W (W [Kred][Nout])
};
constexpr int WS_MAXG = 8;
struct WStreamState {
  GemmDesc g[WS_MAXG];
  int ng;
};

template <int NST, bool MMA = false>
struct WStream {
  WStreamState* st;   // shared memory
  float* bufs;        // NST * WS_SLOT floats
  int next_g, slot_issue, slot_cons, last_slot;
  // iteration state of the GEMM being issued (kept in registers: no divisions, no descriptor reloads per chunk)
  GemmDesc d;
  int oc, rc, noc, nrc;

  __device__ __forceinline__ void load_desc() {
    if (next_g < st->ng) {
      d = st->g[next_g];
      noc = (d.Nout + CH - 1) / CH;
      nrc = (d.Kred + CH - 1) / CH;
    }
    oc = rc = 0;
  }
  __device__ __forceinline__ void issue() {
    if (next_g < st->ng) {
      float* buf = bufs + slot_issue * WS_SLOT;
      if (!d.nn) {
        if (MMA) stage_chunk<false, CHPB>(buf, d.W, d.ldw, oc * CH, rc * CH, min(CH, d.Nout - oc * CH), min(CH, d.Kred - rc * CH));
        else stage_chunk<true, CHP>(buf, d.W, d.ldw, oc * CH, rc * CH, min(CH, d.Nout - oc * CH), min(CH, d.Kred - rc * CH));
      } else {
        stage_chunk<false, CHP>(buf, d.W, d.ldw, rc * CH, oc * CH, min(CH, d.Kred - rc * CH), min(CH, d.Nout - oc * CH));
      }
      if (++rc == nrc) {
        rc = 0;
        if (++oc == noc) { ++next_g; load_desc(); }
      }
    }
    slot_issue = slot_issue + 1 == NST ? 0 : slot_issue + 1;
    cp_async_commit();
  }
  // call once, by all threads, after the descriptors were written to *st and __syncthreads()
  __device__ __forceinline__ void start(WStreamState* s, float* b) {
    st = s; bufs = b; next_g = 0; slot_issue = slot_cons = 0; last_slot = NST - 1;
    load_desc();
#pragma unroll
    for (int i = 0; i < NST - 1; ++i) issue();
  }
  // the most recently consumed ring slot: free to use as scratch until the next gemm_stream call
  __device__ __forceinline__ float* scratch() const { return bufs + last_slot * WS_SLOT; }
};

// warm the L1 with a small read-only vector (biases, LayerNorm affine) so that the first epilogue / LN touch hits
__device__ __forceinline__ void prefetch_vec(const float* p, int n) {
  if (p)
    for (int i = threadIdx.x * 32; i < n; i += NT * 32) asm volatile("prefetch.global.L1 [%0];" ::"l"(p + i));
}

// ---------------------------------------------------------------------------------------------
// bf16 tensor-core GEMM cores (mma.sync.m16n8k16, fp32 accumulate).  Operands stay fp32 in shared memory and are
// rounded to bf16 when the fragments are packed, so the fp32 and bf16 modes share every tile, epilogue and kernel.
// Warp layout over the [TM x 64] output chunk: WR = TM/16 warps along rows, WC = 8/WR along columns; each warp owns
// 16 rows x (64/WC) columns = NB n-blocks of 8.  Fragment lane mapping: g = lane>>2, t = lane&3.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// A fragment of rows [r0, r0+16) x k [kb, kb+16) of a row-major fp32 tile; k >= klim reads as 0
__device__ __forceinline__ void load_a_frag(uint32_t (&a)[4], const float* __restrict__ A, int lda, int r0, int kb, int klim) {
  const int g = (threadIdx.x & 31) >> 2, t = threadIdx.x & 3;
  const float* p0 = A + (r0 + g) * lda + kb + 2 * t;
  const float* p1 = p0 + 8 * lda;
  const bool lo = kb + 2 * t < klim, hi = kb + 2 * t + 8 < klim;
  const float2 z = make_float2(0.f, 0.f);
  const float2 v0 = lo ? *reinterpret_cast<const float2*>(p0) : z;
  const float2 v1 = lo ? *reinterpret_cast<const float2*>(p1) : z;
  const float2 v2 = hi ? *reinterpret_cast<const float2*>(p0 + 8) : z;
  const float2 v3 = hi ? *reinterpret_cast<const float2*>(p1 + 8) : z;
  a[0] = pack_bf16(v0.x, v0.y); a[1] = pack_bf16(v1.x, v1.y); a[2] = pack_bf16(v2.x, v2.y); a[3] = pack_bf16(v3.x, v3.y);
}

template <int TM>
struct MmaShape {
  static constexpr int WR = TM / 16, WC = 8 / WR, NB = 8 / WC;   // NB n-blocks of 8 columns per warp
};

// acc += A[rows][k0..k0+klen) * Wc^T, Wc = chunk [n][k] (stride CHPB, not permuted)
template <int TM>
__device__ __forceinline__ void mma_nt_bf16(float (&acc)[MmaShape<TM>::NB][4], const float* __restrict__ A, int lda, int k0,
                                            const float* __restrict__ Wc, int klen) {
  using S = MmaShape<TM>;
  const int warp = threadIdx.x >> 5, g = (threadIdx.x & 31) >> 2, t = threadIdx.x & 3;
  const int r0 = 16 * (warp % S::WR), c0 = (64 / S::WC) * (warp / S::WR);
  for (int kk = 0; kk < klen; kk += 16) {
    uint32_t a[4];
    load_a_frag(a, A, lda, r0, k0 + kk, k0 + klen);
    const bool lo = kk + 2 * t < klen, hi = kk + 2 * t + 8 < klen;
#pragma unroll
    for (int j = 0; j < S::NB; ++j) {
      const float* wp = Wc + (c0 + 8 * j + g) * CHPB + kk + 2 * t;
      const float2 z = make_float2(0.f, 0.f);
      const float2 w0 = lo ? *reinterpret_cast<const float2*>(wp) : z;
      const float2 w1 = hi ? *reinterpret_cast<const float2*>(wp + 8) : z;
      mma16816(acc[j], a, pack_bf16(w0.x, w0.y), pack_bf16(w1.x, w1.y));
    }
  }
}
// acc += A[rows][n0..n0+nlen) * Wc, Wc = chunk [k][n] (stride CHP)
template <int TM>
__device__ __forceinline__ void mma_nn_bf16(float (&acc)[MmaShape<TM>::NB][4], const float* __restrict__ A, int lda, int n0,
                                            const float* __restrict__ Wc, int nlen) {
  using S = MmaShape<TM>;
  const int warp = threadIdx.x >> 5, g = (threadIdx.x & 31) >> 2, t = threadIdx.x & 3;
  const int r0 = 16 * (warp % S::WR), c0 = (64 / S::WC) * (warp / S::WR);
  for (int kk = 0; kk < nlen; kk += 16) {
    uint32_t a[4];
    load_a_frag(a, A, lda, r0, n0 + kk, n0 + nlen);
    const bool lo = kk + 2 * t < nlen, hi = kk + 2 * t + 8 < nlen;
#pragma unroll
    for (int j = 0; j < S::NB; ++j) {
      const float* wp = Wc + (kk + 2 * t) * CHP + c0 + 8 * j + g;
      const float w00 = lo ? wp[0] : 0.f, w01 = lo ? wp[CHP] : 0.f;
      const float w10 = hi ? wp[8 * CHP] : 0.f, w11 = hi ? wp[9 * CHP] : 0.f;
      mma16816(acc[j], a, pack_bf16(w00, w01), pack_bf16(w10, w11));
    }
  }
}
// After the MMAs a thread holds, per n-block j, (row g: cols 2t,2t+1) and (row g+8: cols 2t,2t+1).  One exchange with the
// lane of the neighbouring t turns that into ONE float4 of 4 contiguous columns: even t keeps row g, odd t row g+8.
// -> row_local (within the CTA tile), column offset (within the 64 chunk) and the float4 for n-block j.
template <int TM>
__device__ __forceinline__ float4 mma_out4(const float (&c)[4], int j, int& row_local, int& col_in_chunk) {
  using S = MmaShape<TM>;
  const int warp = threadIdx.x >> 5, g = (threadIdx.x & 31) >> 2, t = threadIdx.x & 3;
  const bool odd = t & 1;
  // send what the partner needs: even lanes give away their row g+8 pair, odd lanes their row g pair
  const float sx = odd ? c[0] : c[2], sy = odd ? c[1] : c[3];
  const float rx = __shfl_xor_sync(0xffffffffu, sx, 1), ry = __shfl_xor_sync(0xffffffffu, sy, 1);
  row_local = 16 * (warp % S::WR) + (odd ? g + 8 : g);
  col_in_chunk = (64 / S::WC) * (warp / S::WR) + 8 * j + 4 * (t >> 1);
  return odd ? make_float4(rx, ry, c[2], c[3]) : make_float4(c[0], c[1], rx, ry);
}

// GEMM number gi of the stream (must be consumed in declaration order).  Same contract as gemm_tile.
template <int TM, bool NN, int NST, bool MMA, class Epi>
__device__ __forceinline__ void gemm_stream(const float* __restrict__ A, int lda, WStream<NST, MMA>& ws, int gi, Epi epi) {
  constexpr int RM = TM / 16;
  constexpr int NB = MmaShape<TM>::NB;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int Nout = ws.st->g[gi].Nout, Kred = ws.st->g[gi].Kred;
  const int noc = (Nout + CH - 1) / CH, nrc = (Kred + CH - 1) / CH;
  const int total = noc * nrc;
  float acc[MMA ? NB : RM][4];
  int oc = 0, rc = 0;
  for (int t = 0; t < total; ++t) {
    if (rc == 0) {
#pragma unroll
      for (int i = 0; i < (MMA ? NB : RM); ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
    }
    if (gi == 0 && t == 0) ADT_STAMP(16);
    ws.issue();
    if (gi == 0 && t == 0) ADT_STAMP(17);
    cp_async_wait<NST - 1>();
    __syncthreads();
    if (gi == 0 && t == 0) ADT_STAMP(18);
    const float* buf = ws.bufs + ws.slot_cons * WS_SLOT;
    ws.last_slot = ws.slot_cons;
    ws.slot_cons = ws.slot_cons + 1 == NST ? 0 : ws.slot_cons + 1;
    const int rlen = min(CH, Kred - rc * CH);
    if constexpr (MMA) {
      if (!NN) mma_nt_bf16<TM>(reinterpret_cast<float(&)[NB][4]>(acc), A, lda, rc * CH, buf, rlen);
      else mma_nn_bf16<TM>(reinterpret_cast<float(&)[NB][4]>(acc), A, lda, rc * CH, buf, rlen);
    } else {
      if (!NN) mma_nt<RM>(reinterpret_cast<float(&)[RM][4]>(acc), A, lda, rc * CH, buf, rlen);
      else mma_nn<RM>(reinterpret_cast<float(&)[RM][4]>(acc), A, lda, rc * CH, buf, rlen);
    }
    if (gi == 0 && t == 0) ADT_STAMP(19);
    if (rc == nrc - 1) {
      if constexpr (MMA) {
        float4 v[NB];
        int rl = 0, cc[NB];
#pragma unroll
        for (int j = 0; j < NB; ++j) v[j] = mma_out4<TM>(reinterpret_cast<float(&)[NB][4]>(acc)[j], j, rl, cc[j]);
#pragma unroll
        for (int j = 0; j < NB; ++j)
          if (oc * CH + cc[j] < Nout) epi(j, rl, oc * CH + cc[j], v[j]);
      } else {
        const int col = oc * CH + 4 * tx;
        if (col < Nout) {
#pragma unroll
          for (int i = 0; i < RM; ++i) epi(i, ty + 16 * i, col, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
        }
      }
    }
    if (gi == 0 && t == 0) ADT_STAMP(20);
    __syncthreads();
    if (gi == 0 && t == 0) ADT_STAMP(21);
    if (++rc == nrc) { rc = 0; ++oc; }
  }
}

// Weight gradient of a row tile:  dW[n][k] += sum_{r<rows} dY[r][n] * X[r][k]  (vector fp32 atomics into global dW).
// dY: smem tile [.][ldy] (N columns), X: smem tile [.][ldx] (K columns).  dW is [N][K] row-major with ld ldw.
template <bool ATOMIC = true>
__device__ __forceinline__ void wgrad_tile(const float* __restrict__ dY, int ldy, int N, const float* __restrict__ X, int ldx, int K,
                                           int rows, float* __restrict__ dW, long long ldw) {
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  for (int n0 = 0; n0 < N; n0 += CH)
    for (int k0 = 0; k0 < K; k0 += CH) {
      const int n = n0 + 4 * ty, k = k0 + 4 * tx;
      if (n >= N || k >= K) continue;
      float acc[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
      const float* yp = dY + n;
      const float* xp = X + k;
#pragma unroll 4
      for (int r = 0; r < rows; ++r) {
        const float4 y = *reinterpret_cast<const float4*>(yp + r * ldy);
        const float4 x = *reinterpret_cast<const float4*>(xp + r * ldx);
        acc[0][0] = fmaf(y.x, x.x, acc[0][0]); acc[0][1] = fmaf(y.x, x.y, acc[0][1]); acc[0][2] = fmaf(y.x, x.z, acc[0][2]); acc[0][3] = fmaf(y.x, x.w, acc[0][3]);
        acc[1][0] = fmaf(y.y, x.x, acc[1][0]); acc[1][1] = fmaf(y.y, x.y, acc[1][1]); acc[1][2] = fmaf(y.y, x.z, acc[1][2]); acc[1][3] = fmaf(y.y, x.w, acc[1][3]);
        acc[2][0] = fmaf(y.z, x.x, acc[2][0]); acc[2][1] = fmaf(y.z, x.y, acc[2][1]); acc[2][2] = fmaf(y.z, x.z, acc[2][2]); acc[2][3] = fmaf(y.z, x.w, acc[2][3]);
        acc[3][0] = fmaf(y.w, x.x, acc[3][0]); acc[3][1] = fmaf(y.w, x.y, acc[3][1]); acc[3][2] = fmaf(y.w, x.z, acc[3][2]); acc[3][3] = fmaf(y.w, x.w, acc[3][3]);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (n + i < N) {
          float4* dst = reinterpret_cast<float4*>(dW + (long long)(n + i) * ldw + k);
          const float4 val = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
          if (ATOMIC) atomicAdd(dst, val); else *dst = val;
        }
    }
}

// bf16 tensor-core weight gradient: dW[n][k] (+)= sum_{r<rows} dY[r][n] * X[r][k].  M = n, N = k, K = rows of the tile.
// TMR = allocated tile rows (multiple of 16); rows >= `rows` are masked to zero.
template <bool ATOMIC, int TMR>
__device__ __forceinline__ void wgrad_tile_bf16(const float* __restrict__ dY, int ldy, int N, const float* __restrict__ X, int ldx, int K,
                                                int rows, float* __restrict__ dW, long long ldw) {
  const int warp = threadIdx.x >> 5, g = (threadIdx.x & 31) >> 2, t = threadIdx.x & 3;
  const int wn = 16 * (warp & 3), wk = 32 * (warp >> 2);     // warp tile: 16 n x 32 k of the 64x64 output chunk
  for (int n0 = 0; n0 < N; n0 += CH)
    for (int k0 = 0; k0 < K; k0 += CH) {
      if (n0 + wn >= N || k0 + wk >= K) continue;
      float acc[4][4];
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
      const int n = n0 + wn + g;
#pragma unroll 2
      for (int r0 = 0; r0 < TMR && r0 < rows; r0 += 16) {
        const int ra = r0 + 2 * t, rb = ra + 8;
        const bool va = ra < rows, va1 = ra + 1 < rows, vb = rb < rows, vb1 = rb + 1 < rows;
        const bool n_ok = n < N, n8_ok = n + 8 < N;
        uint32_t a[4];
        a[0] = pack_bf16(va && n_ok ? dY[ra * ldy + n] : 0.f, va1 && n_ok ? dY[(ra + 1) * ldy + n] : 0.f);
        a[1] = pack_bf16(va && n8_ok ? dY[ra * ldy + n + 8] : 0.f, va1 && n8_ok ? dY[(ra + 1) * ldy + n + 8] : 0.f);
        a[2] = pack_bf16(vb && n_ok ? dY[rb * ldy + n] : 0.f, vb1 && n_ok ? dY[(rb + 1) * ldy + n] : 0.f);
        a[3] = pack_bf16(vb && n8_ok ? dY[rb * ldy + n + 8] : 0.f, vb1 && n8_ok ? dY[(rb + 1) * ldy + n + 8] : 0.f);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = k0 + wk + 8 * j + g;
          const bool k_ok = k < K;
          const uint32_t b0 = pack_bf16(va && k_ok ? X[ra * ldx + k] : 0.f, va1 && k_ok ? X[(ra + 1) * ldx + k] : 0.f);
          const uint32_t b1 = pack_bf16(vb && k_ok ? X[rb * ldx + k] : 0.f, vb1 && k_ok ? X[(rb + 1) * ldx + k] : 0.f);
          mma16816(acc[j], a, b0, b1);
        }
      }
      // acc[j]: (row n0+wn+g | +8, cols k0+wk+8j+2t,+1) -> float4 per thread after the pair exchange
      const bool odd = t & 1;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float sx = odd ? acc[j][0] : acc[j][2], sy = odd ? acc[j][1] : acc[j][3];
        const float rx = __shfl_xor_sync(0xffffffffu, sx, 1), ry = __shfl_xor_sync(0xffffffffu, sy, 1);
        const int nr = n0 + wn + (odd ? g + 8 : g), kc = k0 + wk + 8 * j + 4 * (t >> 1);
        const float4 val = odd ? make_float4(rx, ry, acc[j][2], acc[j][3]) : make_float4(acc[j][0], acc[j][1], rx, ry);
        if (nr < N && kc < K) {
          float4* dst = reinterpret_cast<float4*>(dW + (long long)nr * ldw + kc);
          if (ATOMIC) atomicAdd(dst, val); else *dst = val;
        }
      }
    }
}

// db[n] += sum_{r<rows} dY[r][n]  (thread per column, 4 independent partial sums; one atomic per column per CTA)
__device__ __forceinline__ void colsum_atomic(const float* __restrict__ dY, int ldy, int N, int rows, float* __restrict__ db) {
  for (int n = threadIdx.x; n < N; n += NT) {
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int r = 0;
    for (; r + 3 < rows; r += 4) {
      s0 += dY[r * ldy + n]; s1 += dY[(r + 1) * ldy + n]; s2 += dY[(r + 2) * ldy + n]; s3 += dY[(r + 3) * ldy + n];
    }
    for (; r < rows; ++r) s0 += dY[r * ldy + n];
    atomicAdd(db + n, (s0 + s1) + (s2 + s3));
  }
}

// Hoisted weight gradients (wide models): instead of reducing dY^T X over its few rows and adding H x H partial sums to the global
// gradient with atomics -- the dominant cost of the backward row-tile kernels at H = 256 -- a CTA only writes the bf16 copies of its
// dY and X tiles; ONE split-K tcgen05 GEMM per weight (adt_gemm_tc, both operands read MN-major) then reduces over all rows.
__device__ __forceinline__ void emit_bf16_tile(const float* __restrict__ T, int ld, int C, int rows, __nv_bfloat16* __restrict__ dst,
                                               long long ldd) {
  const int c4n = C >> 2;
  for (int s = threadIdx.x; s < rows * c4n; s += NT) {
    const int r = s / c4n, c = 4 * (s - r * c4n);
    const float4 v = *reinterpret_cast<const float4*>(T + r * ld + c);
    uint2 o;
    o.x = pack_bf16(v.x, v.y); o.y = pack_bf16(v.z, v.w);
    *reinterpret_cast<uint2*>(dst + (long long)r * ldd + c) = o;
  }
}

// dispatch helper: fp32 FFMA or bf16 tensor-core weight gradient
template <bool MMA, bool ATOMIC, int TMR>
__device__ __forceinline__ void wgrad_any(const float* __restrict__ dY, int ldy, int N, const float* __restrict__ X, int ldx, int K,
                                          int rows, float* __restrict__ dW, long long ldw) {
  if constexpr (MMA) wgrad_tile_bf16<ATOMIC, TMR>(dY, ldy, N, X, ldx, K, rows, dW, ldw);
  else wgrad_tile<ATOMIC>(dY, ldy, N, X, ldx, K, rows, dW, ldw);
}
template <bool MMA>
__host__ __device__ constexpr int tile_pad() { return MMA ? 8 : 4; }

__device__ __forceinline__ float4 f4_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 f4_mul(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float4 f4_scale(float4 a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }

}  // namespace adt
