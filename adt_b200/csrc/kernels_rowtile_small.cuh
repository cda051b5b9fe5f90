// Narrow-model (H == 64) row-tile kernels for the bf16 tensor-core mode, built like kernels_attn_small.cuh: 128-thread CTAs,
// every weight matrix of the kernel resident in shared memory as bf16 (no chunk ring, no per-chunk barriers), operands of all
// products staged once as bf16 tiles (row-major and transposed), accumulators and LayerNorm adjoints kept in MMA fragments.
// One kernel per generic row-tile kernel of kernels_fwd.cuh / kernels_bwd.cuh: pre_fwd, mid_fwd, post_fwd<enc|dec>, pre_bwd,
// mid_bwd, post_bwd<enc|dec> (sasrec/modules.py:644-677 and their adjoints).
#pragma once
#include "common.cuh"
#include "kernels_bwd.cuh"
#include "kernels_attn_small.cuh"

namespace adt {

constexpr int RS_H = 64;                 // model width handled by these kernels
constexpr int RS_LD = RS_H + 8;          // halfword stride of every bf16 tile (row-major and transposed): conflict-free fragments
constexpr int RS_TILE = 64 * RS_LD;      // halfwords per [64][72] tile
constexpr int RS_LF = RS_H + 4;          // float stride of the fp32 input tile (consecutive rows land on different banks)

// The backward kernels (pre_bwd, mid_bwd, post_bwd) run 256-thread CTAs in two roles.  Warps 0-3 (chain warps) run the dgrad chain
// on their 16-row strips.  Warps 4-7 (wgrad warps) compute every weight gradient; warp 4+w takes the output rows chain warp w took in
// the 128-thread version.  Nothing downstream reads a weight gradient, so the chain warps hand each operand tile over through a named
// barrier (bar.arrive) and never wait for the MMAs and atomics of the weight gradients.  Two CTAs stay resident per SM.
constexpr int RS_BWD_NT = 256;
constexpr int RS_CHAIN_NT = 128;         // threads of the chain role
__device__ __forceinline__ void rs_bar_arrive(int id) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(RS_BWD_NT) : "memory"); }
__device__ __forceinline__ void rs_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// 64 rows x 64 columns of a row-major fp32 matrix (row stride ld; rows >= nrows read as zero), scaled, into any of: a row-major
// bf16 tile, a transposed bf16 tile, an fp32 tile [64][64].  N tensors at once: every global load is issued before the first store.
// Threads T0 .. T0 + NT - 1 of the CTA take part.
template <int N, int NT = AS_NT, int T0 = 0>
__device__ __forceinline__ void rs_load(const float* const (&src)[N], const long long (&ld)[N], const int (&nrows)[N], const float (&scale)[N],
                                        __nv_bfloat16* const (&dst)[N], __nv_bfloat16* const (&dstT)[N], float* const (&dstF)[N]) {
  constexpr int NIT = 64 * 16 / NT;      // float4 per thread per tensor
  float4 v[N][NIT];
#pragma unroll
  for (int n = 0; n < N; ++n) {
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int idx = threadIdx.x - T0 + it * NT;
      const int r = idx >> 4, c = (idx & 15) * 4;
      v[n][it] = r < nrows[n] ? __ldg(reinterpret_cast<const float4*>(src[n] + (long long)r * ld[n] + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
#pragma unroll
  for (int n = 0; n < N; ++n) {
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
      const int idx = threadIdx.x - T0 + it * NT;
      const int r = idx >> 4, c = (idx & 15) * 4;
      const float4 x = make_float4(v[n][it].x * scale[n], v[n][it].y * scale[n], v[n][it].z * scale[n], v[n][it].w * scale[n]);
      if (dstF[n]) *reinterpret_cast<float4*>(dstF[n] + r * RS_LF + c) = x;
      if (dst[n]) {
        uint32_t* d = reinterpret_cast<uint32_t*>(dst[n] + r * RS_LD + c);
        d[0] = pack_bf16(x.x, x.y);
        d[1] = pack_bf16(x.z, x.w);
      }
      if (dstT[n]) {
        dstT[n][(c + 0) * RS_LD + r] = __float2bfloat16_rn(x.x);
        dstT[n][(c + 1) * RS_LD + r] = __float2bfloat16_rn(x.y);
        dstT[n][(c + 2) * RS_LD + r] = __float2bfloat16_rn(x.z);
        dstT[n][(c + 3) * RS_LD + r] = __float2bfloat16_rn(x.w);
      }
    }
  }
}

// ---- ldmatrix fragment loaders on row-major [64][72] bf16 tiles (144-byte rows: every 8x8 block load is bank-conflict free) ----
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const __nv_bfloat16* p) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], const __nv_bfloat16* p) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x2_t(uint32_t& b0, uint32_t& b1, const __nv_bfloat16* p) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(b0), "=r"(b1) : "r"(a));
}
// A fragment (rows m0..m0+15, k0..k0+15) of a row-major tile A[m][k]
__device__ __forceinline__ void frag_a(uint32_t (&a)[4], const __nv_bfloat16* A, int m0, int k0) {
  const int l = threadIdx.x & 31;
  ldsm_x4(a, A + (m0 + (l & 7) + 8 * ((l >> 3) & 1)) * RS_LD + k0 + 8 * (l >> 4));
}
// A fragment of the TRANSPOSE of a row-major tile S[k][m]: A[m][k] = S[k][m]
__device__ __forceinline__ void frag_a_t(uint32_t (&a)[4], const __nv_bfloat16* S, int m0, int k0) {
  const int l = threadIdx.x & 31;
  ldsm_x4_t(a, S + (k0 + (l & 7) + 8 * (l >> 4)) * RS_LD + m0 + 8 * ((l >> 3) & 1));
}
// B fragment (k0..k0+15, n0..n0+7) of a row-major tile Bk[k][n]
__device__ __forceinline__ void frag_b_t(uint32_t& b0, uint32_t& b1, const __nv_bfloat16* Bk, int k0, int n0) {
  const int l = threadIdx.x & 15;
  ldsm_x2_t(b0, b1, Bk + (k0 + (l & 7) + 8 * (l >> 3)) * RS_LD + n0);
}

// B fragment (k0..k0+15, n0..n0+7) of an n-major tile Bn[n][k] (nn.Linear weights W[out][in] as the B operand of x W^T)
__device__ __forceinline__ void frag_b(uint32_t& b0, uint32_t& b1, const __nv_bfloat16* Bn, int n0, int k0) {
  const int l = threadIdx.x & 15;
  const unsigned a = (unsigned)__cvta_generic_to_shared(Bn + (n0 + (l & 7)) * RS_LD + k0 + 8 * (l >> 3));
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(b0), "=r"(b1) : "r"(a));
}
// Y[nb] (rows 16w.. ; columns 8nb..) += A[rows][k] * W[n][k]^T   (forward of nn.Linear, both tiles row-major)
__device__ __forceinline__ void rs_fgemm(float (&acc)[8][4], const __nv_bfloat16* __restrict__ A, const __nv_bfloat16* __restrict__ W, int r0) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t a[4];
    frag_a(a, A, r0, 16 * ks);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      uint32_t b0, b1;
      frag_b(b0, b1, W, 8 * nb, 16 * ks);
      mma16816(acc[nb], a, b0, b1);
    }
  }
}

// D[nb] (rows 16w.. ; columns 8nb..) += T[rows][j] * W[j][c]   (T and W row-major; W used through transposing loads)
__device__ __forceinline__ void rs_dgrad(float (&acc)[8][4], const __nv_bfloat16* __restrict__ T, const __nv_bfloat16* __restrict__ W, int r0) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t a[4];
    frag_a(a, T, r0, 16 * ks);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      uint32_t b0, b1;
      frag_b_t(b0, b1, W, 16 * ks, 8 * nb);
      mma16816(acc[nb], a, b0, b1);
    }
  }
}

// weight gradient of one projection from ROW-MAJOR tiles: gW[j][c] += sum_r T[r][j] X[r][c], gb[j] += sum_r T[r][j]; warp w (0..3)
// takes the output rows j = 16w..16w+15
__device__ __forceinline__ void rs_wgrad_rm(const __nv_bfloat16* __restrict__ T, const __nv_bfloat16* __restrict__ X, float* __restrict__ gW,
                                            float* __restrict__ gb, int w) {
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  float acc[8][4], ones[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) acc[nb][0] = acc[nb][1] = acc[nb][2] = acc[nb][3] = 0.f;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t a[4];
    frag_a_t(a, T, 16 * w, 16 * ks);                 // A[m = j][k = r] = T[r][j]
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      uint32_t b0, b1;
      frag_b_t(b0, b1, X, 16 * ks, 8 * nb);          // B[k = r][n = c] = X[r][c]
      mma16816(acc[nb], a, b0, b1);
    }
    mma16816(ones, a, 0x3f803f80u, 0x3f803f80u);     // B = all ones (bf16 1.0): every column of `ones` is a row sum
  }
  const int j0 = 16 * w + g, j1 = j0 + 8;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const float x0 = __shfl_xor_sync(0xffffffffu, acc[nb][0], 1), x1 = __shfl_xor_sync(0xffffffffu, acc[nb][1], 1);
    const float y0 = __shfl_xor_sync(0xffffffffu, acc[nb][2], 1), y1 = __shfl_xor_sync(0xffffffffu, acc[nb][3], 1);
    if ((t & 1) == 0) {
      atomicAdd(reinterpret_cast<float4*>(gW + (long long)j0 * RS_H + 8 * nb + 2 * t), make_float4(acc[nb][0], acc[nb][1], x0, x1));
      atomicAdd(reinterpret_cast<float4*>(gW + (long long)j1 * RS_H + 8 * nb + 2 * t), make_float4(acc[nb][2], acc[nb][3], y0, y1));
    }
  }
  if (t == 0) {
    atomicAdd(gb + j0, ones[0]);
    atomicAdd(gb + j1, ones[2]);
  }
}
__device__ __forceinline__ void rs_wgrad_rm(const __nv_bfloat16* __restrict__ T, const __nv_bfloat16* __restrict__ X, float* __restrict__ gW,
                                            float* __restrict__ gb) {
  rs_wgrad_rm(T, X, gW, gb, threadIdx.x >> 5);
}

template <int NT = AS_NT, int T0 = 0>
__device__ __forceinline__ void rs_load1(const float* src, int rows, float scale, __nv_bfloat16* dst) {
  const float* const s[1] = {src};
  const long long ld[1] = {RS_H};
  const int nr[1] = {rows};
  const float sc[1] = {scale};
  __nv_bfloat16* const d[1] = {dst};
  __nv_bfloat16* const dT[1] = {nullptr};
  float* const dF[1] = {nullptr};
  rs_load<1, NT, T0>(s, ld, nr, sc, d, dT, dF);
}

// -------------------------------------------------------------------------------------------------
// pre_fwd_small_kernel == pre_fwd_kernel (kernels_fwd.cuh): LayerNorm + packed in-projection, H == 64, bf16 mode.
// -------------------------------------------------------------------------------------------------
struct PreFwdSmallSmem {
  static constexpr int W = 0, X = 3 * RS_TILE, N = X + RS_TILE, HALF_END = N + RS_TILE;
  static constexpr size_t XF_BYTES = (size_t)HALF_END * 2;
  static constexpr size_t TOTAL_BYTES = XF_BYTES + (size_t)64 * RS_LF * 4;
};

// LayerNorm of the fp32 tile Xf (rows >= rows: zero in Nb) into the bf16 tile Nb and, when norm_out is given, to global rows row0 ..;
// two threads per row (threads 0 .. 127), two-pass statistics
__device__ __forceinline__ void rs_ln_tile(const float* __restrict__ Xf, const float* __restrict__ ln_g, const float* __restrict__ ln_b,
                                           __nv_bfloat16* __restrict__ Nb, float* __restrict__ norm_out, long long row0, int rows) {
  const int r = threadIdx.x >> 1, half = threadIdx.x & 1;
  const float* xr = Xf + r * RS_LF + 32 * half;
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < 32; c += 4) {
    const float4 u = *reinterpret_cast<const float4*>(xr + c);
    s += (u.x + u.y) + (u.z + u.w);
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  const float mean = s * (1.0f / RS_H);
  float qq = 0.f;
#pragma unroll
  for (int c = 0; c < 32; c += 4) {
    const float4 u = *reinterpret_cast<const float4*>(xr + c);
    const float a = u.x - mean, b = u.y - mean, cc = u.z - mean, d = u.w - mean;
    qq += (a * a + b * b) + (cc * cc + d * d);
  }
  qq += __shfl_xor_sync(0xffffffffu, qq, 1);
  const float rstd = 1.0f / sqrtf(qq * (1.0f / RS_H) + 1e-8f);
  const bool ok = r < rows;
#pragma unroll
  for (int c = 0; c < 32; c += 4) {
    const int col = 32 * half + c;
    const float4 u = *reinterpret_cast<const float4*>(xr + c);
    const float4 ga = __ldg(reinterpret_cast<const float4*>(ln_g + col)), be = __ldg(reinterpret_cast<const float4*>(ln_b + col));
    const float4 n = make_float4((u.x - mean) * rstd * ga.x + be.x, (u.y - mean) * rstd * ga.y + be.y, (u.z - mean) * rstd * ga.z + be.z,
                                 (u.w - mean) * rstd * ga.w + be.w);
    uint32_t* d = reinterpret_cast<uint32_t*>(Nb + r * RS_LD + col);
    d[0] = ok ? pack_bf16(n.x, n.y) : 0u;
    d[1] = ok ? pack_bf16(n.z, n.w) : 0u;
    if (norm_out && ok) *reinterpret_cast<float4*>(norm_out + (long long)(row0 + r) * RS_H + col) = n;
  }
}

__global__ void __launch_bounds__(AS_NT) pre_fwd_small_kernel(const float* __restrict__ x, const float* __restrict__ ln_g,
                                                              const float* __restrict__ ln_b, const float* __restrict__ Win,
                                                              const float* __restrict__ bin, float* __restrict__ q, float* __restrict__ k,
                                                              float* __restrict__ v, float* __restrict__ norm_out, int M, float qscale,
                                                              int kv_from_norm) {
  using SM = PreFwdSmallSmem;
  extern __shared__ __align__(16) uint8_t rs_raw[];
  __nv_bfloat16* hb = reinterpret_cast<__nv_bfloat16*>(rs_raw);
  __nv_bfloat16* Wt = hb + SM::W;
  __nv_bfloat16* Xb = hb + SM::X;
  __nv_bfloat16* Nb = hb + SM::N;
  float* Xf = reinterpret_cast<float*>(rs_raw + SM::XF_BYTES);
  const int row0 = blockIdx.x * 64;
  const int rows = min(64, M - row0);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * w + g, i1 = i0 + 8;
  {
    const float* const src[1] = {x + (long long)row0 * RS_H};
    const long long ld[1] = {RS_H};
    const int nr[1] = {rows};
    const float sc[1] = {1.f};
    __nv_bfloat16* const d[1] = {Xb};
    __nv_bfloat16* const dT[1] = {nullptr};
    float* const dF[1] = {Xf};
    rs_load<1>(src, ld, nr, sc, d, dT, dF);
  }
  {
    const float* const src[3] = {Win, Win + RS_H * RS_H, Win + 2 * RS_H * RS_H};
    const long long ld[3] = {RS_H, RS_H, RS_H};
    const int nr[3] = {64, 64, 64};
    const float sc[3] = {1.f, 1.f, 1.f};
    __nv_bfloat16* const d[3] = {Wt, Wt + RS_TILE, Wt + 2 * RS_TILE};
    __nv_bfloat16* const dT[3] = {nullptr, nullptr, nullptr};
    float* const dF[3] = {nullptr, nullptr, nullptr};
    rs_load<3>(src, ld, nr, sc, d, dT, dF);
  }
  __syncthreads();
  rs_ln_tile(Xf, ln_g, ln_b, Nb, norm_out, row0, rows);
  __syncthreads();
  const __nv_bfloat16* Akv = kv_from_norm ? Nb : Xb;
#pragma unroll 1
  for (int m = 0; m < 3; ++m) {
    float acc[8][4];
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) acc[nb][0] = acc[nb][1] = acc[nb][2] = acc[nb][3] = 0.f;
    rs_fgemm(acc, m == 0 ? Nb : Akv, Wt + m * RS_TILE, 16 * w);
    float* out = m == 0 ? q : m == 1 ? k : v;
    const float sc = m == 0 ? qscale : 1.f;
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      const int c = 8 * nb + 2 * t;
      const float2 b = __ldg(reinterpret_cast<const float2*>(bin + m * RS_H + c));
      if (i0 < rows) *reinterpret_cast<float2*>(out + (long long)(row0 + i0) * RS_H + c) = make_float2((acc[nb][0] + b.x) * sc, (acc[nb][1] + b.y) * sc);
      if (i1 < rows) *reinterpret_cast<float2*>(out + (long long)(row0 + i1) * RS_H + c) = make_float2((acc[nb][2] + b.x) * sc, (acc[nb][3] + b.y) * sc);
    }
  }
}

// -------------------------------------------------------------------------------------------------
// post_fwd_small_kernel == post_fwd_kernel (kernels_fwd.cuh), H == 64, bf16 mode.  Only the context tile and the three weight
// matrices live in shared memory; LayerNorms, residuals, dropout, ReLU and the three chained products stay in MMA fragments
// (accumulators of one product are re-packed as the A fragments of the next).
// -------------------------------------------------------------------------------------------------
struct PostFwdSmallSmem {
  static constexpr int W = 0, C = 3 * RS_TILE;       // Wo, C1, C2 | ctx
  static constexpr size_t TOTAL_BYTES = (size_t)(C + RS_TILE) * 2;
};

// LayerNorm (eps 1e-8, two-pass) of the two rows a thread co-owns with its quad, in place on fragments
__device__ __forceinline__ void frag_ln(float (&v)[8][4], const float* __restrict__ gamma, const float* __restrict__ beta, int t) {
  float s0 = 0.f, s1 = 0.f;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) { s0 += v[nb][0] + v[nb][1]; s1 += v[nb][2] + v[nb][3]; }
  s0 += __shfl_xor_sync(0xffffffffu, s0, 1); s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
  s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
  const float m0 = s0 * (1.0f / RS_H), m1 = s1 * (1.0f / RS_H);
  float q0 = 0.f, q1 = 0.f;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const float a = v[nb][0] - m0, b = v[nb][1] - m0, c = v[nb][2] - m1, d = v[nb][3] - m1;
    q0 += a * a + b * b; q1 += c * c + d * d;
  }
  q0 += __shfl_xor_sync(0xffffffffu, q0, 1); q0 += __shfl_xor_sync(0xffffffffu, q0, 2);
  q1 += __shfl_xor_sync(0xffffffffu, q1, 1); q1 += __shfl_xor_sync(0xffffffffu, q1, 2);
  const float r0 = 1.0f / sqrtf(q0 * (1.0f / RS_H) + 1e-8f), r1 = 1.0f / sqrtf(q1 * (1.0f / RS_H) + 1e-8f);
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const float2 ga = __ldg(reinterpret_cast<const float2*>(gamma + 8 * nb + 2 * t)), be = __ldg(reinterpret_cast<const float2*>(beta + 8 * nb + 2 * t));
    v[nb][0] = (v[nb][0] - m0) * r0 * ga.x + be.x; v[nb][1] = (v[nb][1] - m0) * r0 * ga.y + be.y;
    v[nb][2] = (v[nb][2] - m1) * r1 * ga.x + be.x; v[nb][3] = (v[nb][3] - m1) * r1 * ga.y + be.y;
  }
}

// out[nb] += A * W^T with A given as accumulator fragments (rows of this warp, k = 0..63) and W an n-major weight tile
__device__ __forceinline__ void rs_fgemm_frag(float (&out)[8][4], const float (&a_in)[8][4], const __nv_bfloat16* __restrict__ W) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t a[4];
    a[0] = pack_bf16(a_in[2 * ks][0], a_in[2 * ks][1]);
    a[1] = pack_bf16(a_in[2 * ks][2], a_in[2 * ks][3]);
    a[2] = pack_bf16(a_in[2 * ks + 1][0], a_in[2 * ks + 1][1]);
    a[3] = pack_bf16(a_in[2 * ks + 1][2], a_in[2 * ks + 1][3]);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      uint32_t b0, b1;
      frag_b(b0, b1, W, 8 * nb, 16 * ks);
      mma16816(out[nb], a, b0, b1);
    }
  }
}

// row-site dropout multipliers of this thread's fragment elements (rows r0 / r1 are GLOBAL row indices): element (row, col) draws
// 32-bit word (col & 3) of philox(ctr = (base + row*64 + col) >> 2).  Lanes t and t^1 need the two halves of the same call: the
// even lane evaluates the calls of even column blocks, the odd lane those of odd blocks, halves are exchanged by shuffle.
__device__ __forceinline__ void frag_drop(float (&m)[8][4], const DropDesc& d, long long r0, long long r1, int t) {
  const int odd = t & 1;
#pragma unroll
  for (int np = 0; np < 4; ++np) {
    const int nb = 2 * np + odd;                                   // the block whose call this lane evaluates
    const unsigned long long c0 = (d.base + (unsigned long long)(r0 * RS_H + 8 * nb + 2 * (t & 2))) >> 2;
    const unsigned long long c1 = (d.base + (unsigned long long)(r1 * RS_H + 8 * nb + 2 * (t & 2))) >> 2;
    const float4 a = drop_mul4(d, c0), b = drop_mul4(d, c1);
    // partner needs: from an even lane (block 2np) the upper half (.z,.w); from an odd lane (block 2np+1) the lower half (.x,.y)
    const float ax = __shfl_xor_sync(0xffffffffu, odd ? a.x : a.z, 1), ay = __shfl_xor_sync(0xffffffffu, odd ? a.y : a.w, 1);
    const float bx = __shfl_xor_sync(0xffffffffu, odd ? b.x : b.z, 1), by = __shfl_xor_sync(0xffffffffu, odd ? b.y : b.w, 1);
    // block 2np: even lane owns (.x,.y) of its own call, odd lane takes the partner's upper half
    m[2 * np][0] = odd ? ax : a.x; m[2 * np][1] = odd ? ay : a.y; m[2 * np][2] = odd ? bx : b.x; m[2 * np][3] = odd ? by : b.y;
    // block 2np+1: odd lane owns (.z,.w) of its own call, even lane takes the partner's lower half
    m[2 * np + 1][0] = odd ? a.z : ax; m[2 * np + 1][1] = odd ? a.w : ay; m[2 * np + 1][2] = odd ? b.z : bx; m[2 * np + 1][3] = odd ? b.w : by;
  }
}

__device__ __forceinline__ void cta128_accumulate(double v, double* dst, double* scratch) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) atomicAdd(dst, (scratch[0] + scratch[1]) + (scratch[2] + scratch[3]));
}

template <bool IS_DEC>
__global__ void __launch_bounds__(AS_NT) post_fwd_small_kernel(PostFwdArgs p) {
  using SM = PostFwdSmallSmem;
  extern __shared__ __align__(16) uint8_t rs_raw[];
  __shared__ double red[4];
  __nv_bfloat16* hb = reinterpret_cast<__nv_bfloat16*>(rs_raw);
  __nv_bfloat16* Wt = hb + SM::W;
  __nv_bfloat16* Cs = hb + SM::C;
  const int M = p.M;
  const int row0 = blockIdx.x * 64;
  const int rows = min(64, M - row0);
  const long long g0 = (long long)row0 * RS_H;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * w + g, i1 = i0 + 8;
  const bool v0 = i0 < rows, v1 = i1 < rows;
  rs_load1(p.ctx + g0, rows, 1.f, Cs);
  {
    const float* const src[3] = {p.Wo, p.C1, p.C2};
    const long long ld[3] = {RS_H, RS_H, RS_H};
    const int nr[3] = {64, 64, 64};
    const float sc[3] = {1.f, 1.f, 1.f};
    __nv_bfloat16* const d[3] = {Wt, Wt + RS_TILE, Wt + 2 * RS_TILE};
    __nv_bfloat16* const dT[3] = {nullptr, nullptr, nullptr};
    float* const dF[3] = {nullptr, nullptr, nullptr};
    rs_load<3>(src, ld, nr, sc, d, dT, dF);
  }
  // residual stream at the fragment positions (enc: block input x -> LN1 ; dec: d, added at the very end)
  float res[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    const float2 a = v0 ? __ldg(reinterpret_cast<const float2*>(p.resid + g0 + (long long)i0 * RS_H + c)) : make_float2(0.f, 0.f);
    const float2 b = v1 ? __ldg(reinterpret_cast<const float2*>(p.resid + g0 + (long long)i1 * RS_H + c)) : make_float2(0.f, 0.f);
    res[nb][0] = a.x; res[nb][1] = a.y; res[nb][2] = b.x; res[nb][3] = b.y;
  }
  const int keep0 = v0 ? p.ids[row0 + i0] : 0, keep1 = v1 ? p.ids[row0 + i1] : 0;
  if (!IS_DEC) frag_ln(res, p.ln1_g, p.ln1_b, t);          // Qn = LN1(x)
  __syncthreads();
  // y (enc) / c (dec) = ctx Wo^T + bo (+ Qn)
  float u[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) u[nb][0] = u[nb][1] = u[nb][2] = u[nb][3] = 0.f;
  rs_fgemm(u, Cs, Wt, 16 * w);
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    const float2 b = __ldg(reinterpret_cast<const float2*>(p.bo + c));
    u[nb][0] += b.x; u[nb][1] += b.y; u[nb][2] += b.x; u[nb][3] += b.y;
    if (!IS_DEC) { u[nb][0] += res[nb][0]; u[nb][1] += res[nb][1]; u[nb][2] += res[nb][2]; u[nb][3] += res[nb][3]; }
    if (p.u_save) {
      if (v0) *reinterpret_cast<float2*>(p.u_save + g0 + (long long)i0 * RS_H + c) = make_float2(u[nb][0], u[nb][1]);
      if (v1) *reinterpret_cast<float2*>(p.u_save + g0 + (long long)i1 * RS_H + c) = make_float2(u[nb][2], u[nb][3]);
    }
  }
  if (!IS_DEC) {
    // independence head on the per-head context slices (bf16 context tile): one thread per (row, head)
    if (p.rec || p.acc) {
      const int nh = p.nh, hd = RS_H / nh;
      double nll = 0.0;
      for (int i = threadIdx.x; i < 64 * nh; i += AS_NT) {
        const int r = i / nh, c = i - r * nh;
        if (r >= rows) continue;
        float lg[8];
        float mx = -INFINITY;
        for (int j = 0; j < nh; ++j) {
          float sacc = 0.f;
          for (int dd = 0; dd < hd; ++dd) sacc = fmaf(__bfloat162float(Cs[r * RS_LD + c * hd + dd]), __ldg(p.Wsp + j * hd + dd), sacc);
          lg[j] = sacc + __ldg(p.bsp + j);
          mx = fmaxf(mx, lg[j]);
        }
        float se = 0.f;
        for (int j = 0; j < nh; ++j) se += expf(lg[j] - mx);
        const float lz = mx + logf(se);
        if (p.rec)
          for (int j = 0; j < nh; ++j) p.rec[((long long)(row0 + r) * nh + c) * nh + j] = lg[j] - lz;
        nll -= (double)(lg[c] - lz);
      }
      if (p.acc) cta128_accumulate(nll, p.acc, red);
    }
    frag_ln(u, p.ln2_g, p.ln2_b, t);                       // z = LN2(y)
  }
  // h1 = z C1^T + c1 ; a = relu(drop1(h1))
  float h[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) h[nb][0] = h[nb][1] = h[nb][2] = h[nb][3] = 0.f;
  rs_fgemm_frag(h, u, Wt + RS_TILE);
  float mk[8][4];
  if (p.drop1.enabled) frag_drop(mk, p.drop1, row0 + i0, row0 + i1, t);
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    const float2 b = __ldg(reinterpret_cast<const float2*>(p.c1 + c));
    h[nb][0] += b.x; h[nb][1] += b.y; h[nb][2] += b.x; h[nb][3] += b.y;
    if (p.h1_save) {
      if (v0) *reinterpret_cast<float2*>(p.h1_save + g0 + (long long)i0 * RS_H + c) = make_float2(h[nb][0], h[nb][1]);
      if (v1) *reinterpret_cast<float2*>(p.h1_save + g0 + (long long)i1 * RS_H + c) = make_float2(h[nb][2], h[nb][3]);
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float x = h[nb][e];
      if (p.drop1.enabled) x *= mk[nb][e];
      h[nb][e] = fmaxf(x, 0.f);
    }
  }
  // h2 = a C2^T + c2 ; out = (drop2(h2) + z [+ d]) * keep
  float o[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) o[nb][0] = o[nb][1] = o[nb][2] = o[nb][3] = 0.f;
  rs_fgemm_frag(o, h, Wt + 2 * RS_TILE);
  if (p.drop2.enabled) frag_drop(mk, p.drop2, row0 + i0, row0 + i1, t);
  double sq = 0.0;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    const float2 b = __ldg(reinterpret_cast<const float2*>(p.c2 + c));
    float y[4] = {o[nb][0] + b.x, o[nb][1] + b.y, o[nb][2] + b.x, o[nb][3] + b.y};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (p.drop2.enabled) y[e] *= mk[nb][e];
      y[e] += u[nb][e];
      if (IS_DEC) y[e] += res[nb][e];
    }
    if (keep0 == 0) { y[0] = 0.f; y[1] = 0.f; }
    if (keep1 == 0) { y[2] = 0.f; y[3] = 0.f; }
    if (v0) *reinterpret_cast<float2*>(p.out + g0 + (long long)i0 * RS_H + c) = make_float2(y[0], y[1]);
    if (v1) *reinterpret_cast<float2*>(p.out + g0 + (long long)i1 * RS_H + c) = make_float2(y[2], y[3]);
    if (IS_DEC && p.enc_in) {
      if (v0) { const float2 e = *reinterpret_cast<const float2*>(p.enc_in + g0 + (long long)i0 * RS_H + c); sq += (double)((e.x - y[0]) * (e.x - y[0]) + (e.y - y[1]) * (e.y - y[1])); }
      if (v1) { const float2 e = *reinterpret_cast<const float2*>(p.enc_in + g0 + (long long)i1 * RS_H + c); sq += (double)((e.x - y[2]) * (e.x - y[2]) + (e.y - y[3]) * (e.y - y[3])); }
    }
  }
  if (IS_DEC && p.acc) cta128_accumulate(sq, p.acc, red);
}


// -------------------------------------------------------------------------------------------------
// post_bwd_small_kernel == post_bwd_kernel (kernels_bwd.cuh), H == 64, bf16 mode.  Weights C2, C1, Wo and the attention context
// stay in shared memory; the gradient stream dO -> dh2 -> da -> dh1 -> dz -> dy -> dctx lives in fragments of the chain warps and is
// only parked in a bf16 tile where a weight-gradient product needs all rows of the CTA.  Each of the three weight gradients has its
// own operand tiles, so the chain warps never wait for the wgrad warps.
// -------------------------------------------------------------------------------------------------
struct PostBwdSmallSmem {
  // C2, C1, Wo | ctx | dh2, a (dC2) | dh1, z (dC1) | dy (dWo, with ctx)
  static constexpr int W = 0, C = 3 * RS_TILE, T3 = C + RS_TILE, X3 = T3 + RS_TILE, T5 = X3 + RS_TILE, X5 = T5 + RS_TILE, T8 = X5 + RS_TILE;
  static constexpr size_t LG_BYTES = (size_t)(T8 + RS_TILE) * 2;                      // logits / dlogits [64][nh*nh] fp32 (+ nh)
  static constexpr size_t TOTAL_BYTES = LG_BYTES + (size_t)(64 * 64 + 8) * 4;
};
// named barriers of post_bwd_small_kernel: operand tiles of dC1 / dWo complete, head logits complete, chain warps only
constexpr int RS_BAR_S5 = 1, RS_BAR_S8 = 2, RS_BAR_HEAD = 3, RS_BAR_CHAIN = 4;

// D[nb] += A * W with A given as fragments (rows of this warp, k = j = 0..63) and W[j][c] a row-major weight tile
__device__ __forceinline__ void rs_dgrad_frag(float (&out)[8][4], const float (&a_in)[8][4], const __nv_bfloat16* __restrict__ W) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t a[4];
    a[0] = pack_bf16(a_in[2 * ks][0], a_in[2 * ks][1]);
    a[1] = pack_bf16(a_in[2 * ks][2], a_in[2 * ks][3]);
    a[2] = pack_bf16(a_in[2 * ks + 1][0], a_in[2 * ks + 1][1]);
    a[3] = pack_bf16(a_in[2 * ks + 1][2], a_in[2 * ks + 1][3]);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      uint32_t b0, b1;
      frag_b_t(b0, b1, W, 16 * ks, 8 * nb);
      mma16816(out[nb], a, b0, b1);
    }
  }
}

// fragments -> bf16 tile rows of this thread
__device__ __forceinline__ void frag_store_tile(__nv_bfloat16* __restrict__ T, const float (&v)[8][4], int i0, int i1, int t) {
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    *reinterpret_cast<uint32_t*>(T + i0 * RS_LD + 8 * nb + 2 * t) = pack_bf16(v[nb][0], v[nb][1]);
    *reinterpret_cast<uint32_t*>(T + i1 * RS_LD + 8 * nb + 2 * t) = pack_bf16(v[nb][2], v[nb][3]);
  }
}

// fragment-position loads / stores of a row-major fp32 [M][64] tensor (rows of this thread: i0, i1; validity v0, v1)
__device__ __forceinline__ void frag_load(float (&v)[8][4], const float* __restrict__ src, int i0, int i1, bool v0, bool v1, int t) {
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    const float2 a = (src && v0) ? __ldg(reinterpret_cast<const float2*>(src + (long long)i0 * RS_H + c)) : make_float2(0.f, 0.f);
    const float2 b = (src && v1) ? __ldg(reinterpret_cast<const float2*>(src + (long long)i1 * RS_H + c)) : make_float2(0.f, 0.f);
    v[nb][0] = a.x; v[nb][1] = a.y; v[nb][2] = b.x; v[nb][3] = b.y;
  }
}
__device__ __forceinline__ void frag_store(float* __restrict__ dst, const float (&v)[8][4], int i0, int i1, bool v0, bool v1, int t) {
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    if (v0) *reinterpret_cast<float2*>(dst + (long long)i0 * RS_H + c) = make_float2(v[nb][0], v[nb][1]);
    if (v1) *reinterpret_cast<float2*>(dst + (long long)i1 * RS_H + c) = make_float2(v[nb][2], v[nb][3]);
  }
}

// LayerNorm adjoint entirely on fragments: Y = LN input rows (fragments), D = grad wrt LN output -> grad wrt LN input
__device__ __forceinline__ void frag_ln_bwd(float (&D)[8][4], const float (&Y)[8][4], const float* __restrict__ gamma,
                                            float* __restrict__ ggamma, float* __restrict__ gbeta, bool v0, bool v1, int g, int t) {
  float s0 = 0.f, s1 = 0.f;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) { s0 += Y[nb][0] + Y[nb][1]; s1 += Y[nb][2] + Y[nb][3]; }
  s0 += __shfl_xor_sync(0xffffffffu, s0, 1); s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
  s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
  const float m0 = s0 * (1.0f / RS_H), m1 = s1 * (1.0f / RS_H);
  float q0 = 0.f, q1 = 0.f;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const float a = Y[nb][0] - m0, b = Y[nb][1] - m0, c = Y[nb][2] - m1, d = Y[nb][3] - m1;
    q0 += a * a + b * b; q1 += c * c + d * d;
  }
  q0 += __shfl_xor_sync(0xffffffffu, q0, 1); q0 += __shfl_xor_sync(0xffffffffu, q0, 2);
  q1 += __shfl_xor_sync(0xffffffffu, q1, 1); q1 += __shfl_xor_sync(0xffffffffu, q1, 2);
  const float r0 = 1.0f / sqrtf(q0 * (1.0f / RS_H) + 1e-8f), r1 = 1.0f / sqrtf(q1 * (1.0f / RS_H) + 1e-8f);
  float a10 = 0.f, a20 = 0.f, a11 = 0.f, a21 = 0.f;
  float xh[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    const float2 ga = __ldg(reinterpret_cast<const float2*>(gamma + c));
    xh[nb][0] = (Y[nb][0] - m0) * r0; xh[nb][1] = (Y[nb][1] - m0) * r0;
    xh[nb][2] = (Y[nb][2] - m1) * r1; xh[nb][3] = (Y[nb][3] - m1) * r1;
    float dg0 = D[nb][0] * xh[nb][0] + D[nb][2] * xh[nb][2], dg1 = D[nb][1] * xh[nb][1] + D[nb][3] * xh[nb][3];
    float db0 = D[nb][0] + D[nb][2], db1 = D[nb][1] + D[nb][3];
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) {
      dg0 += __shfl_xor_sync(0xffffffffu, dg0, o); dg1 += __shfl_xor_sync(0xffffffffu, dg1, o);
      db0 += __shfl_xor_sync(0xffffffffu, db0, o); db1 += __shfl_xor_sync(0xffffffffu, db1, o);
    }
    if (g == 0) {
      atomicAdd(ggamma + c, dg0); atomicAdd(ggamma + c + 1, dg1);
      atomicAdd(gbeta + c, db0); atomicAdd(gbeta + c + 1, db1);
    }
    D[nb][0] *= ga.x; D[nb][1] *= ga.y; D[nb][2] *= ga.x; D[nb][3] *= ga.y;
    a10 += D[nb][0] + D[nb][1]; a20 += D[nb][0] * xh[nb][0] + D[nb][1] * xh[nb][1];
    a11 += D[nb][2] + D[nb][3]; a21 += D[nb][2] * xh[nb][2] + D[nb][3] * xh[nb][3];
  }
#pragma unroll
  for (int o = 1; o < 4; o <<= 1) {
    a10 += __shfl_xor_sync(0xffffffffu, a10, o); a20 += __shfl_xor_sync(0xffffffffu, a20, o);
    a11 += __shfl_xor_sync(0xffffffffu, a11, o); a21 += __shfl_xor_sync(0xffffffffu, a21, o);
  }
  a10 *= 1.0f / RS_H; a20 *= 1.0f / RS_H; a11 *= 1.0f / RS_H; a21 *= 1.0f / RS_H;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    D[nb][0] = v0 ? r0 * (D[nb][0] - a10 - xh[nb][0] * a20) : 0.f;
    D[nb][1] = v0 ? r0 * (D[nb][1] - a10 - xh[nb][1] * a20) : 0.f;
    D[nb][2] = v1 ? r1 * (D[nb][2] - a11 - xh[nb][2] * a21) : 0.f;
    D[nb][3] = v1 ? r1 * (D[nb][3] - a11 - xh[nb][3] * a21) : 0.f;
  }
}

template <bool IS_DEC>
__global__ void __launch_bounds__(RS_BWD_NT, 2) post_bwd_small_kernel(PostBwdArgs p) {
  using SM = PostBwdSmallSmem;
  extern __shared__ __align__(16) uint8_t rs_raw[];
  __nv_bfloat16* hb = reinterpret_cast<__nv_bfloat16*>(rs_raw);
  __nv_bfloat16* Wt = hb + SM::W;            // [0] C2, [1] C1, [2] Wo
  __nv_bfloat16* Cs = hb + SM::C;
  __nv_bfloat16* T3 = hb + SM::T3;
  __nv_bfloat16* X3 = hb + SM::X3;
  __nv_bfloat16* T5 = hb + SM::T5;
  __nv_bfloat16* X5 = hb + SM::X5;
  __nv_bfloat16* T8 = hb + SM::T8;
  float* lgs = reinterpret_cast<float*>(rs_raw + SM::LG_BYTES);
  const int M = p.M;
  const int row0 = blockIdx.x * 64;
  const int rows = min(64, M - row0);
  const long long g0 = (long long)row0 * RS_H;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * w + g, i1 = i0 + 8;
  const bool v0 = i0 < rows, v1 = i1 < rows;
  const bool head = !IS_DEC && (p.nll_coef != 0.f || p.drec);
  if (w >= 4) {                              // the wgrad warps stage ctx and the weights while the chain warps start
    rs_load1<RS_BWD_NT - RS_CHAIN_NT, RS_CHAIN_NT>(p.ctx + g0, rows, 1.f, Cs);
    const float* const src[3] = {p.C2, p.C1, p.Wo};
    const long long ld[3] = {RS_H, RS_H, RS_H};
    const int nr[3] = {64, 64, 64};
    const float sc[3] = {1.f, 1.f, 1.f};
    __nv_bfloat16* const d[3] = {Wt, Wt + RS_TILE, Wt + 2 * RS_TILE};
    __nv_bfloat16* const dT[3] = {nullptr, nullptr, nullptr};
    float* const dF[3] = {nullptr, nullptr, nullptr};
    rs_load<3, RS_BWD_NT - RS_CHAIN_NT, RS_CHAIN_NT>(src, ld, nr, sc, d, dT, dF);
  }
  // ---- 1./2. dO, a = relu(h1 m1), dh2 = dO m2 on fragments
  float G[8][4], D2[8][4];
  uint32_t m1bits = 0u;                      // bit (4 nb + e): element kept by dropout 1 AND a > 0
  if (w < 4) {
    frag_load(G, p.dout ? p.dout + g0 : nullptr, i0, i1, v0, v1, t);
    if (IS_DEC && p.enc_in) {
      float O[8][4], E[8][4];
      frag_load(O, p.out + g0, i0, i1, v0, v1, t);
      frag_load(E, p.enc_in + g0, i0, i1, v0, v1, t);
#pragma unroll
      for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
        for (int e = 0; e < 4; ++e) { O[nb][e] = p.mse_coef * (O[nb][e] - E[nb][e]); G[nb][e] += O[nb][e]; O[nb][e] = -O[nb][e]; }
      }
      if (p.denc) frag_store(p.denc + g0, O, i0, i1, v0, v1, t);
    }
    {
      const int k0 = v0 ? p.ids[row0 + i0] : 0, k1 = v1 ? p.ids[row0 + i1] : 0;
#pragma unroll
      for (int nb = 0; nb < 8; ++nb) {
        if (k0 == 0) { G[nb][0] = 0.f; G[nb][1] = 0.f; }
        if (k1 == 0) { G[nb][2] = 0.f; G[nb][3] = 0.f; }
      }
    }
    float A[8][4], mk[8][4];
    frag_load(A, p.h1 + g0, i0, i1, v0, v1, t);
    if (p.drop1.enabled) frag_drop(mk, p.drop1, row0 + i0, row0 + i1, t);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float x = A[nb][e];
        if (p.drop1.enabled) x *= mk[nb][e];
        A[nb][e] = fmaxf(x, 0.f);
        if (A[nb][e] > 0.f) m1bits |= 1u << (4 * nb + e);
      }
    }
    frag_store_tile(X3, A, i0, i1, t);
    if (p.drop2.enabled) frag_drop(mk, p.drop2, row0 + i0, row0 + i1, t);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
      for (int e = 0; e < 4; ++e) D2[nb][e] = p.drop2.enabled ? G[nb][e] * mk[nb][e] : G[nb][e];
    }
    frag_store_tile(T3, D2, i0, i1, t);
  }
  __syncthreads();                           // weights, ctx and the operands of step 3 are in shared memory
  if (w >= 4) {
    // ---- wgrad warps: 3. dC2 += dh2^T a ; 5. dC1 += dh1^T z ; 8. dWo += dy^T ctx (and the bias column sums)
    rs_wgrad_rm(T3, X3, p.gC2, p.gc2, w - 4);
    rs_bar_sync(RS_BAR_S5, RS_BWD_NT);
    rs_wgrad_rm(T5, X5, p.gC1, p.gc1, w - 4);
    rs_bar_sync(RS_BAR_S8, RS_BWD_NT);
    rs_wgrad_rm(T8, Cs, p.gWo, p.gbo, w - 4);
    if (head) {
      // ---- 9. independence-head weight gradient: dWsp[j][d] += sum_{r,c} dl[r][c][j] ctx[r][c*hd+d], dbsp from the CTA's sums
      const int nh = p.nh, hd = RS_H / nh, n2 = nh * nh;
      const float* dbs = lgs + 64 * n2;
      rs_bar_sync(RS_BAR_HEAD, RS_BWD_NT);
      for (int i = threadIdx.x - RS_CHAIN_NT; i < nh * hd; i += RS_BWD_NT - RS_CHAIN_NT) {
        const int j = i / hd, dd = i - j * hd;
        float accw = 0.f;
        for (int r = 0; r < rows; ++r)
          for (int c = 0; c < nh; ++c) accw = fmaf(lgs[r * n2 + c * nh + j], __bfloat162float(Cs[r * RS_LD + c * hd + dd]), accw);
        atomicAdd(p.gWsp + i, accw);
      }
      for (int i = threadIdx.x - RS_CHAIN_NT; i < nh; i += RS_BWD_NT - RS_CHAIN_NT) atomicAdd(p.gbsp + i, dbs[i]);
    }
    return;
  }
  // ---- 4. da = dh2 C2 ; dh1 = da [a>0] m1
  float H1[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) H1[nb][0] = H1[nb][1] = H1[nb][2] = H1[nb][3] = 0.f;
  rs_dgrad_frag(H1, D2, Wt);
  {
    const float sc1 = p.drop1.enabled ? p.drop1.scale : 1.f;
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
      for (int e = 0; e < 4; ++e) H1[nb][e] = (m1bits >> (4 * nb + e)) & 1u ? H1[nb][e] * sc1 : 0.f;
    }
  }
  // ---- 5. z = LN2(y) (enc) / c (dec): operands of dC1 += dh1^T z ; dc1 += colsum(dh1).  Step 6 takes dh1 back from its tile
  // (the same bf16 values its fragments would pack to), so dh1 is not held in registers next to y and z.
  frag_store_tile(T5, H1, i0, i1, t);
  float Y[8][4];
  frag_load(Y, p.u + g0, i0, i1, v0, v1, t);
  {
    float Z[8][4];
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) { Z[nb][0] = Y[nb][0]; Z[nb][1] = Y[nb][1]; Z[nb][2] = Y[nb][2]; Z[nb][3] = Y[nb][3]; }
    if (!IS_DEC) {
      frag_ln(Z, p.ln2_g, p.ln2_b, t);
      if (!v0) { for (int nb = 0; nb < 8; ++nb) { Z[nb][0] = 0.f; Z[nb][1] = 0.f; } }
      if (!v1) { for (int nb = 0; nb < 8; ++nb) { Z[nb][2] = 0.f; Z[nb][3] = 0.f; } }
    }
    frag_store_tile(X5, Z, i0, i1, t);
  }
  __syncwarp();                              // step 6 reads this warp's rows of dh1 through ldmatrix
  rs_bar_arrive(RS_BAR_S5);
  // ---- 6. dz (enc) / dc (dec) = dO + dh1 C1
  float DZ[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) { DZ[nb][0] = G[nb][0]; DZ[nb][1] = G[nb][1]; DZ[nb][2] = G[nb][2]; DZ[nb][3] = G[nb][3]; }
  rs_dgrad(DZ, T5, Wt + RS_TILE, 16 * w);
  if (!IS_DEC) {
    // ---- 7. dy = LN2^T(dz) ; dres = dy
    frag_ln_bwd(DZ, Y, p.ln2_g, p.gln2_g, p.gln2_b, v0, v1, (threadIdx.x >> 2) & 7, t);   // g recomputed: held live it spills at 128 registers
    frag_store(p.dres + g0, DZ, i0, i1, v0, v1, t);
  } else {
    frag_store(p.dres + g0, G, i0, i1, v0, v1, t);     // dd = dO
  }
  // ---- 8. operand of dWo += dy^T ctx ; dbo += colsum(dy) ; dctx = dy Wo
  frag_store_tile(T8, DZ, i0, i1, t);
  rs_bar_arrive(RS_BAR_S8);
  float DC[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) DC[nb][0] = DC[nb][1] = DC[nb][2] = DC[nb][3] = 0.f;
  rs_dgrad_frag(DC, DZ, Wt + 2 * RS_TILE);
  if (head) {
    // ---- 9. independence-head adjoint (per-head logits from the bf16 context tile)
    const int nh = p.nh, hd = RS_H / nh, n2 = nh * nh;
    float* dbs = lgs + 64 * n2;
    for (int i = threadIdx.x; i < nh; i += RS_CHAIN_NT) dbs[i] = 0.f;
    rs_bar_sync(RS_BAR_CHAIN, RS_CHAIN_NT);
    for (int i = threadIdx.x; i < 64 * nh; i += RS_CHAIN_NT) {
      const int r = i / nh, c = i - r * nh;
      float* lg = lgs + r * n2 + c * nh;
      if (r >= rows) {
        for (int j = 0; j < nh; ++j) lg[j] = 0.f;
        continue;
      }
      float mx = -INFINITY;
      for (int j = 0; j < nh; ++j) {
        float sacc = 0.f;
        for (int dd = 0; dd < hd; ++dd) sacc = fmaf(__bfloat162float(Cs[r * RS_LD + c * hd + dd]), __ldg(p.Wsp + j * hd + dd), sacc);
        lg[j] = sacc + __ldg(p.bsp + j);
        mx = fmaxf(mx, lg[j]);
      }
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
    rs_bar_arrive(RS_BAR_HEAD);
    rs_bar_sync(RS_BAR_CHAIN, RS_CHAIN_NT);
    // dctx[r][c*hd+d] += sum_j dl[r][c][j] Wsp[j][d]   (on the fragments)
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int r = e < 2 ? i0 : i1, col = 8 * nb + 2 * t + (e & 1), c = col / hd, dd = col - c * hd;
        const float* dl = lgs + r * n2 + c * nh;
        float add = 0.f;
        for (int j = 0; j < nh; ++j) add = fmaf(dl[j], __ldg(p.Wsp + j * hd + dd), add);
        DC[nb][e] += add;
      }
    }
  }
  frag_store(p.dctx + g0, DC, i0, i1, v0, v1, t);
}

// -------------------------------------------------------------------------------------------------
// pre_bwd_small2_kernel == pre_bwd_kernel (kernels_bwd.cuh): adjoint of LayerNorm + packed QKV in-projection.  The block input lives in fragments (LayerNorm forward and
// adjoint without shared memory), all three upstream gradients (dq, dk, dv) are staged as bf16 tiles in the prologue, so the
// kernel has ONE barrier and no global load on its critical path after the prologue.  Every weight-gradient operand (Tq, Tk, Tv,
// Nb, Xb) is complete at that barrier: the wgrad warps need no further handoff.
// -------------------------------------------------------------------------------------------------
struct PreBwdSmall2Smem {
  static constexpr int W = 0, TQ = 3 * RS_TILE, TK = TQ + RS_TILE, TV = TK + RS_TILE, X = TV + RS_TILE, N = X + RS_TILE;
  static constexpr size_t TOTAL_BYTES = (size_t)(N + RS_TILE) * 2;
};

// Everything of pre_bwd_small2_kernel after its prologue, for all 256 threads: the bf16 tiles Tq (dq scaled by qscale), Tk, Tv (zero in
// rows >= rows) and the weights Wt are in shared memory; Xb and Nb are free tiles (x and LN(x) are staged there).  Xf: the block input
// at the fragment positions of chain warps 0-3 (frag_load of p.x), loaded by the caller so that its latency can hide behind a barrier.
__device__ __forceinline__ void pre_bwd_small_tail(const PreBwdArgs& p, const float (&Xf)[8][4], const __nv_bfloat16* Wt, const __nv_bfloat16* Tq,
                                                   const __nv_bfloat16* Tk, const __nv_bfloat16* Tv, __nv_bfloat16* Xb, __nv_bfloat16* Nb,
                                                   long long row0, int rows) {
  const long long g0 = row0 * RS_H;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * w + g, i1 = i0 + 8;
  const bool v0 = i0 < rows, v1 = i1 < rows;
  if (w < 4) {
    float Nf[8][4];
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) { Nf[nb][0] = Xf[nb][0]; Nf[nb][1] = Xf[nb][1]; Nf[nb][2] = Xf[nb][2]; Nf[nb][3] = Xf[nb][3]; }
    frag_ln(Nf, p.ln_g, p.ln_b, t);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      if (!v0) { Nf[nb][0] = 0.f; Nf[nb][1] = 0.f; }
      if (!v1) { Nf[nb][2] = 0.f; Nf[nb][3] = 0.f; }
    }
    frag_store_tile(Nb, Nf, i0, i1, t);
    if (!p.kv_from_norm) frag_store_tile(Xb, Xf, i0, i1, t);
  }
  __syncthreads();
  if (w >= 4) {   // ---- wgrad warps: dWq += dq^T LN(x) ; dWk += dk^T xkv ; dWv += dv^T xkv (and the bias column sums)
    const __nv_bfloat16* Xkv = p.kv_from_norm ? Nb : Xb;
    rs_wgrad_rm(Tq, Nb, p.gWin, p.gbin, w - 4);
    rs_wgrad_rm(Tk, Xkv, p.gWin + (long long)RS_H * RS_H, p.gbin + RS_H, w - 4);
    rs_wgrad_rm(Tv, Xkv, p.gWin + 2ll * RS_H * RS_H, p.gbin + 2 * RS_H, w - 4);
    return;
  }
  // ---- q projection
  float D[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) D[nb][0] = D[nb][1] = D[nb][2] = D[nb][3] = 0.f;
  rs_dgrad(D, Tq, Wt, 16 * w);
  if (p.dnorm_extra) {
    float E[8][4];
    frag_load(E, p.dnorm_extra + g0, i0, i1, v0, v1, t);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) { D[nb][0] += E[nb][0]; D[nb][1] += E[nb][1]; D[nb][2] += E[nb][2]; D[nb][3] += E[nb][3]; }
  }
  if (!p.kv_from_norm) frag_ln_bwd(D, Xf, p.ln_g, p.gln_g, p.gln_b, v0, v1, g, t);     // encoder: k, v come from x itself
  // ---- k and v projections
  rs_dgrad(D, Tk, Wt + RS_TILE, 16 * w);
  rs_dgrad(D, Tv, Wt + 2 * RS_TILE, 16 * w);
  if (p.kv_from_norm) frag_ln_bwd(D, Xf, p.ln_g, p.gln_g, p.gln_b, v0, v1, g, t);      // decoder: q, k, v all come from LN(x)
  if (p.dx_extra) {
    float E[8][4];
    frag_load(E, p.dx_extra + g0, i0, i1, v0, v1, t);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) { D[nb][0] += E[nb][0]; D[nb][1] += E[nb][1]; D[nb][2] += E[nb][2]; D[nb][3] += E[nb][3]; }
  }
  frag_store(p.dx + g0, D, i0, i1, v0, v1, t);
}

__global__ void __launch_bounds__(RS_BWD_NT, 2) pre_bwd_small2_kernel(PreBwdArgs p) {
  using SM = PreBwdSmall2Smem;
  extern __shared__ __align__(16) uint8_t rs_raw[];
  __nv_bfloat16* hb = reinterpret_cast<__nv_bfloat16*>(rs_raw);
  __nv_bfloat16* Wt = hb + SM::W;
  __nv_bfloat16* Tq = hb + SM::TQ;
  __nv_bfloat16* Tk = hb + SM::TK;
  __nv_bfloat16* Tv = hb + SM::TV;
  __nv_bfloat16* Xb = hb + SM::X;
  __nv_bfloat16* Nb = hb + SM::N;
  const int row0 = blockIdx.x * 64;
  const int rows = min(64, p.M - row0);
  const long long g0 = (long long)row0 * RS_H;
  {
    const float* const src[3] = {p.dq + g0, p.dk + g0, p.dv + g0};
    const long long ld[3] = {RS_H, RS_H, RS_H};
    const int nr[3] = {rows, rows, rows};
    const float sc[3] = {p.qscale, 1.f, 1.f};
    __nv_bfloat16* const d[3] = {Tq, Tk, Tv};
    __nv_bfloat16* const dT[3] = {nullptr, nullptr, nullptr};
    float* const dF[3] = {nullptr, nullptr, nullptr};
    rs_load<3, RS_BWD_NT>(src, ld, nr, sc, d, dT, dF);
  }
  {
    const float* const src[3] = {p.Win, p.Win + RS_H * RS_H, p.Win + 2 * RS_H * RS_H};
    const long long ld[3] = {RS_H, RS_H, RS_H};
    const int nr[3] = {64, 64, 64};
    const float sc[3] = {1.f, 1.f, 1.f};
    __nv_bfloat16* const d[3] = {Wt, Wt + RS_TILE, Wt + 2 * RS_TILE};
    __nv_bfloat16* const dT[3] = {nullptr, nullptr, nullptr};
    float* const dF[3] = {nullptr, nullptr, nullptr};
    rs_load<3, RS_BWD_NT>(src, ld, nr, sc, d, dT, dF);
  }
  float Xf[8][4];
  {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, i0 = 16 * w + (lane >> 2), i1 = i0 + 8;
    if (w < 4) frag_load(Xf, p.x + g0, i0, i1, i0 < rows, i1 < rows, lane & 3);
  }
  pre_bwd_small_tail(p, Xf, Wt, Tq, Tk, Tv, Xb, Nb, row0, rows);
}

// -------------------------------------------------------------------------------------------------
// mid_fwd_small_kernel == mid_fwd_kernel (kernels_fwd.cuh): a = ctx1 Wo1^T + bo1 ; q2 = (a Wq2^T + bq2) s ; k2, v2 = feats Wkv2^T + bkv2.
// `a` goes from the accumulator fragments of the first product straight into the A fragments of the second.
// -------------------------------------------------------------------------------------------------
struct MidFwdSmallSmem {
  static constexpr int W = 0, C = 4 * RS_TILE, F = C + RS_TILE;       // Wo1, Wq2, Wk2, Wv2 | ctx1 | feats
  static constexpr size_t TOTAL_BYTES = (size_t)(F + RS_TILE) * 2;
};

__global__ void __launch_bounds__(AS_NT) mid_fwd_small_kernel(const float* __restrict__ ctx1, const float* __restrict__ feats,
                                                              const float* __restrict__ Wo1, const float* __restrict__ bo1,
                                                              const float* __restrict__ Win2, const float* __restrict__ bin2,
                                                              float* __restrict__ a_out, float* __restrict__ q2, float* __restrict__ k2,
                                                              float* __restrict__ v2, int M, float qscale) {
  using SM = MidFwdSmallSmem;
  extern __shared__ __align__(16) uint8_t rs_raw[];
  __nv_bfloat16* hb = reinterpret_cast<__nv_bfloat16*>(rs_raw);
  __nv_bfloat16* Wt = hb + SM::W;
  __nv_bfloat16* Cs = hb + SM::C;
  __nv_bfloat16* Fs = hb + SM::F;
  const int row0 = blockIdx.x * 64;
  const int rows = min(64, M - row0);
  const long long g0 = (long long)row0 * RS_H;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * w + g, i1 = i0 + 8;
  {
    const float* const src[2] = {ctx1 + g0, feats + g0};
    const long long ld[2] = {RS_H, RS_H};
    const int nr[2] = {rows, rows};
    const float sc[2] = {1.f, 1.f};
    __nv_bfloat16* const d[2] = {Cs, Fs};
    __nv_bfloat16* const dT[2] = {nullptr, nullptr};
    float* const dF[2] = {nullptr, nullptr};
    rs_load<2>(src, ld, nr, sc, d, dT, dF);
  }
  {
    const float* const src[4] = {Wo1, Win2, Win2 + RS_H * RS_H, Win2 + 2 * RS_H * RS_H};
    const long long ld[4] = {RS_H, RS_H, RS_H, RS_H};
    const int nr[4] = {64, 64, 64, 64};
    const float sc[4] = {1.f, 1.f, 1.f, 1.f};
    __nv_bfloat16* const d[4] = {Wt, Wt + RS_TILE, Wt + 2 * RS_TILE, Wt + 3 * RS_TILE};
    __nv_bfloat16* const dT[4] = {nullptr, nullptr, nullptr, nullptr};
    float* const dF[4] = {nullptr, nullptr, nullptr, nullptr};
    rs_load<4>(src, ld, nr, sc, d, dT, dF);
  }
  __syncthreads();
  float acc[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) acc[nb][0] = acc[nb][1] = acc[nb][2] = acc[nb][3] = 0.f;
  rs_fgemm(acc, Cs, Wt, 16 * w);
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    const float2 b = __ldg(reinterpret_cast<const float2*>(bo1 + c));
    acc[nb][0] += b.x; acc[nb][1] += b.y; acc[nb][2] += b.x; acc[nb][3] += b.y;
    if (a_out) {
      if (i0 < rows) *reinterpret_cast<float2*>(a_out + g0 + (long long)i0 * RS_H + c) = make_float2(acc[nb][0], acc[nb][1]);
      if (i1 < rows) *reinterpret_cast<float2*>(a_out + g0 + (long long)i1 * RS_H + c) = make_float2(acc[nb][2], acc[nb][3]);
    }
  }
  {   // q2 = (a Wq2^T + bq2) * s with a taken from the fragments
    float o[8][4];
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) o[nb][0] = o[nb][1] = o[nb][2] = o[nb][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t a[4];
      a[0] = pack_bf16(acc[2 * ks][0], acc[2 * ks][1]);
      a[1] = pack_bf16(acc[2 * ks][2], acc[2 * ks][3]);
      a[2] = pack_bf16(acc[2 * ks + 1][0], acc[2 * ks + 1][1]);
      a[3] = pack_bf16(acc[2 * ks + 1][2], acc[2 * ks + 1][3]);
#pragma unroll
      for (int nb = 0; nb < 8; ++nb) {
        uint32_t b0, b1;
        frag_b(b0, b1, Wt + RS_TILE, 8 * nb, 16 * ks);
        mma16816(o[nb], a, b0, b1);
      }
    }
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      const int c = 8 * nb + 2 * t;
      const float2 b = __ldg(reinterpret_cast<const float2*>(bin2 + c));
      if (i0 < rows) *reinterpret_cast<float2*>(q2 + g0 + (long long)i0 * RS_H + c) = make_float2((o[nb][0] + b.x) * qscale, (o[nb][1] + b.y) * qscale);
      if (i1 < rows) *reinterpret_cast<float2*>(q2 + g0 + (long long)i1 * RS_H + c) = make_float2((o[nb][2] + b.x) * qscale, (o[nb][3] + b.y) * qscale);
    }
  }
#pragma unroll 1
  for (int m = 0; m < 2; ++m) {    // k2, v2 from the encoder features
    float o[8][4];
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) o[nb][0] = o[nb][1] = o[nb][2] = o[nb][3] = 0.f;
    rs_fgemm(o, Fs, Wt + (2 + m) * RS_TILE, 16 * w);
    float* out = m == 0 ? k2 : v2;
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      const int c = 8 * nb + 2 * t;
      const float2 b = __ldg(reinterpret_cast<const float2*>(bin2 + (1 + m) * RS_H + c));
      if (i0 < rows) *reinterpret_cast<float2*>(out + g0 + (long long)i0 * RS_H + c) = make_float2(o[nb][0] + b.x, o[nb][1] + b.y);
      if (i1 < rows) *reinterpret_cast<float2*>(out + g0 + (long long)i1 * RS_H + c) = make_float2(o[nb][2] + b.x, o[nb][3] + b.y);
    }
  }
}

// -------------------------------------------------------------------------------------------------
// mid_bwd_small_kernel == mid_bwd_kernel (kernels_bwd.cuh): adjoint of the decoder's self-attention out-projection and of the
// cross-attention in-projection (q from the self-attention output a, k/v from the encoder features), H == 64, bf16 mode.  Every
// operand except da is staged in the prologue; da is the one tile the wgrad warps wait for.
// -------------------------------------------------------------------------------------------------
struct MidBwdSmallSmem {
  static constexpr int W = 0;                        // Wq2, Wk2, Wv2, Wo1 row-major
  static constexpr int T = 4 * RS_TILE;              // dq2 * s
  static constexpr int A = T + RS_TILE;              // a
  static constexpr int K = A + RS_TILE;              // dk2
  static constexpr int V = K + RS_TILE;              // dv2
  static constexpr int F = V + RS_TILE;              // feats
  static constexpr int C = F + RS_TILE;              // ctx1
  static constexpr int DA = C + RS_TILE;             // grad wrt a
  static constexpr size_t TOTAL_BYTES = (size_t)(DA + RS_TILE) * 2;
};
constexpr int RS_BAR_DA = 1;                         // mid_bwd_small_kernel: da tile complete

__global__ void __launch_bounds__(RS_BWD_NT, 2) mid_bwd_small_kernel(MidBwdArgs p) {
  using SM = MidBwdSmallSmem;
  extern __shared__ __align__(16) uint8_t rs_raw[];
  __nv_bfloat16* hb = reinterpret_cast<__nv_bfloat16*>(rs_raw);
  __nv_bfloat16* Wt = hb + SM::W;
  __nv_bfloat16* T = hb + SM::T;
  __nv_bfloat16* As = hb + SM::A;
  __nv_bfloat16* Kt = hb + SM::K;
  __nv_bfloat16* Vt = hb + SM::V;
  __nv_bfloat16* Fs = hb + SM::F;
  __nv_bfloat16* Cs = hb + SM::C;
  __nv_bfloat16* DAs = hb + SM::DA;
  const int row0 = blockIdx.x * 64;
  const int rows = min(64, p.M - row0);
  const long long g0 = (long long)row0 * RS_H;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * w + g, i1 = i0 + 8;
  {
    const float* const src[3] = {p.dq2 + g0, p.dk2 + g0, p.dv2 + g0};
    const long long ld[3] = {RS_H, RS_H, RS_H};
    const int nr[3] = {rows, rows, rows};
    const float sc[3] = {p.qscale, 1.f, 1.f};
    __nv_bfloat16* const d[3] = {T, Kt, Vt};
    __nv_bfloat16* const dT[3] = {nullptr, nullptr, nullptr};
    float* const dF[3] = {nullptr, nullptr, nullptr};
    rs_load<3, RS_BWD_NT>(src, ld, nr, sc, d, dT, dF);
  }
  {
    const float* const src[4] = {p.Win2, p.Win2 + RS_H * RS_H, p.Win2 + 2 * RS_H * RS_H, p.Wo1};
    const long long ld[4] = {RS_H, RS_H, RS_H, RS_H};
    const int nr[4] = {64, 64, 64, 64};
    const float sc[4] = {1.f, 1.f, 1.f, 1.f};
    __nv_bfloat16* const d[4] = {Wt, Wt + RS_TILE, Wt + 2 * RS_TILE, Wt + 3 * RS_TILE};
    __nv_bfloat16* const dT[4] = {nullptr, nullptr, nullptr, nullptr};
    float* const dF[4] = {nullptr, nullptr, nullptr, nullptr};
    rs_load<4, RS_BWD_NT>(src, ld, nr, sc, d, dT, dF);
  }
  {
    const float* const src[3] = {p.a + g0, p.feats + g0, p.ctx1 + g0};
    const long long ld[3] = {RS_H, RS_H, RS_H};
    const int nr[3] = {rows, rows, rows};
    const float sc[3] = {1.f, 1.f, 1.f};
    __nv_bfloat16* const d[3] = {As, Fs, Cs};
    __nv_bfloat16* const dT[3] = {nullptr, nullptr, nullptr};
    float* const dF[3] = {nullptr, nullptr, nullptr};
    rs_load<3, RS_BWD_NT>(src, ld, nr, sc, d, dT, dF);
  }
  __syncthreads();
  if (w >= 4) {
    // ---- wgrad warps: dWq2 += (dq2 s)^T a ; dWk2 += dk2^T feats ; dWv2 += dv2^T feats ; dWo1 += da^T ctx1 (and the bias sums)
    rs_wgrad_rm(T, As, p.gWin2, p.gbin2, w - 4);
    rs_wgrad_rm(Kt, Fs, p.gWin2 + (long long)RS_H * RS_H, p.gbin2 + RS_H, w - 4);
    rs_wgrad_rm(Vt, Fs, p.gWin2 + 2ll * RS_H * RS_H, p.gbin2 + 2 * RS_H, w - 4);
    rs_bar_sync(RS_BAR_DA, RS_BWD_NT);
    rs_wgrad_rm(DAs, Cs, p.gWo1, p.gbo1, w - 4);
    return;
  }
  // 1. q projection of the cross attention: da = (dq2 s) Wq2
  float D[8][4];
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) D[nb][0] = D[nb][1] = D[nb][2] = D[nb][3] = 0.f;
  rs_dgrad(D, T, Wt, 16 * w);
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {          // da as a bf16 tile (operand of step 3 and of dWo1), own rows only
    *reinterpret_cast<uint32_t*>(DAs + i0 * RS_LD + 8 * nb + 2 * t) = pack_bf16(D[nb][0], D[nb][1]);
    *reinterpret_cast<uint32_t*>(DAs + i1 * RS_LD + 8 * nb + 2 * t) = pack_bf16(D[nb][2], D[nb][3]);
  }
  __syncwarp();                             // step 3 reads this warp's rows of da through ldmatrix
  rs_bar_arrive(RS_BAR_DA);
  // 2. k/v projections of the encoder features: dfeats += dk2 Wk2 + dv2 Wv2
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) D[nb][0] = D[nb][1] = D[nb][2] = D[nb][3] = 0.f;
  rs_dgrad(D, Kt, Wt + RS_TILE, 16 * w);
  rs_dgrad(D, Vt, Wt + 2 * RS_TILE, 16 * w);
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    if (i0 < rows) { float2* d = reinterpret_cast<float2*>(p.dfeats + g0 + (long long)i0 * RS_H + c); const float2 o = *d; *d = make_float2(o.x + D[nb][0], o.y + D[nb][1]); }
    if (i1 < rows) { float2* d = reinterpret_cast<float2*>(p.dfeats + g0 + (long long)i1 * RS_H + c); const float2 o = *d; *d = make_float2(o.x + D[nb][2], o.y + D[nb][3]); }
  }
  // 3. self-attention out-projection: dctx1 = da Wo1
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) D[nb][0] = D[nb][1] = D[nb][2] = D[nb][3] = 0.f;
  rs_dgrad(D, DAs, Wt + 3 * RS_TILE, 16 * w);
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    const int c = 8 * nb + 2 * t;
    if (i0 < rows) *reinterpret_cast<float2*>(p.dctx1 + g0 + (long long)i0 * RS_H + c) = make_float2(D[nb][0], D[nb][1]);
    if (i1 < rows) *reinterpret_cast<float2*>(p.dctx1 + g0 + (long long)i1 * RS_H + c) = make_float2(D[nb][2], D[nb][3]);
  }
}

// -------------------------------------------------------------------------------------------------
// Attention fused into the projection kernels, for sequences of 33 .. 64 positions: one 256-thread CTA per sequence, so the rows of
// its tile are all the keys its queries see.  Warp group g (warps 4g .. 4g+3, 16 rows each) runs the attention of the heads in column
// half g of the model (one head: group 0 alone); the per-head arithmetic is as_fwd_head / as_bwd_head, the body of the separate
// kernels, so every row's results are those of the two-launch path.
// -------------------------------------------------------------------------------------------------
// Columns 32 grp .. 32 grp + 31 of one projection of the fused kernels below: acc (4 column blocks of this warp's rows i0 / i1) plus
// bias, times sc -> fp32 rows of `out` below L and the bf16 tile T the attention reads (rows >= L: zero, as as_load writes them)
__device__ __forceinline__ void rs_store_half(float* __restrict__ out, __nv_bfloat16* __restrict__ T, const float (&acc)[4][4],
                                              const float* __restrict__ bias, float sc, int grp, int i0, int i1, int L, int t) {
  const bool v0 = i0 < L, v1 = i1 < L;
#pragma unroll
  for (int nb = 0; nb < 4; ++nb) {
    const int c = 32 * grp + 8 * nb + 2 * t;
    const float2 bb = __ldg(reinterpret_cast<const float2*>(bias + c));
    const float2 y0 = make_float2((acc[nb][0] + bb.x) * sc, (acc[nb][1] + bb.y) * sc);
    const float2 y1 = make_float2((acc[nb][2] + bb.x) * sc, (acc[nb][3] + bb.y) * sc);
    if (v0) *reinterpret_cast<float2*>(out + (long long)i0 * RS_H + c) = y0;
    if (v1) *reinterpret_cast<float2*>(out + (long long)i1 * RS_H + c) = y1;
    *reinterpret_cast<uint32_t*>(T + i0 * RS_LD + c) = v0 ? pack_bf16(y0.x, y0.y) : 0u;
    *reinterpret_cast<uint32_t*>(T + i1 * RS_LD + c) = v1 ? pack_bf16(y1.x, y1.y) : 0u;
  }
}

// acc[nb] += A[rows 16 wl ..][k] * W[32 grp + 8 nb ..][k]^T: column half grp of rs_fgemm, every column accumulated in rs_fgemm's order
__device__ __forceinline__ void rs_fgemm_half(float (&acc)[4][4], const __nv_bfloat16* __restrict__ A, const __nv_bfloat16* __restrict__ W,
                                              int wl, int grp) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t a[4];
    frag_a(a, A, 16 * wl, 16 * ks);
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
      uint32_t b0, b1;
      frag_b(b0, b1, W, 32 * grp + 8 * nb, 16 * ks);
      mma16816(acc[nb], a, b0, b1);
    }
  }
}

// attention of the heads in column half grp (one head: group 0 alone) from the tiles Qs, Ks, Vs of sequence b (first row row0)
template <int HD>
__device__ __forceinline__ void rs_attn_half(const __nv_bfloat16* Qs, const __nv_bfloat16* Ks, const __nv_bfloat16* Vs, int grp, int wl, int b,
                                             long long row0, int L, int mask_mode, const int* ids, float* ctx, float* lse, const DropDesc& drop) {
  constexpr int NH = RS_H / HD, HPG = NH > 1 ? NH / 2 : 1;       // heads, heads per warp group
  if (NH == 1 && grp == 1) return;
#pragma unroll 1
  for (int hh = 0; hh < HPG; ++hh) {
    const int h = grp * HPG + hh, c0 = h * HD;
    as_fwd_head<HD, RS_LD>(Qs + c0, Ks + c0, Vs + c0, wl, L, RS_H, mask_mode, ids + row0, ctx + row0 * RS_H + c0,
                           lse ? lse + ((long long)b * NH + h) * L : nullptr, drop, drop.base + ((unsigned long long)b * NH + h) * L);
  }
}

struct RsAttnFwdArgs {
  const float* x; const float* ln_g; const float* ln_b; const float* Win; const float* bin;
  float* q; float* k; float* v; float* norm_out;          // norm_out (nullable): LN(x), the decoder's residual d
  float* ctx; float* lse; const int* ids;
  int L, mask_mode, kv_from_norm; float qscale; DropDesc drop;
};

// pre_attn_fwd_small_kernel<HD> == pre_fwd_small_kernel + attn_small_fwd_kernel<HD>.  q, k, v are stored in fp32 (the backward reads
// them) and, rounded once, as the bf16 tiles the attention reads: the values attn_small_fwd_kernel loads.
struct PreAttnFwdSmem {
  static constexpr int W = 0, X = 3 * RS_TILE, N = X + RS_TILE, Q = N + RS_TILE, K = Q + RS_TILE, V = K + RS_TILE, HALF_END = V + RS_TILE;
  static constexpr size_t XF_BYTES = (size_t)HALF_END * 2;
  static constexpr size_t TOTAL_BYTES = XF_BYTES + (size_t)64 * RS_LF * 4;
};

template <int HD>
__global__ void __launch_bounds__(RS_BWD_NT, 2) pre_attn_fwd_small_kernel(RsAttnFwdArgs p) {
  using SM = PreAttnFwdSmem;
  extern __shared__ __align__(16) uint8_t rs_raw[];
  __nv_bfloat16* hb = reinterpret_cast<__nv_bfloat16*>(rs_raw);
  __nv_bfloat16* Wt = hb + SM::W;
  __nv_bfloat16* Xb = hb + SM::X;
  __nv_bfloat16* Nb = hb + SM::N;
  __nv_bfloat16* Qs = hb + SM::Q;
  __nv_bfloat16* Ks = hb + SM::K;
  __nv_bfloat16* Vs = hb + SM::V;
  float* Xf = reinterpret_cast<float*>(rs_raw + SM::XF_BYTES);
  const int b = blockIdx.x, L = p.L;
  const long long row0 = (long long)b * L;
  const int w = threadIdx.x >> 5, grp = w >> 2, wl = w & 3, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * wl + g, i1 = i0 + 8;
  {
    const float* const src[1] = {p.x + row0 * RS_H};
    const long long ld[1] = {RS_H};
    const int nr[1] = {L};
    const float sc[1] = {1.f};
    __nv_bfloat16* const d[1] = {Xb};
    __nv_bfloat16* const dT[1] = {nullptr};
    float* const dF[1] = {Xf};
    rs_load<1, RS_BWD_NT>(src, ld, nr, sc, d, dT, dF);
  }
  {
    const float* const src[3] = {p.Win, p.Win + RS_H * RS_H, p.Win + 2 * RS_H * RS_H};
    const long long ld[3] = {RS_H, RS_H, RS_H};
    const int nr[3] = {64, 64, 64};
    const float sc[3] = {1.f, 1.f, 1.f};
    __nv_bfloat16* const d[3] = {Wt, Wt + RS_TILE, Wt + 2 * RS_TILE};
    __nv_bfloat16* const dT[3] = {nullptr, nullptr, nullptr};
    float* const dF[3] = {nullptr, nullptr, nullptr};
    rs_load<3, RS_BWD_NT>(src, ld, nr, sc, d, dT, dF);
  }
  __syncthreads();
  if (threadIdx.x < AS_NT) rs_ln_tile(Xf, p.ln_g, p.ln_b, Nb, p.norm_out, row0, L);
  __syncthreads();
  // packed in-projection, columns 32 grp .. 32 grp + 31 of q, k and v
  const __nv_bfloat16* Akv = p.kv_from_norm ? Nb : Xb;
#pragma unroll 1
  for (int m = 0; m < 3; ++m) {
    float acc[4][4];
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) acc[nb][0] = acc[nb][1] = acc[nb][2] = acc[nb][3] = 0.f;
    rs_fgemm_half(acc, m == 0 ? Nb : Akv, Wt + m * RS_TILE, wl, grp);
    rs_store_half((m == 0 ? p.q : m == 1 ? p.k : p.v) + row0 * RS_H, m == 0 ? Qs : m == 1 ? Ks : Vs, acc, p.bin + m * RS_H,
                  m == 0 ? p.qscale : 1.f, grp, i0, i1, L, t);
  }
  __syncthreads();
  rs_attn_half<HD>(Qs, Ks, Vs, grp, wl, b, row0, L, p.mask_mode, p.ids, p.ctx, p.lse, p.drop);
}

// mid_attn_fwd_small_kernel<HD> == mid_fwd_small_kernel + attn_small_fwd_kernel<HD> (the decoder's cross attention).  Every warp
// computes the self-attention out-projection a = ctx1 Wo1^T + bo1 of its 16 rows in full (both groups: a is the A operand of the q
// projection and stays in fragments, as in mid_fwd_small_kernel); group g then computes column half g of q2, k2, v2 and the
// attention of the heads in that half.
struct RsMidAttnArgs {
  const float* ctx1; const float* feats; const float* Wo1; const float* bo1; const float* Win2; const float* bin2;
  float* a; float* q2; float* k2; float* v2; float* ctx2; float* lse2; const int* ids;
  int L, mask_mode; float qscale; DropDesc drop;
};
struct MidAttnFwdSmem {
  // Wo1, Wq2, Wk2, Wv2 | ctx1 | feats | q2 | k2 | v2
  static constexpr int W = 0, C = 4 * RS_TILE, F = C + RS_TILE, Q = F + RS_TILE, K = Q + RS_TILE, V = K + RS_TILE;
  static constexpr size_t TOTAL_BYTES = (size_t)(V + RS_TILE) * 2;
};

template <int HD>
__global__ void __launch_bounds__(RS_BWD_NT, 2) mid_attn_fwd_small_kernel(RsMidAttnArgs p) {
  using SM = MidAttnFwdSmem;
  extern __shared__ __align__(16) uint8_t rs_raw[];
  __nv_bfloat16* hb = reinterpret_cast<__nv_bfloat16*>(rs_raw);
  __nv_bfloat16* Wt = hb + SM::W;
  __nv_bfloat16* Cs = hb + SM::C;
  __nv_bfloat16* Fs = hb + SM::F;
  __nv_bfloat16* Qs = hb + SM::Q;
  __nv_bfloat16* Ks = hb + SM::K;
  __nv_bfloat16* Vs = hb + SM::V;
  const int b = blockIdx.x, L = p.L;
  const long long row0 = (long long)b * L, g0 = row0 * RS_H;
  const int w = threadIdx.x >> 5, grp = w >> 2, wl = w & 3, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * wl + g, i1 = i0 + 8;
  {
    const float* const src[2] = {p.ctx1 + g0, p.feats + g0};
    const long long ld[2] = {RS_H, RS_H};
    const int nr[2] = {L, L};
    const float sc[2] = {1.f, 1.f};
    __nv_bfloat16* const d[2] = {Cs, Fs};
    __nv_bfloat16* const dT[2] = {nullptr, nullptr};
    float* const dF[2] = {nullptr, nullptr};
    rs_load<2, RS_BWD_NT>(src, ld, nr, sc, d, dT, dF);
  }
  {
    const float* const src[4] = {p.Wo1, p.Win2, p.Win2 + RS_H * RS_H, p.Win2 + 2 * RS_H * RS_H};
    const long long ld[4] = {RS_H, RS_H, RS_H, RS_H};
    const int nr[4] = {64, 64, 64, 64};
    const float sc[4] = {1.f, 1.f, 1.f, 1.f};
    __nv_bfloat16* const d[4] = {Wt, Wt + RS_TILE, Wt + 2 * RS_TILE, Wt + 3 * RS_TILE};
    __nv_bfloat16* const dT[4] = {nullptr, nullptr, nullptr, nullptr};
    float* const dF[4] = {nullptr, nullptr, nullptr, nullptr};
    rs_load<4, RS_BWD_NT>(src, ld, nr, sc, d, dT, dF);
  }
  __syncthreads();
  {
    float acc[8][4];
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) acc[nb][0] = acc[nb][1] = acc[nb][2] = acc[nb][3] = 0.f;
    rs_fgemm(acc, Cs, Wt, 16 * wl);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      const int c = 8 * nb + 2 * t;
      const float2 bb = __ldg(reinterpret_cast<const float2*>(p.bo1 + c));
      acc[nb][0] += bb.x; acc[nb][1] += bb.y; acc[nb][2] += bb.x; acc[nb][3] += bb.y;
      if (p.a && grp == 0) {
        if (i0 < L) *reinterpret_cast<float2*>(p.a + g0 + (long long)i0 * RS_H + c) = make_float2(acc[nb][0], acc[nb][1]);
        if (i1 < L) *reinterpret_cast<float2*>(p.a + g0 + (long long)i1 * RS_H + c) = make_float2(acc[nb][2], acc[nb][3]);
      }
    }
    float o[4][4];     // q2 = (a Wq2^T + bq2) s, column half grp, with a taken from the fragments
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) o[nb][0] = o[nb][1] = o[nb][2] = o[nb][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t a[4];
      a[0] = pack_bf16(acc[2 * ks][0], acc[2 * ks][1]);
      a[1] = pack_bf16(acc[2 * ks][2], acc[2 * ks][3]);
      a[2] = pack_bf16(acc[2 * ks + 1][0], acc[2 * ks + 1][1]);
      a[3] = pack_bf16(acc[2 * ks + 1][2], acc[2 * ks + 1][3]);
#pragma unroll
      for (int nb = 0; nb < 4; ++nb) {
        uint32_t b0, b1;
        frag_b(b0, b1, Wt + RS_TILE, 32 * grp + 8 * nb, 16 * ks);
        mma16816(o[nb], a, b0, b1);
      }
    }
    rs_store_half(p.q2 + g0, Qs, o, p.bin2, p.qscale, grp, i0, i1, L, t);
  }
#pragma unroll 1
  for (int m = 0; m < 2; ++m) {    // k2, v2 from the encoder features
    float acc[4][4];
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) acc[nb][0] = acc[nb][1] = acc[nb][2] = acc[nb][3] = 0.f;
    rs_fgemm_half(acc, Fs, Wt + (2 + m) * RS_TILE, wl, grp);
    rs_store_half((m == 0 ? p.k2 : p.v2) + g0, m == 0 ? Ks : Vs, acc, p.bin2 + (1 + m) * RS_H, 1.f, grp, i0, i1, L, t);
  }
  __syncthreads();
  rs_attn_half<HD>(Qs, Ks, Vs, grp, wl, b, row0, L, p.mask_mode, p.ids, p.ctx2, p.lse2, p.drop);
}

// attn_pre_bwd_small_kernel<HD> == attn_small_bwd_kernel<HD> + pre_bwd_small2_kernel, for two or four heads (one head of 64 columns
// needs 160 registers in the attention adjoint alone: that would cost the second CTA per SM).  dq (scaled by qscale), dk and dv go
// from the accumulator fragments straight into the bf16 tiles pre_bwd_small2_kernel stages, rounded as it rounds them; the fp32 dq,
// dk, dv buffers are not written.  The attention operands alias tiles that are dead by the time they are needed: dk and dv overwrite
// k and v (read only before the group barrier inside as_bwd_head), LN(x) and x overwrite q and dctx after the attention.
struct RsAttnBwdArgs {
  PreBwdArgs pre;
  const float* q; const float* k; const float* v; const float* dctx; const float* lse; const int* ids;
  int L, mask_mode; DropDesc drop;
};
struct AttnPreBwdSmem {
  // Wq, Wk, Wv | dq s | k -> dk | v -> dv | q -> LN(x) | dctx -> x | dS, P~ of group 0 | dS, P~ of group 1
  static constexpr int W = 0, TQ = 3 * RS_TILE, TK = TQ + RS_TILE, TV = TK + RS_TILE, N = TV + RS_TILE, X = N + RS_TILE, S = X + RS_TILE;
  static constexpr size_t TOTAL_BYTES = (size_t)(S + 4 * RS_TILE) * 2;
};

template <int HD>
__global__ void __launch_bounds__(RS_BWD_NT, 2) attn_pre_bwd_small_kernel(RsAttnBwdArgs a) {
  using SM = AttnPreBwdSmem;
  constexpr int NH = RS_H / HD, HPG = NH / 2;
  static_assert(NH == 2 || NH == 4, "one head per warp group or two");
  extern __shared__ __align__(16) uint8_t rs_raw[];
  __nv_bfloat16* hb = reinterpret_cast<__nv_bfloat16*>(rs_raw);
  __nv_bfloat16* Wt = hb + SM::W;
  __nv_bfloat16* Tq = hb + SM::TQ;
  __nv_bfloat16* Tk = hb + SM::TK;
  __nv_bfloat16* Tv = hb + SM::TV;
  __nv_bfloat16* Nb = hb + SM::N;
  __nv_bfloat16* Xb = hb + SM::X;
  const int b = blockIdx.x, L = a.L;
  const long long row0 = (long long)b * L, g0 = row0 * RS_H;
  const int w = threadIdx.x >> 5, grp = w >> 2, wl = w & 3, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int i0 = 16 * wl + g, i1 = i0 + 8;
  const bool v0 = i0 < L, v1 = i1 < L;
  const float* lse_g = a.lse + ((long long)b * NH + grp * HPG) * L;     // lse of the group's heads, [HPG][L]
  float ls0 = v0 ? lse_g[i0] : 0.f, ls1 = v1 ? lse_g[i1] : 0.f;          // issued early: consumed after the first product
  if (threadIdx.x < 2 * L)                    // the block input, read after the attention: toward L2 now
    asm volatile("prefetch.global.L2 [%0];" ::"l"(a.pre.x + g0 + 32 * threadIdx.x));
  {   // q, k, v, dctx into the tiles of LN(x), dk, dv, x
    const float* const src[4] = {a.q + g0, a.k + g0, a.v + g0, a.dctx + g0};
    const long long ld[4] = {RS_H, RS_H, RS_H, RS_H};
    const int nr[4] = {L, L, L, L};
    const float sc[4] = {1.f, 1.f, 1.f, 1.f};
    __nv_bfloat16* const d[4] = {Nb, Tk, Tv, Xb};
    __nv_bfloat16* const dT[4] = {nullptr, nullptr, nullptr, nullptr};
    float* const dF[4] = {nullptr, nullptr, nullptr, nullptr};
    rs_load<4, RS_BWD_NT>(src, ld, nr, sc, d, dT, dF);
  }
  {
    const float* const src[3] = {a.pre.Win, a.pre.Win + RS_H * RS_H, a.pre.Win + 2 * RS_H * RS_H};
    const long long ld[3] = {RS_H, RS_H, RS_H};
    const int nr[3] = {64, 64, 64};
    const float sc[3] = {1.f, 1.f, 1.f};
    __nv_bfloat16* const d[3] = {Wt, Wt + RS_TILE, Wt + 2 * RS_TILE};
    __nv_bfloat16* const dT[3] = {nullptr, nullptr, nullptr};
    float* const dF[3] = {nullptr, nullptr, nullptr};
    rs_load<3, RS_BWD_NT>(src, ld, nr, sc, d, dT, dF);
  }
  __syncthreads();
  __nv_bfloat16* dSt = hb + SM::S + 2 * grp * RS_TILE;
  __nv_bfloat16* Pt = dSt + RS_TILE;
  const float qscale = a.pre.qscale;
  const auto group_sync = [grp] {             // the four warps of this group (immediate barrier ids)
    if (grp) asm volatile("bar.sync 2, 128;" ::: "memory");
    else asm volatile("bar.sync 1, 128;" ::: "memory");
  };
#pragma unroll 1
  for (int hh = 0; hh < HPG; ++hh) {
    const int h = grp * HPG + hh, c0 = h * HD;
    if (hh) {
      group_sync();                           // the previous head's key-side products have read dS and P~
      ls0 = v0 ? lse_g[hh * L + i0] : 0.f;
      ls1 = v1 ? lse_g[hh * L + i1] : 0.f;
    }
    as_bwd_head<HD, RS_LD>(Nb + c0, Tk + c0, Tv + c0, Xb + c0, dSt, Pt, wl, L, a.mask_mode, a.ids + row0, ls0, ls1, a.drop,
                           a.drop.base + ((unsigned long long)b * NH + h) * L,
                           [&](int which, const float (&o)[HD / 8][4]) {
                             __nv_bfloat16* T = (which == 0 ? Tq : which == 1 ? Tk : Tv) + c0;
                             const float sc = which == 0 ? qscale : 1.f;
#pragma unroll
                             for (int db = 0; db < HD / 8; ++db) {
                               *reinterpret_cast<uint32_t*>(T + i0 * RS_LD + 8 * db + 2 * t) = v0 ? pack_bf16(o[db][0] * sc, o[db][1] * sc) : 0u;
                               *reinterpret_cast<uint32_t*>(T + i1 * RS_LD + 8 * db + 2 * t) = v1 ? pack_bf16(o[db][2] * sc, o[db][3] * sc) : 0u;
                             }
                           },
                           group_sync);
  }
  float Xf[8][4];                             // the block input, issued before the barrier that waits for the other group's heads
  if (w < 4) frag_load(Xf, a.pre.x + g0, i0, i1, v0, v1, t);
  __syncthreads();                            // dq s, dk, dv complete; the q and dctx tiles are free
  pre_bwd_small_tail(a.pre, Xf, Wt, Tq, Tk, Tv, Xb, Nb, row0, L);
}

}  // namespace adt
