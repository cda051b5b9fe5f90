// Generic row-tile ops used to compose the post-LN backbones (Bert4Rec-ADT, /root/reference/bert4rec/model/modules.py):
// linear fwd/bwd with fused bias/activation, dropout+residual+LayerNorm fwd/bwd, activation adjoint, softmax
// cross-entropy over logits rows, small-table embedding gradients.  Same building blocks as the SASRec kernels.
#pragma once
#include "common.cuh"
#include "kernels_bwd.cuh"

namespace adt {

__device__ __forceinline__ float gelu_f(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_grad(float x) {
  return 0.5f * (1.f + erff(x * 0.70710678118654752f)) + x * 0.3989422804014327f * expf(-0.5f * x * x);
}
// act codes: 0 none, 1 relu, 2 gelu (erf), 3 elu, 4 elu + 1 (the covariance stream of STOSA, stosa/modules.py:232-234)
__device__ __forceinline__ float act_f(float x, int act) {
  return act == 1 ? fmaxf(x, 0.f) : act == 2 ? gelu_f(x) : act == 3 ? (x > 0.f ? x : expm1f(x)) : act == 4 ? (x > 0.f ? x : expm1f(x)) + 1.f : x;
}
__device__ __forceinline__ float act_g(float x, int act) {
  return act == 1 ? (x > 0.f ? 1.f : 0.f) : act == 2 ? gelu_grad(x) : act >= 3 ? (x > 0.f ? 1.f : expf(x)) : 1.f;
}

// y = act((x W^T + b) * scale) ; optional pre-activation copy.  x [M,K] row-major, W [N,K] (nn.Linear), y [M,N].
struct LinearFwdArgs {
  const float* x; const float* W; const float* b; float* y; float* pre;
  int M, K, N, act; float scale; int ldy;
};
template <int TM, bool MMA>
__global__ void __launch_bounds__(NT) linear_fwd_kernel(LinearFwdArgs p) {
  extern __shared__ __align__(16) float smem[];
  const int ld = p.K + tile_pad<MMA>();
  float* Xs = smem;
  float* Ws = Xs + TM * ld;
  const int row0 = blockIdx.x * TM;
  __shared__ WStreamState wst;
  if (threadIdx.x == 0) {
    wst.g[0] = GemmDesc{p.W, p.K, p.N, p.K, 0};
    wst.ng = 1;
  }
  __syncthreads();
  WStream<WS_NST, MMA> ws;
  ws.start(&wst, Ws);
  load_tile<TM>(Xs, ld, p.x, p.K, 0, p.K, row0, p.M);
  tile_sync();
  const bool vec = ((p.N | p.ldy) & 3) == 0;     // output width / stride not a multiple of 4 -> scalar epilogue
  gemm_stream<TM, false, WS_NST, MMA>(Xs, ld, ws, 0, [&](int, int r, int col, float4 a) {
    if (row0 + r >= p.M) return;
    const long long o = (long long)(row0 + r) * p.ldy + col;
    if (vec) {
      if (p.b) a = f4_add(a, __ldg(reinterpret_cast<const float4*>(p.b + col)));
      a = f4_scale(a, p.scale);
      if (p.pre) st4(p.pre + o, a);
      st4(p.y + o, make_float4(act_f(a.x, p.act), act_f(a.y, p.act), act_f(a.z, p.act), act_f(a.w, p.act)));
    } else {
      const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (col + c < p.N) {
          const float t = (av[c] + (p.b ? p.b[col + c] : 0.f)) * p.scale;
          if (p.pre) p.pre[o + c] = t;
          p.y[o + c] = act_f(t, p.act);
        }
    }
  });
}

// dx = dy W (optionally += into dx) ; gW += dy^T x ; gb += colsum(dy).   dy [M,N], x [M,K], W [N,K].
struct LinearBwdArgs {
  const float* x; const float* W; const float* dy; float* dx; float* gW; float* gb;
  int M, K, N, accumulate_dx; float scale; int lddy;
};
template <int TM, bool MMA>
__global__ void __launch_bounds__(NT) linear_bwd_kernel(LinearBwdArgs p) {
  extern __shared__ __align__(16) float smem[];
  const int N4 = (p.N + 3) & ~3;
  const int ldx = p.K + tile_pad<MMA>(), ldy = N4 + tile_pad<MMA>();
  float* Xs = smem;
  float* Ys = Xs + TM * ldx;
  float* Ws = Ys + TM * ldy;
  const int row0 = blockIdx.x * TM;
  const int rows = min(TM, p.M - row0);
  __shared__ WStreamState wst;
  if (threadIdx.x == 0) {
    wst.g[0] = GemmDesc{p.W, p.K, p.K, p.N, 1};
    wst.ng = p.dx ? 1 : 0;
  }
  __syncthreads();
  WStream<WS_NST, MMA> ws;
  ws.start(&wst, Ws);
  if (p.gW) load_tile<TM>(Xs, ldx, p.x, p.K, 0, p.K, row0, p.M);
  if (((p.N | p.lddy) & 3) == 0) {
    tile_foreach4<TM>(p.N, [&](int r, int c) {
      float4 g = zero4();
      if (row0 + r < p.M) g = f4_scale(ld4(p.dy + (long long)(row0 + r) * p.lddy + c), p.scale);
      st4(Ys + r * ldy + c, g);
    });
  } else {
    for (int i = threadIdx.x; i < TM * N4; i += NT) {
      const int r = i / N4, c = i - r * N4;
      Ys[r * ldy + c] = (row0 + r < p.M && c < p.N) ? p.dy[(long long)(row0 + r) * p.lddy + c] * p.scale : 0.f;
    }
  }
  tile_sync();
  if (p.gW) wgrad_any<MMA, true, TM>(Ys, ldy, p.N, Xs, ldx, p.K, rows, p.gW, p.K);
  if (p.gb) colsum_atomic(Ys, ldy, p.N, rows, p.gb);
  if (p.dx)
    gemm_stream<TM, true, WS_NST, MMA>(Ys, ldy, ws, 0, [&](int, int r, int col, float4 a) {
      if (row0 + r >= p.M) return;
      float* d = p.dx + (long long)(row0 + r) * p.K + col;
      st4(d, p.accumulate_dx ? f4_add(a, ld4(d)) : a);
    });
}

// y = act(x), elementwise
__global__ void __launch_bounds__(256) act_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, long long n4, int act) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    reinterpret_cast<float4*>(y)[i] = make_float4(act_f(v.x, act), act_f(v.y, act), act_f(v.z, act), act_f(v.w, act));
  }
}
// dpre = dy * act'(pre)
__global__ void __launch_bounds__(256) act_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ pre, float* __restrict__ dpre,
                                                      long long n4, int act) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 g = reinterpret_cast<const float4*>(dy)[i], x = reinterpret_cast<const float4*>(pre)[i];
    reinterpret_cast<float4*>(dpre)[i] = make_float4(g.x * act_g(x.x, act), g.y * act_g(x.y, act), g.z * act_g(x.z, act), g.w * act_g(x.w, act));
  }
}

// mode 0 (DropResidualNormalizeLayer, modules.py:104-117): y = LN(dropout(a) + r)
// mode 1 (BertEmbedding, modules.py:42-48)               : y = dropout(LN(a + r))
// Warp per row, U columns per lane (H <= 32 U): U = 8 up to H = 256, 16 up to 512.
struct DrlArgs {
  const float* a; const float* r; const float* gamma; const float* beta; float* y;
  const float* dy; float* da; float* dr; float* ggamma; float* gbeta;
  int M, H, mode; float eps; DropDesc drop;
};
template <int U>
__global__ void __launch_bounds__(NT) drl_fwd_kernel(DrlArgs p) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int H = p.H;
  for (int row = blockIdx.x * (NT / 32) + w; row < p.M; row += gridDim.x * (NT / 32)) {
    float s[U];
    float sum = 0.f;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = l + 32 * u;
      float v = 0.f;
      if (c < H) {
        const long long gi = (long long)row * H + c;
        v = p.a[gi];
        if (p.mode == 0 && p.drop.enabled) v *= drop_mul1(p.drop, p.drop.base + (unsigned long long)gi);
        if (p.r) v += p.r[gi];
      }
      s[u] = v;
      sum += v;
    }
    const float mean = warp_sum(sum) / (float)H;
    float var = 0.f;
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (l + 32 * u < H) { const float t = s[u] - mean; var += t * t; }
    const float rstd = 1.0f / sqrtf(warp_sum(var) / (float)H + p.eps);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = l + 32 * u;
      if (c < H) {
        const long long gi = (long long)row * H + c;
        float o = (s[u] - mean) * rstd * p.gamma[c] + p.beta[c];
        if (p.mode == 1 && p.drop.enabled) o *= drop_mul1(p.drop, p.drop.base + (unsigned long long)gi);
        p.y[gi] = o;
      }
    }
  }
}

template <int U>
__global__ void __launch_bounds__(NT) drl_bwd_kernel(DrlArgs p) {
  __shared__ float red[2 * (NT / 32) * 32 * U];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int H = p.H;
  constexpr int NW = NT / 32;
  float dg[U], db[U];
#pragma unroll
  for (int u = 0; u < U; ++u) dg[u] = db[u] = 0.f;
  for (int row = blockIdx.x * NW + w; row < p.M; row += gridDim.x * NW) {
    float s[U], g[U], m[U];
    float sum = 0.f;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = l + 32 * u;
      float v = 0.f, gg = 0.f, mm = 1.f;
      if (c < H) {
        const long long gi = (long long)row * H + c;
        if (p.drop.enabled) mm = drop_mul1(p.drop, p.drop.base + (unsigned long long)gi);
        v = p.a[gi];
        if (p.mode == 0) v *= mm;
        if (p.r) v += p.r[gi];
        gg = p.dy[gi];
        if (p.mode == 1) gg *= mm;
      }
      s[u] = v; g[u] = gg; m[u] = mm;
      sum += v;
    }
    const float mean = warp_sum(sum) / (float)H;
    float var = 0.f;
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (l + 32 * u < H) { const float t = s[u] - mean; var += t * t; }
    const float rstd = 1.0f / sqrtf(warp_sum(var) / (float)H + p.eps);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = l + 32 * u;
      if (c < H) {
        const float xh = (s[u] - mean) * rstd, gg = g[u] * p.gamma[c];
        s1 += gg; s2 += gg * xh;
        dg[u] += g[u] * xh; db[u] += g[u];
      }
    }
    s1 = warp_sum(s1) / (float)H;
    s2 = warp_sum(s2) / (float)H;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int c = l + 32 * u;
      if (c < H) {
        const long long gi = (long long)row * H + c;
        const float xh = (s[u] - mean) * rstd;
        const float ds = rstd * (g[u] * p.gamma[c] - s1 - xh * s2);
        if (p.da) p.da[gi] = p.mode == 0 ? ds * m[u] : ds;
        if (p.dr) p.dr[gi] = ds;
      }
    }
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int c = l + 32 * u;
    if (c < H) { red[w * H + c] = dg[u]; red[(NW + w) * H + c] = db[u]; }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < H; c += NT) {
    float a = 0.f, b = 0.f;
    for (int i = 0; i < NW; ++i) { a += red[i * H + c]; b += red[(NW + i) * H + c]; }
    atomicAdd(p.ggamma + c, a);
    atomicAdd(p.gbeta + c, b);
  }
}

// s[row] = A[ia[row]] + B[ib[row]] + C[ic[row]]   (BertEmbedding's three lookups, modules.py:43-45); tables may be NULL
__global__ void __launch_bounds__(256) gather3_kernel(const int* __restrict__ ia, const float* __restrict__ A, const int* __restrict__ ib,
                                                      const float* __restrict__ B, const int* __restrict__ ic, const float* __restrict__ C,
                                                      float* __restrict__ s, int M, int H) {
  const int h4 = H >> 2;
  const long long n = (long long)M * h4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int row = (int)(i / h4), c4 = (int)(i - (long long)row * h4);
    float4 o = __ldg(reinterpret_cast<const float4*>(A + (long long)ia[row] * H) + c4);
    if (B) o = f4_add(o, __ldg(reinterpret_cast<const float4*>(B + (long long)ib[row] * H) + c4));
    if (C) o = f4_add(o, __ldg(reinterpret_cast<const float4*>(C + (long long)ic[row] * H) + c4));
    reinterpret_cast<float4*>(s)[i] = o;
  }
}
// table_grad[ids[row]] += dx[row] for ids != padding_idx  (small tables: positions, sentence types)
__global__ void __launch_bounds__(256) small_table_grad_kernel(const int* __restrict__ ids, const float* __restrict__ dx,
                                                               float* __restrict__ g, int M, int H, int padding_idx) {
  const int h4 = H >> 2;
  const long long n = (long long)M * h4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int row = (int)(i / h4), c4 = (int)(i - (long long)row * h4);
    const int id = ids[row];
    if (id == padding_idx) continue;
    atomicAdd(reinterpret_cast<float4*>(g + (long long)id * H) + c4, reinterpret_cast<const float4*>(dx)[i]);
  }
}

// softmax cross-entropy over logits rows [R,V] with integer labels (all rows are valid: the caller gathers them).
// fwd: lse[r], acc += sum_r (lse[r] - logits[r][label[r]]) ; bwd (in place): logits <- (softmax - onehot) * coef
__global__ void __launch_bounds__(NT) softmax_ce_kernel(float* __restrict__ logits, const int* __restrict__ labels, float* __restrict__ lse,
                                                        double* __restrict__ acc, int R, int V, int backward, float coef) {
  __shared__ float redf[NT / 32];
  __shared__ double redd[NT / 32];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  double local = 0.0;
  for (int r = blockIdx.x; r < R; r += gridDim.x) {
    float* row = logits + (long long)r * V;
    const int lab = labels[r];
    if (!backward) {
      float mx = -INFINITY;
      for (int c = threadIdx.x; c < V; c += NT) mx = fmaxf(mx, row[c]);
      mx = warp_max(mx);
      if (l == 0) redf[w] = mx;
      __syncthreads();
      mx = redf[0];
      for (int i = 1; i < NT / 32; ++i) mx = fmaxf(mx, redf[i]);
      __syncthreads();
      float se = 0.f;
      for (int c = threadIdx.x; c < V; c += NT) se += expf(row[c] - mx);
      se = warp_sum(se);
      if (l == 0) redf[w] = se;
      __syncthreads();
      se = 0.f;
      for (int i = 0; i < NT / 32; ++i) se += redf[i];
      __syncthreads();
      const float ls = mx + logf(se);
      if (threadIdx.x == 0) {
        lse[r] = ls;
        local += (double)(ls - row[lab]);
      }
    } else {
      const float ls = lse[r];
      for (int c = threadIdx.x; c < V; c += NT) row[c] = (expf(row[c] - ls) - (c == lab ? 1.f : 0.f)) * coef;
    }
  }
  if (!backward && acc) cta_accumulate(local, acc, redd);
}

}  // namespace adt
