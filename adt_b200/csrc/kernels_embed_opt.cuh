// Embedding backward (K2: stable radix sort by item id + segmented scatter-add) and the fused
// table/dense optimiser pass (K6).  Reference semantics: torch embedding_dense_backward with padding_idx=0
// for the four lookups of one step (sasrec/model.py:34,53,72,73), main.py:170-173 (||E|| weight decay,
// clip_grad_norm_, Adam).
#pragma once
#include "common.cuh"
#include "kernels_bwd.cuh"

namespace adt {

constexpr int SORT_WCH = 512;   // sorted-array elements owned by one warp per radix pass

// key/value of logical element e of the concatenated lookup list: src = e / M (0 seq, 1 dec, 2 pos, 3 neg)
struct SortSrc {
  const int* ids[4];
  int M;
};

template <bool FIRST>
__device__ __forceinline__ int sort_key(const SortSrc& s, const int* keys_in, int e) {
  if (FIRST) {
    const int src = e / s.M;
    return s.ids[src][e - src * s.M];
  }
  return keys_in[e];
}

template <bool FIRST>
__global__ void __launch_bounds__(256) radix_hist_kernel(SortSrc s, const int* __restrict__ keys_in, int N, int shift,
                                                         int* __restrict__ hist, int nW) {
  __shared__ int cnt[8][256];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int gw = blockIdx.x * 8 + w;
  for (int d = l; d < 256; d += 32) cnt[w][d] = 0;
  __syncwarp();
  if (gw < nW) {
    const int end = min(N, (gw + 1) * SORT_WCH);
    for (int e = gw * SORT_WCH + l; e < end; e += 32) atomicAdd(&cnt[w][(sort_key<FIRST>(s, keys_in, e) >> shift) & 255], 1);
    __syncwarp();
    for (int d = l; d < 256; d += 32) hist[d * nW + gw] = cnt[w][d];
  }
}

// in-place exclusive scan of n ints, single CTA of 1024 threads, coalesced tiles of 4096 with a running carry
__global__ void __launch_bounds__(1024) exclusive_scan_kernel(int* __restrict__ data, int n) {
  __shared__ int wsum[32];
  __shared__ int carry_s;
  const int l = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 4096) {
    const int i0 = base + 4 * threadIdx.x;
    int v[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) v[c] = (i0 + c < n) ? data[i0 + c] : 0;
    const int s = v[0] + v[1] + v[2] + v[3];
    int incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (l >= o) incl += t;
    }
    if (l == 31) wsum[w] = incl;
    __syncthreads();
    if (w == 0) {
      int x = wsum[l];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, x, o);
        if (l >= o) x += t;
      }
      wsum[l] = x;
    }
    __syncthreads();
    const int carry = carry_s;
    int run = carry + incl - s + (w > 0 ? wsum[w - 1] : 0);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      if (i0 + c < n) data[i0 + c] = run;
      run += v[c];
    }
    __syncthreads();
    if (threadIdx.x == 1023) carry_s = carry + wsum[31];
    __syncthreads();
  }
}

// large inputs: one 4096-element tile per CTA, local exclusive scan in place + the tile total into tsum[tile]; tsum is then
// scanned by exclusive_scan_kernel (one CTA) and added back by the scatter kernel when it reads its offsets
__global__ void __launch_bounds__(1024) scan_tiles_kernel(int* __restrict__ data, int n, int* __restrict__ tsum) {
  __shared__ int wsum[32];
  const int l = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int i0 = blockIdx.x * 4096 + 4 * threadIdx.x;
  int v[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) v[c] = (i0 + c < n) ? data[i0 + c] : 0;
  const int s = v[0] + v[1] + v[2] + v[3];
  int incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (l >= o) incl += t;
  }
  if (l == 31) wsum[w] = incl;
  __syncthreads();
  if (w == 0) {
    int x = wsum[l];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, x, o);
      if (l >= o) x += t;
    }
    wsum[l] = x;
  }
  __syncthreads();
  int run = incl - s + (w > 0 ? wsum[w - 1] : 0);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    if (i0 + c < n) data[i0 + c] = run;
    run += v[c];
  }
  if (threadIdx.x == 1023) tsum[blockIdx.x] = wsum[31];
}

template <bool FIRST>
__global__ void __launch_bounds__(256) radix_scatter_kernel(SortSrc s, const int* __restrict__ keys_in, const int* __restrict__ vals_in,
                                                            int N, int shift, const int* __restrict__ hist, int nW,
                                                            int* __restrict__ keys_out, int* __restrict__ vals_out,
                                                            const int* __restrict__ tsum) {
  __shared__ int off[8][256];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int gw = blockIdx.x * 8 + w;
  if (gw >= nW) return;
  for (int d = l; d < 256; d += 32) {
    const int idx = d * nW + gw;
    off[w][d] = hist[idx] + (tsum ? tsum[idx >> 12] : 0);
  }
  __syncwarp();
  const int end = min(N, (gw + 1) * SORT_WCH);
  for (int base = gw * SORT_WCH; base < end; base += 32) {
    const int e = base + l;
    const bool ok = e < end;
    const int key = ok ? sort_key<FIRST>(s, keys_in, e) : 0;
    const int val = ok ? (FIRST ? e : vals_in[e]) : 0;
    const int d = ok ? ((key >> shift) & 255) : (256 + l);   // invalid lanes never match anybody
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int rank = __popc(peers & ((1u << l) - 1u));
    int dst = 0;
    if (ok) dst = off[w][d] + rank;
    __syncwarp();
    if (ok && rank == 0) off[w][d] += __popc(peers);
    __syncwarp();
    if (ok) {
      keys_out[dst] = key;
      vals_out[dst] = val;
    }
  }
}

// -------------------------------------------------------------------------------------------------
// Segmented scatter-add over the sorted (id, element) list.
// Row value of element e (src = e / M, row = e % M), H floats:
//   src 0/1: dx_{enc,dec}[row] * m_emb(row, :) * sqrt(H)        (adjoint of K1 wrt the table)
//   src 2/3: c{pos,neg}[row] * feats[row]                        (adjoint of the pos/neg logits)
// Phase 1: one warp per 32-entry block of the sorted list, entries summed sequentially in sorted (= original)
//          order; runs fully inside the block are stored to dE, runs crossing a block edge leave a head/tail partial.
// Phase 2: one warp per block that opens a crossing run: tail + following heads, in order.  Deterministic.
// -------------------------------------------------------------------------------------------------
struct ScatterArgs {
  const int* keys; const int* vals; int N; int M; int H;
  const float* dx_enc; const float* dx_dec; const float* feats; const float* cpos; const float* cneg;
  float scale;
  DropDesc drop_enc, drop_dec;
  float* dE; float* head; float* tail; int* has_tail;
};

__device__ __forceinline__ float4 scatter_row4(const ScatterArgs& a, int e, int c) {
  const int src = e / a.M, row = e - src * a.M;
  const long long gi = (long long)row * a.H + c;
  if (src < 2) {
    float4 g = ld4((src == 0 ? a.dx_enc : a.dx_dec) + gi);
    const DropDesc& d = src == 0 ? a.drop_enc : a.drop_dec;
    if (d.enabled) g = f4_mul(g, drop_mul4(d, (d.base + (unsigned long long)gi) >> 2));
    return f4_scale(g, a.scale);
  }
  const float cf = (src == 2 ? a.cpos : a.cneg)[row];
  return f4_scale(ld4(a.feats + gi), cf);
}

// NS = float4 per lane: 1 for H <= 128, 2 for H <= 256, 4 for H <= 512 (phase 2: 2 up to H = 256, else 4)
template <int NS>
__global__ void __launch_bounds__(256) scatter_phase1_kernel(ScatterArgs a) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int g = blockIdx.x * 8 + w;
  const int base = g * 32;
  if (base >= a.N) return;
  const int cnt = min(32, a.N - base);
  const int key_l = l < cnt ? a.keys[base + l] : -1;
  const int val_l = l < cnt ? a.vals[base + l] : 0;
  const int prev_key = base > 0 ? a.keys[base - 1] : -1;
  const int next_key = base + 32 < a.N ? a.keys[base + 32] : -2;
  const int h4 = a.H >> 2;
  float4 acc[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) acc[s] = zero4();
  int run_start = 0;
  bool tail_written = false;
  // entries are consumed strictly in sorted order (deterministic sums), but the row loads of four consecutive entries are
  // issued together so that a warp keeps several independent HBM requests in flight
  for (int j0 = 0; j0 < cnt; j0 += 4) {
    float4 v[4][NS];
    float cf[4];
    // 1. raw loads only (addresses depend on nothing but the shuffled element index): four rows in flight per warp
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = j0 + u;
      const int key = __shfl_sync(0xffffffffu, key_l, j & 31);
      const int e = __shfl_sync(0xffffffffu, val_l, j & 31);
      #pragma unroll
      for (int s = 0; s < NS; ++s) v[u][s] = zero4();
      cf[u] = 0.f;
      if (j < cnt && key != 0) {
        const int src = e / a.M, row = e - src * a.M;
        const float* base = src == 0 ? a.dx_enc : src == 1 ? a.dx_dec : a.feats;
        cf[u] = src < 2 ? a.scale : __ldg((src == 2 ? a.cpos : a.cneg) + row);
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          const int c4 = l + 32 * s;
          if (c4 < h4) v[u][s] = ld4(base + (long long)row * a.H + 4 * c4);
        }
      }
    }
    // 2. dropout mask / coefficient (same operation order as scatter_row4)
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = j0 + u;
      const int e = __shfl_sync(0xffffffffu, val_l, j & 31);
      const int src = e / a.M, row = e - src * a.M;
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const int c4 = l + 32 * s;
        if (src < 2) {
          const DropDesc& d = src == 0 ? a.drop_enc : a.drop_dec;
          if (d.enabled && c4 < h4 && cf[u] != 0.f)
            v[u][s] = f4_mul(v[u][s], drop_mul4(d, (d.base + (unsigned long long)((long long)row * a.H + 4 * c4)) >> 2));
        }
        v[u][s] = f4_scale(v[u][s], cf[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = j0 + u;
      if (j >= cnt) break;
      const int key = __shfl_sync(0xffffffffu, key_l, j);
      const int key_next = j + 1 < cnt ? __shfl_sync(0xffffffffu, key_l, j + 1) : -3;
      if (key == 0) { run_start = j + 1; continue; }   // padding_idx rows get no gradient
      const bool fresh = (j == run_start);
#pragma unroll
      for (int s = 0; s < NS; ++s) acc[s] = fresh ? v[u][s] : f4_add(acc[s], v[u][s]);
      if (j == cnt - 1 || key_next != key) {
        const bool from_before = (run_start == 0) && (key == prev_key);
        const bool goes_after = (j == cnt - 1) && (key == next_key);
        float* dst;
        if (from_before) dst = a.head + (long long)g * a.H;
        else if (goes_after) { dst = a.tail + (long long)g * a.H; tail_written = true; }
        else dst = a.dE + (long long)key * a.H;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          const int c4 = l + 32 * s;
          if (c4 < h4) st4(dst + 4 * c4, acc[s]);
        }
        run_start = j + 1;
      }
    }
  }
  if (l == 0) a.has_tail[g] = tail_written ? 1 : 0;
}

template <int NS>
__global__ void __launch_bounds__(256) scatter_phase2_kernel(ScatterArgs a) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int g = blockIdx.x * 8 + w;
  const int nb = (a.N + 31) / 32;
  if (g >= nb || !a.has_tail[g]) return;
  const int key = a.keys[g * 32 + 31];
  const int h4 = a.H >> 2;
  float4 acc[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    const int c4 = l + 32 * s;
    acc[s] = c4 < h4 ? ld4(a.tail + (long long)g * a.H + 4 * c4) : zero4();
  }
  // the run continues through every following block that starts with the same key: find its length 32 blocks at a time (one
  // key probe per lane), then add the heads strictly in block order with the loads of eight blocks in flight (popular items
  // span hundreds of blocks; a dependent load per block was the whole cost of this kernel)
  int g2 = g + 1;
  while (g2 < nb) {
    const int probe = g2 + l;
    const bool same = probe < nb && a.keys[probe * 32] == key;
    const unsigned ok = __ballot_sync(0xffffffffu, same);
    const int len = ok == 0xffffffffu ? 32 : __ffs(~ok) - 1;     // leading blocks that belong to the run
    for (int b0 = 0; b0 < len; b0 += 8) {
      float4 hv[8][NS];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          const int c4 = l + 32 * s;
          hv[u][s] = (b0 + u < len && c4 < h4) ? ld4(a.head + (long long)(g2 + b0 + u) * a.H + 4 * c4) : zero4();
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (b0 + u < len) {
#pragma unroll
          for (int s = 0; s < NS; ++s) acc[s] = f4_add(acc[s], hv[u][s]);
        }
      }
    }
    if (len < 32) break;
    g2 += 32;
  }
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    const int c4 = l + 32 * s;
    if (c4 < h4) st4(a.dE + (long long)key * a.H + 4 * c4, acc[s]);
  }
}

// -------------------------------------------------------------------------------------------------
// Optimiser pass (K6).
// -------------------------------------------------------------------------------------------------
// out += sum x^2 (double)
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ x, long long n, double* __restrict__ out) {
  __shared__ double red[8];
  double s = 0.0;
  const long long n4 = n >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    s += (double)(v.x * v.x + v.y * v.y) + (double)(v.z * v.z + v.w * v.w);
  }
  if (blockIdx.x == 0)
    for (long long i = (n4 << 2) + threadIdx.x; i < n; i += blockDim.x) s += (double)x[i] * (double)x[i];
  cta_accumulate(s, out, red);
}

// fused: g[i] += (wd / sqrt(*normsq)) * w[i] for i >= decay_off (gradient of wd*||W||_F on the trailing table segment, main.py:170),
// then out += sum g^2 over the whole buffer (clip_grad_norm_'s total norm).  decay_off is a multiple of 4.
__global__ void __launch_bounds__(256) sumsq_decay_kernel(float* __restrict__ g, const float* __restrict__ w, long long n, long long decay_off,
                                                          float wd, const double* __restrict__ normsq, double* __restrict__ out) {
  __shared__ double red[8];
  const float coef = wd / (float)sqrt(*normsq);
  double s = 0.0;
  const long long n4 = n >> 2, d4 = decay_off >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 v = reinterpret_cast<float4*>(g)[i];
    if (i >= d4) {
      const float4 p = reinterpret_cast<const float4*>(w)[i];
      v = make_float4(fmaf(coef, p.x, v.x), fmaf(coef, p.y, v.y), fmaf(coef, p.z, v.z), fmaf(coef, p.w, v.w));
      reinterpret_cast<float4*>(g)[i] = v;
    }
    s += (double)(v.x * v.x + v.y * v.y) + (double)(v.z * v.z + v.w * v.w);
  }
  if (blockIdx.x == 0)
    for (long long i = (n4 << 2) + threadIdx.x; i < n; i += blockDim.x) {
      float x = g[i];
      if (i >= decay_off) { x = fmaf(coef, w[i], x); g[i] = x; }
      s += (double)x * (double)x;
    }
  cta_accumulate(s, out, red);
}

// g += (wd / sqrt(*normsq)) * w     -- gradient of wd*||W||_F  (main.py:170)
__global__ void __launch_bounds__(256) norm_decay_grad_kernel(float* __restrict__ g, const float* __restrict__ w, long long n, float wd,
                                                              const double* __restrict__ normsq) {
  const float coef = wd / (float)sqrt(*normsq);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    g[i] = fmaf(coef, w[i], g[i]);
}

struct AdamArgs {
  float* p; float* g; float* m; float* v; long long n;
  float lr, beta1, beta2, eps, weight_decay;   // weight_decay: classic L2 (evolution.py:111), 0 in main.py
  float bc1, bc2;                              // 1-beta1^t, 1-beta2^t
  float max_norm;                              // <=0: no clipping
  const double* gnormsq;                       // device scalar: sum of squares of ALL grads
  const int* step_dev;                         // optional device step count (overrides bc1/bc2)
  __nv_bfloat16* mirror; long long mirror_n;   // optional bf16 copy of p[0 .. mirror_n) (mirror_n % 4 == 0)
};

// torch.nn.utils.clip_grad_norm_ + torch.optim.Adam (single tensor semantics), fused.  g is left holding the
// clipped gradient (like the reference's .grad after clip_grad_norm_).
__global__ void __launch_bounds__(256) adam_kernel(AdamArgs a) {
  float coef = 1.f;
  if (a.max_norm > 0.f) {
    const float tn = (float)sqrt(*a.gnormsq);
    coef = fminf(a.max_norm / (tn + 1e-6f), 1.0f);
  }
  __shared__ float bc_s[2];
  if (threadIdx.x == 0) {       // one thread evaluates the double-precision bias corrections for the CTA
    float b1 = a.bc1, b2 = a.bc2;
    if (a.step_dev) {
      const double t = (double)*a.step_dev;
      b1 = (float)(1.0 - pow((double)a.beta1, t));
      b2 = (float)(1.0 - pow((double)a.beta2, t));
    }
    bc_s[0] = b1; bc_s[1] = b2;
  }
  __syncthreads();
  const float bc1 = bc_s[0], bc2 = bc_s[1];
  const float step = a.lr / bc1;
  const float isb2 = 1.0f / sqrtf(bc2);
  const float ob1 = 1.f - a.beta1, ob2 = 1.f - a.beta2;
  auto upd = [&](float& g, float& p, float& m, float& v) {
    g *= coef;
    float ge = g;
    if (a.weight_decay != 0.f) ge = fmaf(a.weight_decay, p, ge);
    m = a.beta1 * m + ob1 * ge;
    v = a.beta2 * v + ob2 * ge * ge;
    p = p - step * (m / (sqrtf(v) * isb2 + a.eps));
  };
  // 128-bit streaming body (the four arrays are 16-byte aligned segments of the flat buffers), scalar tail
  const long long n4 = a.n >> 2;
  float4* g4 = reinterpret_cast<float4*>(a.g);
  float4* p4 = reinterpret_cast<float4*>(a.p);
  float4* m4 = reinterpret_cast<float4*>(a.m);
  float4* v4 = reinterpret_cast<float4*>(a.v);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 g = g4[i], p = p4[i], m = m4[i], v = v4[i];
    upd(g.x, p.x, m.x, v.x); upd(g.y, p.y, m.y, v.y); upd(g.z, p.z, m.z, v.z); upd(g.w, p.w, m.w, v.w);
    g4[i] = g; m4[i] = m; v4[i] = v; p4[i] = p;
    if (a.mirror && 4 * i < a.mirror_n) {
      uint2 pk;
      pk.x = pack_bf16(p.x, p.y); pk.y = pack_bf16(p.z, p.w);
      *reinterpret_cast<uint2*>(a.mirror + 4 * i) = pk;
    }
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (long long)gridDim.x * blockDim.x) {
    float g = a.g[i], p = a.p[i], m = a.m[i], v = a.v[i];
    upd(g, p, m, v);
    a.g[i] = g; a.m[i] = m; a.v[i] = v; a.p[i] = p;
  }
}

// ---- segmented Adam: torch.optim.Adam's per-parameter semantics on the flat buffers ------------------------------------
// torch skips parameters whose .grad is None (no moment decay, no weight decay, no step increment) and keeps one step count
// PER PARAMETER (sasrec/evolution.py:111,316-318: the supernet only produces gradients for the 4 active candidate blocks of a
// layer).  Work list: chunk c covers elements [chunk_start[c], chunk_start[c] + chunk_len[c]) of segment chunk_seg[c]; seg_step[s]
// is that segment's own step count (already incremented for this step by adam_seg_step_kernel).
struct AdamSegArgs {
  AdamArgs a;
  const long long* chunk_start; const int* chunk_len; const int* chunk_seg; int n_chunks;
  int* seg_step; const int* active_seg; int n_active;
};

__global__ void adam_seg_step_kernel(AdamSegArgs s) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < s.n_active; i += gridDim.x * blockDim.x) s.seg_step[s.active_seg[i]] += 1;
}

__global__ void __launch_bounds__(256) adam_seg_kernel(AdamSegArgs s) {
  const AdamArgs& a = s.a;
  float coef = 1.f;
  if (a.max_norm > 0.f) {
    const float tn = (float)sqrt(*a.gnormsq);
    coef = fminf(a.max_norm / (tn + 1e-6f), 1.0f);
  }
  const float ob1 = 1.f - a.beta1, ob2 = 1.f - a.beta2;
  for (int c = blockIdx.x; c < s.n_chunks; c += gridDim.x) {
    __shared__ float bc_s[2];
    __syncthreads();
    if (threadIdx.x == 0) {
      const double t = (double)s.seg_step[s.chunk_seg[c]];
      bc_s[0] = (float)(1.0 - pow((double)a.beta1, t));
      bc_s[1] = (float)(1.0 - pow((double)a.beta2, t));
    }
    __syncthreads();
    const float step = a.lr / bc_s[0];
    const float isb2 = 1.0f / sqrtf(bc_s[1]);
    const long long b = s.chunk_start[c];
    const int n = s.chunk_len[c];
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      float g = a.g[b + i] * coef, p = a.p[b + i], m = a.m[b + i], v = a.v[b + i];
      a.g[b + i] = g;
      if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, p, g);
      m = a.beta1 * m + ob1 * g;
      v = a.beta2 * v + ob2 * g * g;
      a.m[b + i] = m; a.v[b + i] = v;
      a.p[b + i] = p - step * (m / (sqrtf(v) * isb2 + a.eps));
    }
  }
}

// out[0] = #{i : ids[i] != 0} as a double (the BCE normaliser of main.py:151-153 only depends on the batch: under data
// parallelism it is all-reduced beside the forward pass instead of between forward and backward)
__global__ void __launch_bounds__(256) count_nonzero_kernel(const int* __restrict__ ids, int n, double* __restrict__ out) {
  __shared__ double red[8];
  double s = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) s += ids[i] != 0 ? 1.0 : 0.0;
  cta_accumulate(s, out, red);
}

// test helper: materialise the dropout keep-multipliers for elements [0, n) of a site
__global__ void philox_mask_kernel(float* __restrict__ out, long long n, DropDesc d) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = d.enabled ? drop_mul1(d, d.base + (unsigned long long)i) : 1.f;
}

}  // namespace adt
