// Forward pass of the encoder / decoder blocks for WIDE models (H >= 128, bf16 mode): every linear layer is one tcgen05 GEMM
// (adt_gemm_tc: TMA-fed 128 x 128 tiles, fp32 accumulators in TMEM) over ALL rows, and the row-wise work between the GEMMs --
// LayerNorm, dropout, ReLU, residuals, pad mask, the independence head and the reconstruction error -- runs in small warp-per-row
// kernels that read fp32 once and hand the next GEMM its bf16 operand.  Same math, same saved activations and same Philox dropout
// streams as the row-tile kernels of kernels_fwd.cuh (reference: sasrec/modules.py:644-655 encoder, :666-677 decoder); the row-tile
// kernels keep their whole [TM, H] fp32 tiles in shared memory and feed mma.sync from them, which caps them near 30 TFLOP/s at H = 256.
#pragma once
#include "common.cuh"

namespace adt {

// columns of a row owned by a lane: float4 at 4*lane + 128*j, j < RV.  Every warp-per-row kernel below is instantiated for RV = 2
// (H <= 256) and RV = 4 (256 < H <= 512); rv_kernel picks the instantiation from H at launch.
#define rv_kernel(K, H) ((H) > 256 ? K<4> : K<2>)

struct RowLnArgs {
  const float* x; const float* g; const float* b;
  float* y;                    // nullable: LN(x) fp32
  __nv_bfloat16* yb;           // nullable: LN(x) bf16
  __nv_bfloat16* xb;           // nullable: x bf16
  int M, H;
};

__device__ __forceinline__ void st_bf16x4(__nv_bfloat16* p, float4 v) {
  uint2 o;
  o.x = pack_bf16(v.x, v.y); o.y = pack_bf16(v.z, v.w);
  *reinterpret_cast<uint2*>(p) = o;
}

// LayerNorm of a row held as v[RV] by the warp (eps 1e-8, two-pass statistics like ln_tile)
template <int RV>
__device__ __forceinline__ void warp_ln(float4 (&v)[RV], int H, int lane, const float* __restrict__ g, const float* __restrict__ b) {
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < RV; ++j)
    if (4 * lane + 128 * j < H) sum += (v[j].x + v[j].y) + (v[j].z + v[j].w);
  const float mean = warp_sum(sum) / (float)H;
  float var = 0.f;
#pragma unroll
  for (int j = 0; j < RV; ++j)
    if (4 * lane + 128 * j < H) {
      const float a0 = v[j].x - mean, a1 = v[j].y - mean, a2 = v[j].z - mean, a3 = v[j].w - mean;
      var += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
    }
  const float rstd = 1.0f / sqrtf(warp_sum(var) / (float)H + 1e-8f);
#pragma unroll
  for (int j = 0; j < RV; ++j) {
    const int c = 4 * lane + 128 * j;
    if (c < H) {
      const float4 ga = __ldg(reinterpret_cast<const float4*>(g + c)), be = __ldg(reinterpret_cast<const float4*>(b + c));
      v[j] = make_float4((v[j].x - mean) * rstd * ga.x + be.x, (v[j].y - mean) * rstd * ga.y + be.y, (v[j].z - mean) * rstd * ga.z + be.z,
                         (v[j].w - mean) * rstd * ga.w + be.w);
    }
  }
}

template <int RV>
__global__ void __launch_bounds__(256) row_ln_cast_kernel(RowLnArgs a) {
  const int lane = threadIdx.x & 31;
  for (int row = blockIdx.x * 8 + (threadIdx.x >> 5); row < a.M; row += gridDim.x * 8) {
    const long long off = (long long)row * a.H;
    float4 v[RV];
#pragma unroll
    for (int j = 0; j < RV; ++j) {
      const int c = 4 * lane + 128 * j;
      v[j] = c < a.H ? *reinterpret_cast<const float4*>(a.x + off + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      if (a.xb && c < a.H) st_bf16x4(a.xb + off + c, v[j]);
    }
    warp_ln<RV>(v, a.H, lane, a.g, a.b);
#pragma unroll
    for (int j = 0; j < RV; ++j) {
      const int c = 4 * lane + 128 * j;
      if (c < a.H) {
        if (a.y) *reinterpret_cast<float4*>(a.y + off + c) = v[j];
        if (a.yb) st_bf16x4(a.yb + off + c, v[j]);
      }
    }
  }
}

// independence head of the encoder block on the attention context (modules.py:696-703, kernels_fwd.cuh post_fwd):
//   rec[r][c][:] = log_softmax(ctx[r, head c] Ws^T + bs) ; nll_acc += -sum_c rec[r][c][c]          (nh <= 8)
__global__ void __launch_bounds__(256) sparse_head_fwd_kernel(const float* __restrict__ ctx, const float* __restrict__ Wsp,
                                                              const float* __restrict__ bsp, float* __restrict__ rec, double* __restrict__ acc,
                                                              int M, int H, int nh) {
  __shared__ double red[8];
  const int lane = threadIdx.x & 31, hd = H / nh;
  double nll = 0.0;
  for (int row = blockIdx.x * 8 + (threadIdx.x >> 5); row < M; row += gridDim.x * 8) {
    const float* xr = ctx + (long long)row * H;
    for (int c = 0; c < nh; ++c) {
      float lg[8];
      float mx = -INFINITY;
      for (int j = 0; j < nh; ++j) {
        float s = 0.f;
        for (int d = lane; d < hd; d += 32) s = fmaf(xr[c * hd + d], __ldg(Wsp + j * hd + d), s);
        lg[j] = warp_sum(s) + bsp[j];
        mx = fmaxf(mx, lg[j]);
      }
      float se = 0.f;
      for (int j = 0; j < nh; ++j) se += expf(lg[j] - mx);
      const float lz = mx + logf(se);
      if (lane == 0) {
        if (rec)
          for (int j = 0; j < nh; ++j) rec[((long long)row * nh + c) * nh + j] = lg[j] - lz;
        nll -= (double)(lg[c] - lz);
      }
    }
  }
  if (acc) cta_accumulate(nll, acc, red);
}

// a = relu(h1 * m1) as the bf16 operand of the second FFN GEMM (h1 = pre-dropout hidden, saved in fp32 by the first GEMM)
__global__ void __launch_bounds__(256) relu_drop_cast_kernel(const float* __restrict__ h1, __nv_bfloat16* __restrict__ out, long long n4,
                                                             DropDesc drop) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 h = *(reinterpret_cast<const float4*>(h1) + i);
    if (drop.enabled) h = f4_mul(h, drop_mul4(drop, (drop.base >> 2) + (unsigned long long)i));
    st_bf16x4(out + 4 * i, make_float4(fmaxf(h.x, 0.f), fmaxf(h.y, 0.f), fmaxf(h.z, 0.f), fmaxf(h.w, 0.f)));
  }
}

__global__ void __launch_bounds__(256) cast_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out, long long n4) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x)
    st_bf16x4(out + 4 * i, *(reinterpret_cast<const float4*>(x) + i));
}

// block output.  encoder: out = (h2*m2 + LN2(y)) * keep ; decoder: out = (h2*m2 + c + d) * keep, mse_acc += sum (enc_in - out)^2
struct RowOutArgs {
  const float* h2; const float* u;        // u = y (enc) or c (dec)
  const float* resid;                     // dec: d
  const float* ln_g; const float* ln_b;   // enc: LN2
  const int* ids; const float* enc_in;
  float* out; double* acc;
  int M, H, is_dec;
  DropDesc drop2;
};

template <int RV>
__global__ void __launch_bounds__(256) row_out_kernel(RowOutArgs a) {
  __shared__ double red[8];
  const int lane = threadIdx.x & 31;
  double sq = 0.0;
  for (int row = blockIdx.x * 8 + (threadIdx.x >> 5); row < a.M; row += gridDim.x * 8) {
    const long long off = (long long)row * a.H;
    float4 v[RV];
#pragma unroll
    for (int j = 0; j < RV; ++j) {
      const int c = 4 * lane + 128 * j;
      v[j] = c < a.H ? *reinterpret_cast<const float4*>(a.u + off + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (!a.is_dec) warp_ln<RV>(v, a.H, lane, a.ln_g, a.ln_b);
    const bool keep = a.ids[row] != 0;
#pragma unroll
    for (int j = 0; j < RV; ++j) {
      const int c = 4 * lane + 128 * j;
      if (c >= a.H) continue;
      float4 h2 = *reinterpret_cast<const float4*>(a.h2 + off + c);
      if (a.drop2.enabled) h2 = f4_mul(h2, drop_mul4(a.drop2, (a.drop2.base + (unsigned long long)(off + c)) >> 2));
      float4 o = f4_add(h2, v[j]);
      if (a.is_dec) o = f4_add(o, *reinterpret_cast<const float4*>(a.resid + off + c));
      if (!keep) o = make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(a.out + off + c) = o;
      if (a.is_dec && a.enc_in) {
        const float4 e = *reinterpret_cast<const float4*>(a.enc_in + off + c);
        const float dx = e.x - o.x, dy = e.y - o.y, dz = e.z - o.z, dw = e.w - o.w;
        sq += (double)(dx * dx + dy * dy) + (double)(dz * dz + dw * dw);
      }
    }
  }
  if (a.is_dec && a.acc) cta_accumulate(sq, a.acc, red);
}

}  // namespace adt

// =====================================================================================================================
// Backward pass of the same path.  Every product is a tcgen05 GEMM over all rows -- dgrad reads the fp32->bf16 weight MN-major,
// wgrad reads the bf16 dY / X matrices MN-major with split K -- and the row-wise adjoints below sit between them.  Column sums (bias
// and LayerNorm gradients) are kept per lane across the rows a warp walks, merged per CTA in shared memory, then added with one
// atomic per column per CTA.
// =====================================================================================================================
namespace adt {

template <int RV>
__device__ __forceinline__ void lane_cols_to_smem(float* __restrict__ sm, const float4 (&p)[RV], int H, int lane) {
#pragma unroll
  for (int j = 0; j < RV; ++j) {
    const int c = 4 * lane + 128 * j;
    if (c < H) { atomicAdd(sm + c, p[j].x); atomicAdd(sm + c + 1, p[j].y); atomicAdd(sm + c + 2, p[j].z); atomicAdd(sm + c + 3, p[j].w); }
  }
}
__device__ __forceinline__ void smem_cols_to_global(const float* __restrict__ sm, float* __restrict__ g, int H) {
  if (g)
    for (int c = threadIdx.x; c < H; c += blockDim.x) atomicAdd(g + c, sm[c]);
}

// adjoint of the block output and of the second FFN layer's epilogue (post_bwd step 1/2):
//   dO = (dout + mse_coef (out - enc_in)) * keep ; dh2 = dO * m2 ; a = relu(h1 * m1)
struct RowPostPrepArgs {
  const float* dout; const float* out; const float* enc_in; float mse_coef; float* denc;
  const int* ids; const float* h1;
  float* g;                    // dO fp32 (enc: becomes dz after the C1 dgrad accumulates into it ; dec: becomes dc)
  float* g_copy;               // dec: second copy of dO = dd (gradient reaching d through the residual); nullable
  __nv_bfloat16* dh2b; __nv_bfloat16* ab;
  float* gc2;
  int M, H, is_dec;
  DropDesc drop1, drop2;
};

template <int RV>
__global__ void __launch_bounds__(256) row_post_prep_kernel(RowPostPrepArgs a) {
  __shared__ float cs[128 * RV];
  const int lane = threadIdx.x & 31;
  for (int c = threadIdx.x; c < a.H; c += 256) cs[c] = 0.f;
  __syncthreads();
  float4 part[RV];
#pragma unroll
  for (int j = 0; j < RV; ++j) part[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int row = blockIdx.x * 8 + (threadIdx.x >> 5); row < a.M; row += gridDim.x * 8) {
    const long long off = (long long)row * a.H;
    const bool keep = a.ids[row] != 0;
#pragma unroll
    for (int j = 0; j < RV; ++j) {
      const int c = 4 * lane + 128 * j;
      if (c >= a.H) continue;
      const long long gi = off + c;
      float4 g = a.dout ? *reinterpret_cast<const float4*>(a.dout + gi) : make_float4(0.f, 0.f, 0.f, 0.f);
      if (a.is_dec && a.enc_in) {
        const float4 o = *reinterpret_cast<const float4*>(a.out + gi), e = *reinterpret_cast<const float4*>(a.enc_in + gi);
        const float4 d = make_float4(a.mse_coef * (o.x - e.x), a.mse_coef * (o.y - e.y), a.mse_coef * (o.z - e.z), a.mse_coef * (o.w - e.w));
        g = f4_add(g, d);
        if (a.denc) *reinterpret_cast<float4*>(a.denc + gi) = make_float4(-d.x, -d.y, -d.z, -d.w);
      }
      if (!keep) g = make_float4(0.f, 0.f, 0.f, 0.f);
      float4 h = *reinterpret_cast<const float4*>(a.h1 + gi);
      if (a.drop1.enabled) h = f4_mul(h, drop_mul4(a.drop1, (a.drop1.base + (unsigned long long)gi) >> 2));
      float4 d2 = g;
      if (a.drop2.enabled) d2 = f4_mul(d2, drop_mul4(a.drop2, (a.drop2.base + (unsigned long long)gi) >> 2));
      *reinterpret_cast<float4*>(a.g + gi) = g;
      if (a.g_copy) *reinterpret_cast<float4*>(a.g_copy + gi) = g;
      st_bf16x4(a.dh2b + gi, d2);
      st_bf16x4(a.ab + gi, make_float4(fmaxf(h.x, 0.f), fmaxf(h.y, 0.f), fmaxf(h.z, 0.f), fmaxf(h.w, 0.f)));
      part[j] = f4_add(part[j], d2);
    }
  }
  lane_cols_to_smem<RV>(cs, part, a.H, lane);
  __syncthreads();
  smem_cols_to_global(cs, a.gc2, a.H);
}

// dh1 = da * [h1 m1 > 0] * m1 -> bf16 ; gc1 += colsum(dh1)        (post_bwd step 4)
template <int RV>
__global__ void __launch_bounds__(256) row_dh1_kernel(const float* __restrict__ da, const float* __restrict__ h1, __nv_bfloat16* __restrict__ dh1b,
                                                      float* __restrict__ gc1, int M, int H, DropDesc drop1) {
  __shared__ float cs[128 * RV];
  const int lane = threadIdx.x & 31;
  for (int c = threadIdx.x; c < H; c += 256) cs[c] = 0.f;
  __syncthreads();
  float4 part[RV];
#pragma unroll
  for (int j = 0; j < RV; ++j) part[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int row = blockIdx.x * 8 + (threadIdx.x >> 5); row < M; row += gridDim.x * 8) {
#pragma unroll
    for (int j = 0; j < RV; ++j) {
      const int c = 4 * lane + 128 * j;
      if (c >= H) continue;
      const long long gi = (long long)row * H + c;
      const float4 h = *reinterpret_cast<const float4*>(h1 + gi), d = *reinterpret_cast<const float4*>(da + gi);
      float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
      if (drop1.enabled) m = drop_mul4(drop1, (drop1.base + (unsigned long long)gi) >> 2);
      const float4 o = make_float4(h.x * m.x > 0.f ? d.x * m.x : 0.f, h.y * m.y > 0.f ? d.y * m.y : 0.f, h.z * m.z > 0.f ? d.z * m.z : 0.f,
                                   h.w * m.w > 0.f ? d.w * m.w : 0.f);
      st_bf16x4(dh1b + gi, o);
      part[j] = f4_add(part[j], o);
    }
  }
  lane_cols_to_smem<RV>(cs, part, H, lane);
  __syncthreads();
  smem_cols_to_global(cs, gc1, H);
}

// LayerNorm adjoint: dx = LN^T(g) (+ extra) ; gln_g += sum g * xhat ; gln_b += sum g ; optional bf16 copy of dx and gb += colsum(dx)
struct RowLnBwdArgs {
  const float* x; const float* g; const float* ln_g; const float* extra;
  float* dx; __nv_bfloat16* dxb; float* gln_g; float* gln_b; float* gb;
  int M, H;
};

template <int RV>
__global__ void __launch_bounds__(256) row_ln_bwd_kernel(RowLnBwdArgs a) {
  __shared__ float cs[3 * 128 * RV];
  const int lane = threadIdx.x & 31, H = a.H;
  for (int c = threadIdx.x; c < 3 * H; c += 256) cs[c] = 0.f;
  __syncthreads();
  float4 pg[RV], pb[RV], pc[RV];
#pragma unroll
  for (int j = 0; j < RV; ++j) pg[j] = pb[j] = pc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int row = blockIdx.x * 8 + (threadIdx.x >> 5); row < a.M; row += gridDim.x * 8) {
    const long long off = (long long)row * H;
    float4 xv[RV], gv[RV];
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < RV; ++j) {
      const int c = 4 * lane + 128 * j;
      xv[j] = gv[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c < H) {
        xv[j] = *reinterpret_cast<const float4*>(a.x + off + c);
        gv[j] = *reinterpret_cast<const float4*>(a.g + off + c);
        sum += (xv[j].x + xv[j].y) + (xv[j].z + xv[j].w);
      }
    }
    const float mean = warp_sum(sum) / (float)H;
    float var = 0.f;
#pragma unroll
    for (int j = 0; j < RV; ++j)
      if (4 * lane + 128 * j < H) {
        const float a0 = xv[j].x - mean, a1 = xv[j].y - mean, a2 = xv[j].z - mean, a3 = xv[j].w - mean;
        var += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
      }
    const float rstd = 1.0f / sqrtf(warp_sum(var) / (float)H + 1e-8f);
    float s1 = 0.f, s2 = 0.f;
    float4 gg[RV];
#pragma unroll
    for (int j = 0; j < RV; ++j) {
      const int c = 4 * lane + 128 * j;
      gg[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c < H) {
        const float4 w = __ldg(reinterpret_cast<const float4*>(a.ln_g + c));
        xv[j] = make_float4((xv[j].x - mean) * rstd, (xv[j].y - mean) * rstd, (xv[j].z - mean) * rstd, (xv[j].w - mean) * rstd);   // xhat
        gg[j] = f4_mul(gv[j], w);
        s1 += (gg[j].x + gg[j].y) + (gg[j].z + gg[j].w);
        s2 += (gg[j].x * xv[j].x + gg[j].y * xv[j].y) + (gg[j].z * xv[j].z + gg[j].w * xv[j].w);
        pg[j] = f4_add(pg[j], f4_mul(gv[j], xv[j]));
        pb[j] = f4_add(pb[j], gv[j]);
      }
    }
    s1 = warp_sum(s1) / (float)H;
    s2 = warp_sum(s2) / (float)H;
#pragma unroll
    for (int j = 0; j < RV; ++j) {
      const int c = 4 * lane + 128 * j;
      if (c >= H) continue;
      float4 d = make_float4(rstd * (gg[j].x - s1 - xv[j].x * s2), rstd * (gg[j].y - s1 - xv[j].y * s2), rstd * (gg[j].z - s1 - xv[j].z * s2),
                             rstd * (gg[j].w - s1 - xv[j].w * s2));
      if (a.extra) d = f4_add(d, *reinterpret_cast<const float4*>(a.extra + off + c));
      *reinterpret_cast<float4*>(a.dx + off + c) = d;
      if (a.dxb) st_bf16x4(a.dxb + off + c, d);
      pc[j] = f4_add(pc[j], d);
    }
  }
  lane_cols_to_smem<RV>(cs, pg, H, lane);
  lane_cols_to_smem<RV>(cs + H, pb, H, lane);
  if (a.gb) lane_cols_to_smem<RV>(cs + 2 * H, pc, H, lane);
  __syncthreads();
  smem_cols_to_global(cs, a.gln_g, H);
  smem_cols_to_global(cs + H, a.gln_b, H);
  smem_cols_to_global(cs + 2 * H, a.gb, H);
}

// up to three fp32 [M,H] matrices, scaled, packed as column blocks of one bf16 [M, ld] matrix ; gb_i += colsum(scale_i * src_i)
struct RowPackArgs {
  const float* src[3]; float scale[3]; float* gb[3];
  __nv_bfloat16* dst; long long ld; int n, M, H;
};

template <int RV>
__global__ void __launch_bounds__(256) row_pack_kernel(RowPackArgs a) {
  __shared__ float cs[3 * 128 * RV];
  const int lane = threadIdx.x & 31, H = a.H;
  for (int c = threadIdx.x; c < 3 * H; c += 256) cs[c] = 0.f;
  __syncthreads();
  float4 part[3][RV];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < RV; ++j) part[i][j] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int row = blockIdx.x * 8 + (threadIdx.x >> 5); row < a.M; row += gridDim.x * 8) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      if (i >= a.n) continue;
#pragma unroll
      for (int j = 0; j < RV; ++j) {
        const int c = 4 * lane + 128 * j;
        if (c >= H) continue;
        const float4 v = f4_scale(*reinterpret_cast<const float4*>(a.src[i] + (long long)row * H + c), a.scale[i]);
        st_bf16x4(a.dst + (long long)row * a.ld + i * H + c, v);
        part[i][j] = f4_add(part[i][j], v);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 3; ++i)
    if (i < a.n && a.gb[i]) lane_cols_to_smem<RV>(cs + i * H, part[i], H, lane);
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 3; ++i)
    if (i < a.n) smem_cols_to_global(cs + i * H, a.gb[i], H);
}

// adjoint of the independence head (post_bwd step 9): dl = nll_coef (softmax - onehot) [+ log-softmax adjoint of drec] ;
//   dctx[r, head c] += dl[c] Ws ; gWs += sum dl[c]^T ctx[r, head c] ; gbs += sum dl[c]          (hd a multiple of 32, nh <= 8, H <= 128 RV)
template <int RV>
__global__ void __launch_bounds__(256) sparse_head_bwd_kernel(const float* __restrict__ ctx, const float* __restrict__ Wsp,
                                                              const float* __restrict__ bsp, const float* __restrict__ drec, float nll_coef,
                                                              float* __restrict__ dctx, float* __restrict__ gWsp, float* __restrict__ gbsp, int M,
                                                              int H, int nh) {
  __shared__ float gw[128 * RV];
  __shared__ float gbv[8];
  __shared__ float dls[8][8];          // per warp: dl[j] of the (row, head) being processed
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, hd = H / nh, tpd = hd >> 5, nflat = H >> 5;
  for (int c = threadIdx.x; c < H; c += 256) gw[c] = 0.f;
  if (threadIdx.x < 8) gbv[threadIdx.x] = 0.f;
  __syncthreads();
  // this lane's share of gWs: flat slot i <-> (class j = i / tpd, column d = lane + 32 (i % tpd)); slots are compile-time indices
  float accw[4 * RV], accb[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) accb[i] = 0.f;
#pragma unroll
  for (int i = 0; i < 4 * RV; ++i) accw[i] = 0.f;
  for (int row = blockIdx.x * 8 + w; row < M; row += gridDim.x * 8) {
    const float* xr = ctx + (long long)row * H;
    float* dr_out = dctx + (long long)row * H;
    for (int c = 0; c < nh; ++c) {
      float lg[8];
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        lg[j] = -INFINITY;
        if (j < nh) {
          float s = 0.f;
          for (int d = lane; d < hd; d += 32) s = fmaf(xr[c * hd + d], __ldg(Wsp + j * hd + d), s);
          lg[j] = warp_sum(s) + bsp[j];
          mx = fmaxf(mx, lg[j]);
        }
      }
      float se = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < nh) se += expf(lg[j] - mx);
      const float* dr = drec ? drec + ((long long)row * nh + c) * nh : nullptr;
      float gsum = 0.f;
      if (dr) for (int j = 0; j < nh; ++j) gsum += dr[j];
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < nh) {
          const float pj = expf(lg[j] - mx) / se;
          float dl = nll_coef * (pj - (j == c ? 1.f : 0.f));
          if (dr) dl += dr[j] - pj * gsum;
          accb[j] += dl;                       // identical in every lane; lane 0's copy is used
          if (lane == 0) dls[w][j] = dl;
        }
      __syncwarp();
      for (int d = lane; d < hd; d += 32) {
        float add = 0.f;
        for (int j = 0; j < nh; ++j) add = fmaf(dls[w][j], __ldg(Wsp + j * hd + d), add);
        dr_out[c * hd + d] += add;
      }
#pragma unroll
      for (int i = 0; i < 4 * RV; ++i)
        if (i < nflat) {
          const int j = i / tpd, t = i - j * tpd;
          accw[i] = fmaf(dls[w][j], xr[c * hd + lane + 32 * t], accw[i]);
        }
    }
  }
#pragma unroll
  for (int i = 0; i < 4 * RV; ++i)
    if (i < nflat) {
      const int j = i / tpd, t = i - j * tpd;
      atomicAdd(gw + j * hd + lane + 32 * t, accw[i]);
    }
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (j < nh) atomicAdd(gbv + j, accb[j]);
  }
  __syncthreads();
  smem_cols_to_global(gw, gWsp, H);
  if (threadIdx.x < nh) atomicAdd(gbsp + threadIdx.x, gbv[threadIdx.x]);
}

}  // namespace adt

// =====================================================================================================================
// Attention for long sequences (64 < L <= 256) as strided-batch tcgen05 GEMMs over (sequence, head) + one warp-per-row
// softmax kernel.  S = q k^T and P, dS live in HBM as [B*nh][L][Lp] matrices (82 MB fp32 at C1: HBM-cheap next to the
// generic kernel's 14 TFLOP/s) -- same masks, same Philox dropout stream, same lse as attn_fwd_kernel / attn_bwd_kernel.
// =====================================================================================================================
namespace adt {

struct AttnRowArgs {
  const float* S;              // [Z][L][Lp] scores (q pre-scaled)
  const float* dP;             // bwd: dctx v^T, same layout
  const float* lse_in;         // bwd: saved row log-sum-exp [Z][L]
  float* lse_out;              // fwd (nullable)
  __nv_bfloat16* Pb;           // fwd: dropout(softmax) ; bwd: softmax * mask  (operand of ctx / dv)
  __nv_bfloat16* dSb;          // bwd: p * (dp - delta)                          (operand of dq / dk)
  const int* key_ids;          // mask_mode 1
  int Z, L, Lp, nh, mask_mode, bwd;
  DropDesc drop;
};

// one warp per (z, i) row; lane owns keys 8*lane .. 8*lane+7 (L <= 256)
__global__ void __launch_bounds__(256) attn_row_kernel(AttnRowArgs a) {
  const int lane = threadIdx.x & 31;
  const long long nrows = (long long)a.Z * a.L;
  for (long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); row < nrows; row += (long long)gridDim.x * 8) {
    const int z = (int)(row / a.L), i = (int)(row - (long long)z * a.L), b = z / a.nh;
    const int nj = a.mask_mode == 0 ? i + 1 : a.L;
    const int j0 = 8 * lane;
    const float* srow = a.S + row * a.Lp;
    float sv[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) sv[c] = -INFINITY;
    if (j0 < nj) {
      const float4 s0 = *reinterpret_cast<const float4*>(srow + j0), s1 = *reinterpret_cast<const float4*>(srow + j0 + 4);
      sv[0] = s0.x; sv[1] = s0.y; sv[2] = s0.z; sv[3] = s0.w; sv[4] = s1.x; sv[5] = s1.y; sv[6] = s1.z; sv[7] = s1.w;
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      if (j0 + c >= nj) sv[c] = -INFINITY;
      else if (a.mask_mode == 1 && a.key_ids[b * a.L + j0 + c] == 0) sv[c] = -1e9f;
    }
    float mv[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) mv[c] = 1.f;
    if (a.drop.enabled && j0 < nj) drop_mul8_attn(a.drop, a.drop.base + (unsigned long long)row, ((a.L + 7) & ~7) >> 3, lane, mv);
    float out0[8], out1[8];
    if (!a.bwd) {
      float mx = -INFINITY;
#pragma unroll
      for (int c = 0; c < 8; ++c) mx = fmaxf(mx, sv[c]);
      mx = warp_max(mx);
      float sum = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) { sv[c] = sv[c] == -INFINITY ? 0.f : expf(sv[c] - mx); sum += sv[c]; }
      sum = warp_sum(sum);
      const float inv = 1.0f / sum;
      if (a.lse_out && lane == 0) a.lse_out[row] = mx + logf(sum);
#pragma unroll
      for (int c = 0; c < 8; ++c) out0[c] = sv[c] * mv[c] * inv;
    } else {
      const float ls = a.lse_in[row];
      float dv8[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) dv8[c] = 0.f;
      if (j0 < nj) {
        const float4 d0 = *reinterpret_cast<const float4*>(a.dP + row * a.Lp + j0), d1 = *reinterpret_cast<const float4*>(a.dP + row * a.Lp + j0 + 4);
        dv8[0] = d0.x; dv8[1] = d0.y; dv8[2] = d0.z; dv8[3] = d0.w; dv8[4] = d1.x; dv8[5] = d1.y; dv8[6] = d1.z; dv8[7] = d1.w;
      }
      float delta = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float pj = sv[c] == -INFINITY ? 0.f : expf(sv[c] - ls);
        const float dp = sv[c] == -INFINITY ? 0.f : dv8[c] * mv[c];
        delta = fmaf(dp, pj, delta);
        sv[c] = pj; dv8[c] = dp;
      }
      delta = warp_sum(delta);
#pragma unroll
      for (int c = 0; c < 8; ++c) { out0[c] = sv[c] * mv[c]; out1[c] = sv[c] * (dv8[c] - delta); }
    }
    // every column up to Lp is written (zeros beyond the visible keys): the following GEMMs reduce over all L columns
    if (j0 < a.Lp) {
      uint4 o;
      o.x = pack_bf16(out0[0], out0[1]); o.y = pack_bf16(out0[2], out0[3]); o.z = pack_bf16(out0[4], out0[5]); o.w = pack_bf16(out0[6], out0[7]);
      *reinterpret_cast<uint4*>(a.Pb + row * a.Lp + j0) = o;
      if (a.bwd) {
        o.x = pack_bf16(out1[0], out1[1]); o.y = pack_bf16(out1[2], out1[3]); o.z = pack_bf16(out1[4], out1[5]); o.w = pack_bf16(out1[6], out1[7]);
        *reinterpret_cast<uint4*>(a.dSb + row * a.Lp + j0) = o;
      }
    }
  }
}

}  // namespace adt
