// nn.Linear on the 5th-generation tensor cores: C[M,N] (fp32) = act((A[M,K] . B[N,K]^T + bias[N]) * scale)  with A, B bf16 K-major.
// One GEMM serves the three products of a linear layer (bert4rec/model/modules.py:57-72, :128-139, bert.py:80-90; the wide
// contractions of the H = 256 shapes, SURVEY 8a rows a19 / a6-a10):
//   forward   y  = x W^T        A = x   [M,K]      B = W    [N,K]
//   dgrad     dx = dy W         A = dy  [M,N]      B = W read MN-major (b_mn: the operand is stored [K][N], N contiguous)
//   wgrad     dW = dy^T x       A = dy, B = x, both read MN-major (a_mn, b_mn: stored [K][M] / [K][N]) -- no transposed copies;
//                               split_k CTAs share one output tile and add their partial sums with vector atomics
// An MN-major K-slab is loaded as 64-column boxes of 64 K-rows (128-byte rows, SWIZZLE_128B): exactly the canonical MN-major
// layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units with LBO = one box (8 KB) and SBO = 8 K-rows (1 KB).
// Structure: one 128 x BN output tile per CTA; warp 0 = TMA producer (A and B K-slabs of 64 through an NS-stage ring), warp 1 =
// tcgen05.mma issuer (accumulator 128 x BN fp32 in TMEM), warps 2-5 = epilogue (tcgen05.ld -> bias / scale / activation -> fp32
// rows to HBM, thread == output row).  K, M, N are arbitrary: TMA zero-fills out-of-bounds rows / columns, stores are masked.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

#include "../../include/adt_b200.h"
#include "tc.cuh"

using namespace adt;

namespace {

constexpr int GM = 128;            // output rows per CTA (= TMEM lanes)
constexpr int G_THREADS = 192;

struct GemmTcArgs {
  float* C; float* pre; const float* bias; long long ldc;
  int M, N, K, act, accumulate; float scale;
  int a_mn, b_mn, kb_per_split;
  float* C2; int n_split;     // columns >= n_split (a multiple of 32) are written to C2 at column (col - n_split)
  int causal_skip;            // output tiles entirely above the diagonal (n0 > m0 + 127) are never read by the caller: skip them
  int tiles_n, tiles_m, n_work, n_split_k;   // work items = tiles_n x tiles_m x (batch | K splits)
  int stage;                                 // the launch reserved the chunk staging area of the coalesced epilogue
  int batch_inner, nbatch;    // strided batch: blockIdx.z = zo * batch_inner + zi selects the matrices (nbatch <= 1: blockIdx.z = K split)
  long long c_so, c_si;       // element offsets of C per outer / inner batch index
  // linear + cross-entropy epilogues (MODE 1 / 2 of gemm_tc_kernel; C, pre, act, split K and batching unused there).  Columns are
  // local to one vocabulary chunk: the B map, bias and g_bias start at its first row, labels are shifted by label_off.
  const int* labels; int label_off;
  float2* part;               // MODE 1: per-tile (max, sum exp) of every row, [tiles_n][M]
  float* zlab;                // MODE 1: z[r, label[r]] when the label falls in this chunk
  const float* lse;           // MODE 2: per-row log-sum-exp of the forward
  float coef; const float* coef_dev;     // MODE 2: dS = coef * (*coef_dev) * (softmax - onehot)
  __nv_bfloat16* ds; long long ld_ds;    // MODE 2: bf16 dS [M][ld_ds]
  float* g_bias;              // MODE 2: += fp32 column sums of dS (NULL: no bias)
};

__device__ __forceinline__ float g_gelu(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float g_act(float x, int act) {
  return act == 1 ? fmaxf(x, 0.f) : act == 2 ? g_gelu(x) : act == 3 ? (x > 0.f ? x : expm1f(x)) : act == 4 ? (x > 0.f ? x : expm1f(x)) + 1.f : x;
}

// one 32-column chunk of a row: pre-activation copy, activation (compiled out for act == 0: a per-element switch on a run-time `act`
// cost a constant-bank jump per element), then store / accumulate / atomic add (split K)
template <bool ACT>
__device__ __forceinline__ void epi_chunk(const GemmTcArgs& a, float (&v)[32], float* __restrict__ crow, float* __restrict__ prow, int nb, bool vec,
                                          bool atomic) {
  if (vec) {
#pragma unroll
    for (int c = 0; c < 32; c += 4) {
      float4 o = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
      if (prow) *reinterpret_cast<float4*>(prow + c) = o;
      if (ACT) o = make_float4(g_act(o.x, a.act), g_act(o.y, a.act), g_act(o.z, a.act), g_act(o.w, a.act));
      if (atomic) { atomicAdd(reinterpret_cast<float4*>(crow + c), o); continue; }
      if (a.accumulate) {
        const float4 old = *reinterpret_cast<const float4*>(crow + c);
        o = make_float4(o.x + old.x, o.y + old.y, o.z + old.z, o.w + old.w);
      }
      *reinterpret_cast<float4*>(crow + c) = o;
    }
  } else {
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      if (nb + c < a.N) {
        if (prow) prow[c] = v[c];
        float o = ACT ? g_act(v[c], a.act) : v[c];
        if (atomic) { atomicAdd(crow + c, o); continue; }
        if (a.accumulate) o += crow[c];
        crow[c] = o;
      }
    }
  }
}

// Coalesced variant for full 32-column chunks: the warp parks its 32 x 32 chunk in shared memory (thread == row while reading TMEM) and
// writes it back four rows per instruction, 128 contiguous bytes per row -- a thread-per-row store touches 32 different lines with
// 16 bytes each, twice the L2 write requests for the same bytes.
template <bool ACT>
__device__ __forceinline__ void epi_chunk_staged(const GemmTcArgs& a, float (&v)[32], float* __restrict__ stage, float* __restrict__ cbase, int row0,
                                                 bool atomic) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int c = 0; c < 32; c += 4) {
    float4 o = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
    if (ACT) o = make_float4(g_act(o.x, a.act), g_act(o.y, a.act), g_act(o.z, a.act), g_act(o.w, a.act));
    *reinterpret_cast<float4*>(stage + lane * 36 + c) = o;
  }
  __syncwarp();
  const int sub = lane >> 3, c4 = (lane & 7) * 4;
#pragma unroll
  for (int r = 0; r < 32; r += 4) {
    const int rr = r + sub;
    if (row0 + rr < a.M) {
      float4 o = *reinterpret_cast<const float4*>(stage + rr * 36 + c4);
      float* dst = cbase + (long long)rr * a.ldc + c4;
      if (atomic) { atomicAdd(reinterpret_cast<float4*>(dst), o); continue; }
      if (a.accumulate) {
        const float4 old = *reinterpret_cast<const float4*>(dst);
        o = make_float4(o.x + old.x, o.y + old.y, o.z + old.z, o.w + old.w);
      }
      *reinterpret_cast<float4*>(dst) = o;
    }
  }
  __syncwarp();
}

// Persistent: a CTA walks work items w = blockIdx.x, blockIdx.x + gridDim.x, ... where an item is one 128 x BN output tile of one
// matrix of the batch (or one K split of it).  The TMA ring and the two TMEM accumulators run ACROSS items: while the epilogue warps
// drain item i, the producer is already loading item i+1 and the MMA warp fills the other accumulator -- the H x H layers and the
// attention products of a block are thousands of 2-4-slab items whose per-CTA set-up (barriers, TMEM allocation, first TMA round trip)
// otherwise costs more than their math.
struct WorkItem { int m0, n0, zi, zo, kb0, nkb; bool skip; };
__device__ __forceinline__ WorkItem g_item(const GemmTcArgs& a, int w, int BN) {
  WorkItem it;
  const int tn = w % a.tiles_n, r = w / a.tiles_n, tm = r % a.tiles_m, z = r / a.tiles_m;
  it.n0 = tn * BN; it.m0 = tm * GM;
  const int nkb_all = (a.K + 63) / 64;
  if (a.nbatch > 1) { it.zi = z % a.batch_inner; it.zo = z / a.batch_inner; it.kb0 = 0; it.nkb = nkb_all; }
  else { it.zi = it.zo = 0; it.kb0 = z * a.kb_per_split; it.nkb = min(a.kb_per_split, nkb_all - it.kb0); }
  it.skip = a.causal_skip && it.n0 > it.m0 + GM - 1;       // tile entirely above the diagonal: never read by the caller
  return it;
}

// Epilogue of the fused vocabulary head (adt_linear_ce_fwd / _bwd): z = acc + bias[v] leaves TMEM and is consumed on chip.
//   MODE 1: the thread owning row r keeps a running (max, sum exp) over the tile's columns and writes it to part[tile_n][r]; it also
//           takes z[r, label[r]] from the same accumulator when the label falls in the tile.  The scores never reach HBM.
//   MODE 2: dS = c (exp(z - lse[r]) - [v == label[r]]) in fp32; its column sums go to g_bias (atomics, one per column per warp and
//           tile), then it is rounded to bf16 and stored as [M][ld_ds] rows, 64 contiguous bytes per half-warp, via the staging chunk.
template <int BN, int MODE>
__device__ __forceinline__ void ce_epilogue(const GemmTcArgs& a, uint32_t tmem_base, uint64_t* tfull, uint64_t* tempty, float* __restrict__ stage,
                                            int q, int lane) {
  const float c = MODE == 2 ? a.coef * (a.coef_dev ? *a.coef_dev : 1.f) : 0.f;
  int n = 0;
  for (int w = blockIdx.x; w < a.n_work; w += gridDim.x) {
    const WorkItem it = g_item(a, w, BN);
    const int acc = n & 1;
    tc::mbar_wait(tfull + acc, (n >> 1) & 1);
    tc::tc_fence_after();
    const int row = it.m0 + 32 * q + lane;
    const bool live = row < a.M;
    const int lab = live ? __ldg(a.labels + row) - a.label_off : -1;
    const float ls = MODE == 2 && live ? __ldg(a.lse + row) : 0.f;
    float m = -INFINITY, s = 0.f, zl = 0.f;
    bool has = false;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      float v[32];
      tc::tmem_ld32(tmem_base + ((uint32_t)(32 * q) << 16) + acc * BN + c0, v);
      if (c0 + 32 == BN) {
        tc::tc_fence_before();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(tempty + acc);
      }
      const int nb = it.n0 + c0;
      if (nb >= a.N) continue;             // warp-uniform
      if (a.bias) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (nb + j < a.N) v[j] += __ldg(a.bias + nb + j);
      }
      if constexpr (MODE == 1) {
        float cm = -INFINITY;
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (nb + j < a.N) cm = fmaxf(cm, v[j]);
        if (lab >= nb && lab < nb + 32) {
          has = true;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (nb + j == lab) zl = v[j];
        }
        const float mn = fmaxf(m, cm);
        float t = 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j) t += nb + j < a.N ? __expf(v[j] - mn) : 0.f;
        s = s * __expf(m - mn) + t;
        m = mn;
      } else {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          float4 o;
          o.x = live && nb + j < a.N ? c * (__expf(v[j] - ls) - (nb + j == lab ? 1.f : 0.f)) : 0.f;
          o.y = live && nb + j + 1 < a.N ? c * (__expf(v[j + 1] - ls) - (nb + j + 1 == lab ? 1.f : 0.f)) : 0.f;
          o.z = live && nb + j + 2 < a.N ? c * (__expf(v[j + 2] - ls) - (nb + j + 2 == lab ? 1.f : 0.f)) : 0.f;
          o.w = live && nb + j + 3 < a.N ? c * (__expf(v[j + 3] - ls) - (nb + j + 3 == lab ? 1.f : 0.f)) : 0.f;
          *reinterpret_cast<float4*>(stage + lane * 36 + j) = o;
        }
        __syncwarp();
        if (a.g_bias) {                    // lane == column: fp32 sum over the warp's 32 rows (dead rows hold 0)
          float cs = 0.f;
#pragma unroll 8
          for (int r = 0; r < 32; ++r) cs += stage[r * 36 + lane];
          if (nb + lane < a.N) atomicAdd(a.g_bias + nb + lane, cs);
        }
        const int hr = lane >> 4, cc = (lane & 15) * 2, row0 = it.m0 + 32 * q;
#pragma unroll 4
        for (int r = 0; r < 32; r += 2) {
          const int rr = r + hr;
          if (row0 + rr >= a.M || nb + cc >= a.N) continue;
          const float2 p = *reinterpret_cast<const float2*>(stage + rr * 36 + cc);
          __nv_bfloat16* dst = a.ds + (long long)(row0 + rr) * a.ld_ds + nb + cc;
          if (nb + cc + 1 < a.N) *reinterpret_cast<__nv_bfloat162*>(dst) = __floats2bfloat162_rn(p.x, p.y);
          else *dst = __float2bfloat16_rn(p.x);
        }
        __syncwarp();
      }
    }
    if constexpr (MODE == 1) {
      if (live) {
        a.part[(long long)(it.n0 / BN) * a.M + row] = make_float2(m, s);
        if (has) a.zlab[row] = zl;
      }
    }
    ++n;
  }
}

template <int BN, int NS, int MODE = 0>
__global__ void __launch_bounds__(G_THREADS, 1) gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                                                               GemmTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  constexpr int A_STAGE = GM * 128, B_STAGE = BN * 128;        // one 64-wide K slab (128 bytes per row)
  uint8_t* sA = smem;
  uint8_t* sB = sA + NS * A_STAGE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + NS * B_STAGE);
  uint64_t* full = bars;
  uint64_t* empty = bars + NS;
  uint64_t* tfull = bars + 2 * NS;        // [2] accumulator ready
  uint64_t* tempty = bars + 2 * NS + 2;   // [2] accumulator drained (one arrival per epilogue warp)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NS + 4);
  float* stage_all = reinterpret_cast<float*>(sB + NS * B_STAGE + 256);     // [4 epilogue warps][32][36] chunk staging
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool split = a.nbatch <= 1 && a.n_split_k > 1;

  if (threadIdx.x == 0) {
    tc::tma_prefetch_desc(&tmA);
    tc::tma_prefetch_desc(&tmB);
    for (int i = 0; i < NS; ++i) { tc::mbar_init(full + i, 1); tc::mbar_init(empty + i, 1); }
    for (int i = 0; i < 2; ++i) { tc::mbar_init(tfull + i, 1); tc::mbar_init(tempty + i, 4); }
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc<2 * BN>(tmem_slot);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int g = 0;                                             // slabs issued so far (ring position)
      for (int w = blockIdx.x; w < a.n_work; w += gridDim.x) {
        const WorkItem it = g_item(a, w, BN);
        if (it.skip) continue;
        for (int kb = 0; kb < it.nkb; ++kb, ++g) {
          const int st = g % NS;
          tc::mbar_wait(empty + st, ((g / NS) & 1) ^ 1);
          tc::mbar_arrive_expect_tx(full + st, A_STAGE + B_STAGE);
          const int kc = (it.kb0 + kb) * 64;
          if (a.a_mn) {
#pragma unroll
            for (int i = 0; i < GM / 64; ++i) tc::tma_load_4d(sA + st * A_STAGE + i * 8192, &tmA, it.m0 + 64 * i, kc, it.zi, it.zo, full + st);
          } else {
            tc::tma_load_4d(sA + st * A_STAGE, &tmA, kc, it.m0, it.zi, it.zo, full + st);
          }
          if (a.b_mn) {
#pragma unroll
            for (int i = 0; i < BN / 64; ++i) tc::tma_load_4d(sB + st * B_STAGE + i * 8192, &tmB, it.n0 + 64 * i, kc, it.zi, it.zo, full + st);
          } else {
            tc::tma_load_4d(sB + st * B_STAGE, &tmB, kc, it.n0, it.zi, it.zo, full + st);
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = tc::idesc_bf16_f32(GM, BN) | (a.a_mn ? 1u << 15 : 0u) | (a.b_mn ? 1u << 16 : 0u);
      const uint64_t a_step = a.a_mn ? 128 : 2, b_step = a.b_mn ? 128 : 2;     // 16 K per MMA: 16 rows of 128 B, or 32 B inside a row
      int g = 0, n = 0;                                      // slabs consumed, items done
      for (int w = blockIdx.x; w < a.n_work; w += gridDim.x) {
        const WorkItem it = g_item(a, w, BN);
        if (it.skip) continue;
        const int acc = n & 1;
        tc::mbar_wait(tempty + acc, ((n >> 1) & 1) ^ 1);
        tc::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < it.nkb; ++kb, ++g) {
          const int st = g % NS;
          tc::mbar_wait(full + st, (g / NS) & 1);
          tc::tc_fence_after();
          const uint32_t sa = tc::smem_u32(sA + st * A_STAGE), sb = tc::smem_u32(sB + st * B_STAGE);
          const uint64_t ad = a.a_mn ? tc::smem_desc_mn_sw128(sa, 8192) : tc::smem_desc_k_sw128(sa);
          const uint64_t bd = a.b_mn ? tc::smem_desc_mn_sw128(sb, 8192) : tc::smem_desc_k_sw128(sb);
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4)
            tc::mma_bf16_ss(d_tmem, ad + (uint64_t)k4 * a_step, bd + (uint64_t)k4 * b_step, idesc, (kb | k4) != 0);
          tc::mma_commit(empty + st);
        }
        tc::mma_commit(tfull + acc);
        ++n;
      }
    }
  } else if constexpr (MODE != 0) {
    ce_epilogue<BN, MODE>(a, tmem_base, tfull, tempty, stage_all + (warp & 3) * (32 * 36), warp & 3, lane);
  } else {
    const int q = warp & 3;
    const bool vec = ((a.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.C) & 15) == 0) && (!a.pre || (reinterpret_cast<uintptr_t>(a.pre) & 15) == 0);
    int n = 0;
    for (int w = blockIdx.x; w < a.n_work; w += gridDim.x) {
      const WorkItem it = g_item(a, w, BN);
      if (it.skip) continue;
      const int acc = n & 1;
      tc::mbar_wait(tfull + acc, (n >> 1) & 1);
      tc::tc_fence_after();
      const int row = it.m0 + 32 * q + lane;
      const bool first_split = !split || it.kb0 == 0;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        float v[32];
        tc::tmem_ld32(tmem_base + ((uint32_t)(32 * q) << 16) + acc * BN + c0, v);
        if (c0 + 32 == BN) {                 // accumulator fully read: hand it back to the MMA warp
          tc::tc_fence_before();
          __syncwarp();
          if (lane == 0) tc::mbar_arrive(tempty + acc);
        }
        const int nb = it.n0 + c0;
        if (nb >= a.N) continue;             // warp-uniform
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          float x = v[c];
          if (a.bias && first_split && nb + c < a.N) x += __ldg(a.bias + nb + c);
          v[c] = x * a.scale;
        }
        float* cmat = (a.C2 && nb >= a.n_split ? a.C2 - a.n_split : a.C) + it.zo * a.c_so + it.zi * a.c_si;
        if (a.stage && vec && nb + 32 <= a.N && !a.pre) {          // warp-uniform: full chunk, no pre-activation copy -> coalesced rows
          const int row0 = it.m0 + 32 * q;
          float* cbase = cmat + (long long)row0 * a.ldc + nb;
          if (a.act == 0) epi_chunk_staged<false>(a, v, stage_all + q * (32 * 36), cbase, row0, split);
          else epi_chunk_staged<true>(a, v, stage_all + q * (32 * 36), cbase, row0, split);
          continue;
        }
        if (row >= a.M) continue;
        float* crow = cmat + (long long)row * a.ldc + nb;
        float* prow = a.pre ? a.pre + (long long)row * a.ldc + nb : nullptr;
        if (a.act == 0) epi_chunk<false>(a, v, crow, prow, nb, vec && nb + 32 <= a.N, split);
        else epi_chunk<true>(a, v, crow, prow, nb, vec && nb + 32 <= a.N, split);
      }
      ++n;
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc<2 * BN>(tmem_base);
}

// fp32 [R][C] (row stride ld) -> bf16 TRANSPOSE [C][ldt] (ldt >= R, multiple of 8), through a 32 x 32 smem tile
__global__ void __launch_bounds__(256) to_bf16_t_kernel(const float* __restrict__ x, long long ld, __nv_bfloat16* __restrict__ y, long long ldt,
                                                        int R, int C) {
  __shared__ float tile[32][33];
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    const int r = r0 + j, c = c0 + tx;
    tile[j][tx] = (r < R && c < C) ? x[(long long)r * ld + c] : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const int c = c0 + j, r = r0 + tx;
    if (c < C && r < R) y[(long long)c * ldt + r] = __float2bfloat16_rn(tile[tx][j]);
  }
}

// fp32 [R][C] (row stride ld) -> bf16 [R][ldy]
__global__ void __launch_bounds__(256) to_bf16_ld_kernel(const float* __restrict__ x, long long ld, __nv_bfloat16* __restrict__ y, long long ldy,
                                                         long long R, int C) {
  const long long n = R * (long long)C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C;
    const int c = (int)(i - r * C);
    y[r * ldy + c] = __float2bfloat16_rn(x[r * ld + c]);
  }
}

// out[c] (+)= sum_r x[r][c]   (bias gradient): 32 columns x 8 row groups per CTA, atomics across the row blocks
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ x, long long ld, int R, int C, float* __restrict__ out) {
  __shared__ float red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + tx;
  float s = 0.f;
  if (c < C)
    for (int r = blockIdx.y * 8 + ty; r < R; r += gridDim.y * 8) s += x[(long long)r * ld + c];
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) t += red[j][tx];
    atomicAdd(out + c, t);
  }
}

}  // namespace

// also used by the fused attention kernels of flash_tc.cu
namespace adt {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}
// bf16 row-major [rows][cols] with row stride ld elements; box = [box_rows][64 cols], 128-byte swizzle, zero fill out of bounds
int g_make_map(CUtensorMap* m, const void* base, long long rows, long long cols, long long ld, int box_rows, long long n_inner = 1,
               long long s_inner = 0, long long n_outer = 1, long long s_outer = 0) {
  // (an MN-major operand passes rows = K, cols = M or N and box_rows = 64: 64 x 64 boxes)
  // always 4-D {cols, rows, inner batch, outer batch}; a plain matrix is a batch of one (the batch strides are then never used, but
  // must still be multiples of 16 bytes)
  EncodeTiledFn enc = g_encode();
  if (!enc) return ADT_E_CUDA;
  if (n_inner <= 1 && n_outer <= 1) { s_inner = ld * rows; s_outer = ld * rows; }
  if (s_inner == 0) s_inner = ld * rows;
  if (s_outer == 0) s_outer = s_inner * n_inner;
  cuuint64_t gdim[4] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)(n_inner > 0 ? n_inner : 1), (cuuint64_t)(n_outer > 0 ? n_outer : 1)};
  cuuint64_t gstr[3] = {(cuuint64_t)ld * 2, (cuuint64_t)s_inner * 2, (cuuint64_t)s_outer * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)box_rows, 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? ADT_OK : ADT_E_CUDA;
}
}  // namespace adt

namespace {

template <int BN, int NS, int MODE = 0>
int g_launch(const CUtensorMap& tmA, const CUtensorMap& tmB, GemmTcArgs k, int splits, cudaStream_t s, bool stage = false) {
  k.stage = stage ? 1 : 0;
  const size_t smem = 1024 + (size_t)NS * (GM * 128 + BN * 128) + 256 + (stage ? 4 * 32 * 36 * 4 : 0);
  cudaFuncSetAttribute(gemm_tc_kernel<BN, NS, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k.tiles_n = (k.N + BN - 1) / BN; k.tiles_m = (k.M + GM - 1) / GM;
  k.n_split_k = k.nbatch > 1 ? 1 : splits;
  const long long work = (long long)k.tiles_n * k.tiles_m * splits;
  if (work > 0x7fffffff) return ADT_E_SHAPE;
  k.n_work = (int)work;
  // resident CTAs: the two accumulators take 2 * BN of the 512 TMEM columns, the ring its shared memory
  int per_sm = (int)((227 * 1024) / (smem + 1024));
  if (per_sm > 512 / (2 * BN)) per_sm = 512 / (2 * BN);
  if (per_sm < 1) per_sm = 1;
  const int grid = (int)(work < 148ll * per_sm ? work : 148ll * per_sm);
  gemm_tc_kernel<BN, NS, MODE><<<grid, G_THREADS, smem, s>>>(tmA, tmB, k);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}

// Folds one vocabulary chunk's per-tile (max, sum exp) into the running per-row state; after the last chunk it writes lse[r] and adds
// sum_r (lse[r] - z[r, label[r]]) into the fp64 accumulator (as adt_softmax_ce_fwd does).
__global__ void __launch_bounds__(256) ce_merge_kernel(const float2* __restrict__ part, int ntiles, float2* __restrict__ state,
                                                       const float* __restrict__ zlab, float* __restrict__ lse, double* __restrict__ acc, int R,
                                                       int first, int last) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  double loss = 0.0;
  if (r < R) {
    float m = -INFINITY, s = 0.f;
    if (!first) { const float2 st = state[r]; m = st.x; s = st.y; }
    for (int t = 0; t < ntiles; ++t) {
      const float2 p = part[(long long)t * R + r];
      const float mn = fmaxf(m, p.x);
      s = s * __expf(m - mn) + p.y * __expf(p.x - mn);
      m = mn;
    }
    if (last) {
      const float l = m + logf(s);
      lse[r] = l;
      loss = (double)(l - zlab[r]);
    } else {
      state[r] = make_float2(m, s);
    }
  }
  if (last) {
    for (int o = 16; o; o >>= 1) loss += __shfl_xor_sync(0xffffffffu, loss, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(acc, loss);
  }
}

// Scratch of the fused head for a vocabulary chunk of vc columns (a multiple of 128): bf16 dS [R][vc] (backward), then the forward's
// per-tile partials [vc / 128][R] float2, the running per-row (max, sum exp) and z[r, label[r]].  Each area is 256-byte aligned.
struct CeLayout { long long part, state, zlab, total; };
long long ce_a256(long long b) { return (b + 255) & ~255ll; }
CeLayout ce_layout(long long R, long long vc) {
  CeLayout l;
  l.part = ce_a256(2 * R * vc);
  l.state = l.part + ce_a256(8 * R * (vc / 128));
  l.zlab = l.state + ce_a256(8 * R);
  l.total = l.zlab + ce_a256(4 * R);
  return l;
}
// widest chunk (a multiple of 128, at most V rounded up) whose layout fits in `bytes`; 0 if not even 128 columns fit
long long ce_chunk128(long long R, long long V, long long bytes) {
  const long long vmax = (V + 127) / 128 * 128;
  long long vc = bytes > 12 * R ? (bytes - 12 * R) / (264 * R) * 128 : 0;     // 2 R + 8 R / 128 bytes per column, then the alignment
  if (vc > vmax) vc = vmax;
  while (vc >= 128 && ce_layout(R, vc).total > bytes) vc -= 128;
  return vc >= 128 ? vc : 0;
}

}  // namespace

namespace adt {
int set_error(int code, const char* msg);
}

extern "C" int adt_linear_ce_plan(int32_t R, int32_t V, int32_t H, int64_t scratch_bytes, int32_t* vocab_chunk, int64_t* min_scratch_bytes) {
  if (R <= 0 || V <= 0 || H <= 0) return set_error(ADT_E_SHAPE, "linear_ce_plan: R, V and H must be positive");
  if (min_scratch_bytes) *min_scratch_bytes = ce_layout(R, 128).total;
  const long long vc = ce_chunk128(R, V, scratch_bytes);
  if (vocab_chunk) *vocab_chunk = (int32_t)(vc < V ? vc : V);
  if (!vc) return set_error(ADT_E_SHAPE, "linear_ce_plan: scratch_bytes is below the minimum for one 128-column vocabulary chunk");
  return ADT_OK;
}

namespace {
// shared validation of adt_linear_ce_fwd / _bwd: returns the vocabulary chunk (multiple of 128) or an ADT_E_* code (< 0)
long long ce_check(const adt_linear_ce_args* a, bool bwd) {
  if (a->R <= 0 || a->V <= 0 || a->H <= 0 || a->ldx < a->H || a->ldw < a->H || (a->ldx & 7) || (a->ldw & 7))
    return set_error(ADT_E_SHAPE, "linear_ce: R, V, H must be positive, ldx and ldw multiples of 8 and >= H");
  if (!a->x_bf16 || !a->w_bf16 || !a->labels || !a->lse || !a->scratch || (bwd ? !a->dx || !a->g_w : !a->loss_acc))
    return set_error(ADT_E_SHAPE, "linear_ce: x_bf16, w_bf16, labels, lse, scratch and loss_acc (forward) or dx, g_w (backward) are required");
  if ((reinterpret_cast<uintptr_t>(a->x_bf16) | reinterpret_cast<uintptr_t>(a->w_bf16) | reinterpret_cast<uintptr_t>(a->scratch)) & 15)
    return set_error(ADT_E_ALIGN, "linear_ce: x_bf16, w_bf16 and scratch must be 16-byte aligned");
  const long long vc = ce_chunk128(a->R, a->V, a->scratch_bytes);
  if (!vc) return set_error(ADT_E_SHAPE, "linear_ce: scratch_bytes is below adt_linear_ce_plan's min_scratch_bytes");
  return vc;
}

template <int MODE>
int ce_launch(const adt_linear_ce_args* a, GemmTcArgs k, long long v0, int nc, cudaStream_t s) {
  CUtensorMap tmA, tmB;
  const __nv_bfloat16* w = reinterpret_cast<const __nv_bfloat16*>(a->w_bf16) + v0 * a->ldw;
  if (int e = g_make_map(&tmA, a->x_bf16, a->R, a->H, a->ldx, GM)) return e;
  if (int e = g_make_map(&tmB, w, nc, a->H, a->ldw, 128)) return e;
  k.M = a->R; k.N = nc; k.K = a->H; k.scale = 1.f; k.nbatch = 1; k.batch_inner = 1;
  k.bias = a->bias ? a->bias + v0 : nullptr;
  k.labels = a->labels; k.label_off = (int)v0;
  const int nkb = (a->H + 63) / 64;
  k.kb_per_split = nkb;
  return nkb <= 4 ? g_launch<128, 2, MODE>(tmA, tmB, k, 1, s, MODE == 2)
       : nkb <= 16 ? g_launch<128, 3, MODE>(tmA, tmB, k, 1, s, MODE == 2) : g_launch<128, 6, MODE>(tmA, tmB, k, 1, s, MODE == 2);
}
}  // namespace

extern "C" int adt_linear_ce_fwd(const adt_linear_ce_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  const long long vc = ce_check(a, false);
  if (vc < 0) return (int)vc;
  const CeLayout lay = ce_layout(a->R, vc);
  uint8_t* base = reinterpret_cast<uint8_t*>(a->scratch);
  GemmTcArgs k;
  memset(&k, 0, sizeof(k));
  k.part = reinterpret_cast<float2*>(base + lay.part);
  k.zlab = reinterpret_cast<float*>(base + lay.zlab);
  for (long long v0 = 0; v0 < a->V; v0 += vc) {
    const int nc = (int)(a->V - v0 < vc ? a->V - v0 : vc);
    if (ce_launch<1>(a, k, v0, nc, s)) return set_error(ADT_E_CUDA, "linear_ce_fwd: tcgen05 launch failed");
    ce_merge_kernel<<<(a->R + 255) / 256, 256, 0, s>>>(k.part, (nc + 127) / 128, reinterpret_cast<float2*>(base + lay.state), k.zlab, a->lse, a->loss_acc,
                                                       a->R, v0 == 0, v0 + nc >= a->V);
    if (cudaGetLastError() != cudaSuccess) return set_error(ADT_E_CUDA, "linear_ce_fwd: merge launch failed");
  }
  return ADT_OK;
}

extern "C" int adt_linear_ce_bwd(const adt_linear_ce_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  const long long vc = ce_check(a, true);
  if (vc < 0) return (int)vc;
  __nv_bfloat16* ds = reinterpret_cast<__nv_bfloat16*>(a->scratch);
  GemmTcArgs k;
  memset(&k, 0, sizeof(k));
  k.lse = a->lse; k.coef = a->coef; k.coef_dev = a->coef_dev; k.ds = ds; k.ld_ds = vc;
  const int H = a->H;
  for (long long v0 = 0; v0 < a->V; v0 += vc) {
    const int nc = (int)(a->V - v0 < vc ? a->V - v0 : vc);
    k.g_bias = a->g_bias ? a->g_bias + v0 : nullptr;
    if (ce_launch<2>(a, k, v0, nc, s)) return set_error(ADT_E_CUDA, "linear_ce_bwd: tcgen05 launch failed");
    // dx (+)= dS W[v0 : v0 + nc]   (W read MN-major: no transposed copy)
    adt_gemm_tc_args g;
    memset(&g, 0, sizeof(g));
    g.a_bf16 = ds; g.lda = vc; g.b_bf16 = reinterpret_cast<const __nv_bfloat16*>(a->w_bf16) + v0 * a->ldw; g.ldb = a->ldw; g.b_mn = 1;
    g.c = a->dx; g.ldc = H; g.M = a->R; g.N = H; g.K = nc; g.accumulate = v0 > 0; g.scale = 1.f;
    if (adt_gemm_tc(&g, s_)) return set_error(ADT_E_CUDA, "linear_ce_bwd: dgrad GEMM failed");
    // g_W[v0 : v0 + nc] += dS^T x   (dS and x read MN-major, K = R split across CTAs as LinearFn's wgrad does)
    memset(&g, 0, sizeof(g));
    g.a_bf16 = ds; g.lda = vc; g.a_mn = 1; g.b_bf16 = a->x_bf16; g.ldb = a->ldx; g.b_mn = 1;
    g.c = a->g_w + v0 * H; g.ldc = H; g.M = nc; g.N = H; g.K = a->R; g.accumulate = 1; g.scale = 1.f;
    const int tiles = ((nc + 127) / 128) * ((H + 127) / 128), kspl = 148 / tiles, kmax = (a->R + 63) / 64;
    g.split_k = kspl < 1 ? 1 : kspl < kmax ? kspl : kmax;
    if (adt_gemm_tc(&g, s_)) return set_error(ADT_E_CUDA, "linear_ce_bwd: wgrad GEMM failed");
  }
  return ADT_OK;
}

extern "C" int adt_gemm_tc(const adt_gemm_tc_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  // an MN-major operand is stored [K][ld] with its M (or N) extent contiguous
  const long long a_in = a->a_mn ? a->M : a->K, b_in = a->b_mn ? a->N : a->K;
  if (a->M <= 0 || a->N <= 0 || a->K <= 0 || (a->lda & 7) || (a->ldb & 7) || a->lda < a_in || a->ldb < b_in || (!a->c2 && a->ldc < a->N)) return ADT_E_SHAPE;
  if ((reinterpret_cast<uintptr_t>(a->a_bf16) | reinterpret_cast<uintptr_t>(a->b_bf16)) & 15) return ADT_E_ALIGN;
  if (a->split_k > 1 && (a->act || a->pre)) return ADT_E_SHAPE;      // partial sums are only linear before the activation
  const long long bi = a->batch_inner > 0 ? a->batch_inner : 1, bo = a->batch_outer > 0 ? a->batch_outer : 1;
  const bool batched = bi * bo > 1;
  if (batched && (a->split_k > 1 || a->pre || a->c2 || bi * bo > 65535 || ((a->a_si | a->a_so | a->b_si | a->b_so) & 7) || ((a->c_si | a->c_so) & 3)))
    return ADT_E_SHAPE;
  CUtensorMap tmA, tmB;
  GemmTcArgs k;
  k.C = a->c; k.pre = a->pre; k.bias = a->bias; k.ldc = a->ldc; k.M = a->M; k.N = a->N; k.K = a->K; k.act = a->act; k.accumulate = a->accumulate;
  k.scale = a->scale == 0.f ? 1.f : a->scale;
  k.a_mn = a->a_mn ? 1 : 0; k.b_mn = a->b_mn ? 1 : 0;
  k.C2 = a->c2; k.n_split = a->n_split;
  k.batch_inner = (int)bi; k.nbatch = (int)(bi * bo); k.c_so = a->c_so; k.c_si = a->c_si;
  k.causal_skip = a->causal_skip ? 1 : 0;
  if (k.C2 && (k.n_split <= 0 || (k.n_split & 31) || a->ldc < k.n_split || a->ldc < a->N - k.n_split)) return ADT_E_SHAPE;
  const int nkb = (a->K + 63) / 64;
  int splits = a->split_k > 1 ? (a->split_k < nkb ? a->split_k : nkb) : 1;
  k.kb_per_split = (nkb + splits - 1) / splits;
  splits = (nkb + k.kb_per_split - 1) / k.kb_per_split;
  if (batched) splits = (int)(bi * bo);          // the third work dimension walks the batch instead of K splits
  if (splits > 1 && !a->accumulate) {
    if (cudaMemset2DAsync(a->c, (size_t)a->ldc * 4, 0, (size_t)a->N * 4, (size_t)a->M, s) != cudaSuccess) return ADT_E_CUDA;
  }
  if (k.a_mn) { if (int e = g_make_map(&tmA, a->a_bf16, a->K, a->M, a->lda, 64, bi, a->a_si, bo, a->a_so)) return e; }
  else if (int e = g_make_map(&tmA, a->a_bf16, a->M, a->K, a->lda, GM, bi, a->a_si, bo, a->a_so)) return e;
  // narrow outputs waste less of the tile with 64 columns; wide ones amortise the A slab over 128
  // (256-column tiles were measured SLOWER at the C1 shapes: fewer, longer CTAs, two per SM instead of three)
  const int bn = a->N <= 64 ? 64 : 128;
  if (k.b_mn) { if (int e = g_make_map(&tmB, a->b_bf16, a->K, a->N, a->ldb, 64, bi, a->b_si, bo, a->b_so)) return e; }
  else if (int e = g_make_map(&tmB, a->b_bf16, a->N, a->K, a->ldb, bn, bi, a->b_si, bo, a->b_so)) return e;
  // short K ranges (the H x H layers of a block: 4 slabs) leave the ring idle: a shallow ring lets 2-3 CTAs share an SM, so one CTA's
  // epilogue and prologue overlap another's main loop
  const int slabs = k.kb_per_split;
  // (the output-bound short-K launches also stage their chunks for 128-byte-row stores; two CTAs per SM either way)
  if (bn == 64) return slabs <= 16 ? g_launch<64, 4>(tmA, tmB, k, splits, s, slabs <= 4) : g_launch<64, 6>(tmA, tmB, k, splits, s);
  // (eight epilogue warps -- two per lane quarter -- were measured slower too: 8.5 -> 8.9 ms/step)
  // (a 4-stage ring with one CTA per SM was measured slower: 8.5 -> 10.3 ms/step at C1 -- two resident CTAs hide more latency than a deeper ring)
  return slabs <= 4 ? g_launch<128, 2>(tmA, tmB, k, splits, s, true) : slabs <= 16 ? g_launch<128, 3>(tmA, tmB, k, splits, s) : g_launch<128, 6>(tmA, tmB, k, splits, s);
}

extern "C" int adt_to_bf16_t(const float* x, int64_t ld, void* y_bf16, int64_t ldt, int32_t R, int32_t C, adt_stream_t s_) {
  if (R <= 0 || C <= 0 || ldt < R || ld < C) return ADT_E_SHAPE;
  dim3 grid((C + 31) / 32, (R + 31) / 32);
  to_bf16_t_kernel<<<grid, 256, 0, (cudaStream_t)s_>>>(x, ld, reinterpret_cast<__nv_bfloat16*>(y_bf16), ldt, R, C);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}

extern "C" int adt_to_bf16_ld(const float* x, int64_t ld, void* y_bf16, int64_t ldy, int64_t R, int32_t C, adt_stream_t s_) {
  if (R <= 0 || C <= 0 || ldy < C || ld < C) return ADT_E_SHAPE;
  const long long blocks = (R * (long long)C + 255) / 256;
  to_bf16_ld_kernel<<<(int)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, (cudaStream_t)s_>>>(x, ld, reinterpret_cast<__nv_bfloat16*>(y_bf16), ldy, R, C);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}

extern "C" int adt_colsum(const float* x, int64_t ld, int32_t R, int32_t C, float* out, adt_stream_t s_) {
  if (R <= 0 || C <= 0) return ADT_E_SHAPE;
  int gy = (R + 255) / 256;
  if (gy > 64) gy = 64;
  colsum_kernel<<<dim3((C + 31) / 32, gy), 256, 0, (cudaStream_t)s_>>>(x, ld, R, C, out);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}
