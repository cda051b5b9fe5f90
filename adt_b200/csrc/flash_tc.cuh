// Building blocks shared by the fused tcgen05 attention kernels (flash_tc.cu: dot-product attention; wflash_tc.cu: STOSA-ADT's
// Wasserstein attention): 128-row tiles of bf16 operands read through 4-D TMA maps {column in head, row, head, sequence}, one
// [128 rows x 64 bf16] box with 128-byte swizzle per 64 columns, the tcgen05 products over them and the Philox dropout of one row.
// Everything here is inlined into its kernels; the anonymous namespace gives each translation unit its own copy.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>

#include "common.cuh"
#include "tc.cuh"

namespace adt {

int g_make_map(CUtensorMap* m, const void* base, long long rows, long long cols, long long ld, int box_rows, long long n_inner,
               long long s_inner, long long n_outer, long long s_outer);

namespace {

constexpr int FT = 128;                 // rows of a query / key tile = TMEM lanes = threads
constexpr int BOX = FT * 128;           // one [128 rows x 64 bf16] box
constexpr float LOG2E = 1.4426950408889634f;

struct FlashArgs {
  float* ctx; float* lse;                                   // forward
  const float* lse_in; const float* delta;                  // backward
  float* dq; float* dk; float* dv;
  const int* key_ids;
  int L, H, nh, hd, ks, mask_mode, nstage;
  DropDesc drop;
};

__device__ __forceinline__ uint8_t* align1024(uint8_t* p) {
  return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(p) + 1023) & ~(uintptr_t)1023);
}

// dropout multipliers of keys jb .. jb+31 of row i (Philox counter (base + z L + i) * ceil8(L)/8 + j/8, as attn_row_kernel)
__device__ __forceinline__ void drop32(float (&mv)[32], int i, int jb, bool row_ok, unsigned long long drow, const FlashArgs& a) {
#pragma unroll
  for (int k = 0; k < 32; ++k) mv[k] = 1.f;
  if (!a.drop.enabled || !row_ok) return;
  const int nj = a.mask_mode == 0 ? min(i + 1, a.L) : a.L, lp8 = ((a.L + 7) & ~7) >> 3;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    if (jb + 8 * g >= nj) continue;
    float m8[8];
    drop_mul8_attn(a.drop, drow, lp8, (jb >> 3) + g, m8);
#pragma unroll
    for (int k = 0; k < 8; ++k) mv[8 * g + k] = m8[k];
  }
}

// 32 values of row `r` as bf16 into a [128 rows][128 cols] tile (two 64-column boxes, 128-byte swizzle), columns c0 .. c0+31
__device__ __forceinline__ void st_row32(uint8_t* tile, int r, int c0, const float (&x)[32]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const int cc = (c0 >> 3) + g;
    uint4 o;
    o.x = pack_bf16(x[8 * g], x[8 * g + 1]); o.y = pack_bf16(x[8 * g + 2], x[8 * g + 3]);
    o.z = pack_bf16(x[8 * g + 4], x[8 * g + 5]); o.w = pack_bf16(x[8 * g + 6], x[8 * g + 7]);
    *reinterpret_cast<uint4*>(tile + (cc >> 3) * BOX + r * 128 + (((cc & 7) ^ (r & 7)) << 4)) = o;
  }
}

// one [128 x hd] tile (ks boxes) of rows row0.. of head h of sequence b
__device__ __forceinline__ void load_tile(uint8_t* dst, const CUtensorMap* m, int ks, int row0, int h, int b, uint64_t* bar) {
  for (int c = 0; c < ks; ++c) tc::tma_load_4d(dst + c * BOX, m, 64 * c, row0, h, b, bar);
}

// D (+)= A B^T with both operands K-major [128 rows][hd] tiles, K = hd  (S = q k^T, dP~ = dctx v^T)
__device__ __forceinline__ void mma_kk(uint32_t d, const uint8_t* A, const uint8_t* Bm, int hd) {
  const uint32_t idesc = tc::idesc_bf16_f32(FT, FT), sa = tc::smem_u32(A), sb = tc::smem_u32(Bm);
  for (int k = 0; k < hd / 16; ++k) {
    const uint32_t off = (k >> 2) * BOX;
    tc::mma_bf16_ss(d, tc::smem_desc_k_sw128(sa + off) + 2 * (k & 3), tc::smem_desc_k_sw128(sb + off) + 2 * (k & 3), idesc, k != 0);
  }
}

// D (+)= A B over K = 128 tile rows, N = 64 ks: A is a [128][128] bf16 tile read K-major (a_mn = 0: rows = M) or MN-major (a_mn = 1:
// rows = K); B is a [128 rows = K][hd] tile read MN-major
__device__ __forceinline__ void mma_xn(uint32_t d, const uint8_t* A, int a_mn, const uint8_t* Bm, int ks, bool acc) {
  const uint32_t idesc = tc::idesc_bf16_f32(FT, 64 * ks) | (a_mn ? 1u << 15 : 0u) | (1u << 16), sa = tc::smem_u32(A), sb = tc::smem_u32(Bm);
  const uint64_t bd = tc::smem_desc_mn_sw128(sb, BOX);
  for (int k = 0; k < FT / 16; ++k) {
    const uint64_t ad = a_mn ? tc::smem_desc_mn_sw128(sa, BOX) + 128 * k : tc::smem_desc_k_sw128(sa + (k >> 2) * BOX) + 2 * (k & 3);
    tc::mma_bf16_ss(d, ad, bd + 128 * k, idesc, acc || k != 0);
  }
}

// this thread's row of a fp32 [128 x 64 ks] TMEM accumulator -> out[col0 .. col0 + hd) times s (out NULL: read only, rows >= L)
__device__ __forceinline__ void store_acc(uint32_t t, float* __restrict__ out, int col0, int hd, int ks, float s) {
  for (int c0 = 0; c0 < 64 * ks; c0 += 32) {
    float v[32];
    tc::tmem_ld32(t + c0, v);
    if (!out) continue;
    float* p = out + col0 + c0;
#pragma unroll
    for (int k = 0; k < 32; k += 4)
      if (c0 + k < hd) *reinterpret_cast<float4*>(p + k) = make_float4(v[k] * s, v[k + 1] * s, v[k + 2] * s, v[k + 3] * s);
  }
}

// TMA map of the head-h column block (H / nh columns) of a bf16 [B*L][ld] matrix: {column in head, row, head, sequence}
int head_map(CUtensorMap* m, const __nv_bfloat16* base, int B, int L, int H, int nh, long long ld) {
  const int hd = H / nh;
  return g_make_map(m, base, L, hd, ld, FT, nh, hd, B, (long long)L * ld);
}

}  // namespace
}  // namespace adt
