// K7: full-catalog scoring with fused per-user top-K.
// Replaces `predict(full=True)` + host-side masking/argpartition/sort of the whole score row
// (/root/reference/sasrec/model.py:91-96, sasrec/utils.py:718-731, stosa/trainer.py:604-614).
//
// Exact path (this file, fp32 FFMA tiles): scores never leave the SM; every CTA keeps a sorted top-K list per
// user in shared memory and only [splits][U][K] (score,id) pairs are written; a second kernel merges the splits.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include "../../include/adt_b200.h"
#include "common.cuh"

using namespace adt;

namespace {

constexpr int UT = 64;        // users per CTA
constexpr int KMAX = 64;

struct TopkArgs {
  const float* feats; const float* E; const int* seen_indptr; const int* seen_idx;
  float* part_scores; int* part_ids; float* out_scores; int* out_ids;
  const int* user_mask;                        // optional [U]: only users with a non-zero entry are scored / written
  const int* answers; double* metric_acc;      // optional fused HR/NDCG/MRR epilogue of the merge kernel
  long long part_stride;                       // elements between two splits' lists in part_scores / part_ids (merge kernel)
  float* dense_out; long long dense_ld;        // WRITE_ALL mode: the whole score row [U][dense_ld] (predict(full=True))
  int U, H, n_items, item_offset, K, n_splits;
  const float* bias;                           // BIAS kernels: [n_items] added to every score (local index, like E)
};

// get_full_sort_score (sasrec/utils.py:686-708) for ONE held-out answer per user, accumulated over users:
// acc[0] HIT@5, acc[1] NDCG@5, acc[2] HIT@10, acc[3] NDCG@10, acc[4] MRR (over the returned list), acc[5] #users.
// `first` = 0-based position of the answer in the user's best-first list, or -1.
__device__ __forceinline__ void metric_accumulate(double* acc, int first) {
  atomicAdd(acc + 5, 1.0);
  if (first < 0) return;
  const double g = 1.0 / log2((double)first + 2.0);
  if (first < 5) { atomicAdd(acc + 0, 1.0); atomicAdd(acc + 1, g); }
  if (first < 10) { atomicAdd(acc + 2, 1.0); atomicAdd(acc + 3, g); }
  atomicAdd(acc + 4, 1.0 / ((double)first + 1.0));
}

// first position p in [lo, hi) of the sorted id list with idx[p] >= item
__device__ __forceinline__ int seen_lower_bound(const int* __restrict__ idx, int lo, int hi, int item) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (idx[mid] < item) lo = mid + 1; else hi = mid;
  }
  return lo;
}
// [sb, se) = the part of the user's sorted seen list that falls into this CTA's catalog split (found once per CTA): for
// most (user, split) pairs it is empty and the test costs no memory access at all
__device__ __forceinline__ bool is_seen(const TopkArgs& a, int sb, int se, int item) {
  if (sb >= se) return false;
  const int p = seen_lower_bound(a.seen_idx, sb, se, item);
  return p < se && a.seen_idx[p] == item;
}

// better(a,b): a ranks strictly before b  (score desc, then id asc -- deterministic under exact ties)
__device__ __forceinline__ bool better(float sa, int ia, float sb, int ib) { return sa > sb || (sa == sb && ia < ib); }

// BIAS: scores are <f, e> + bias[i], the bias added once after the full dot product of the tile, before anything compares them;
// the re-score kernel of the tensor-core path adds it after the same sequential fmaf chain, so the two stay bit-identical
template <bool WRITE_ALL, bool BIAS>
__global__ void __launch_bounds__(NT) score_topk_kernel(TopkArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int H = a.H, K = a.K;
  const int ld = H + 4;
  float* Fs = smem;                       // [UT][ld]
  float* Sc = Fs + UT * ld;               // [UT][CHP]
  float* Ws = Sc + UT * CHP;              // staging
  float* Ls = Ws + WS_FLOATS;             // [UT][K] scores
  int* Li = reinterpret_cast<int*>(Ls + UT * K);   // [UT][K] ids
  int* Ln = Li + UT * K;                  // [UT] fill counts
  int* Sb = Ln + UT;                      // [UT] seen-list range of this split
  int* Se = Sb + UT;
  const int split = blockIdx.x, u0 = blockIdx.y * UT;
  const int per = (a.n_items + a.n_splits - 1) / a.n_splits;
  const int it0 = split * per, it1 = min(a.n_items, it0 + per);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;

  if (a.user_mask) {     // fix-up launches of the tensor-core path: almost every tile has nothing to do
    int any = 0;
    for (int i = threadIdx.x; i < UT; i += NT) any |= (u0 + i < a.U && a.user_mask[u0 + i] != 0) ? 1 : 0;
    if (!__syncthreads_or(any)) return;
  }
  load_tile<UT>(Fs, ld, a.feats, H, 0, H, u0, a.U);
  for (int i = threadIdx.x; i < UT; i += NT) {
    Ln[i] = 0;
    int sb = 0, se = 0;
    if (a.seen_indptr && u0 + i < a.U) {
      const int hi = a.seen_indptr[u0 + i + 1];
      sb = seen_lower_bound(a.seen_idx, a.seen_indptr[u0 + i], hi, a.item_offset + it0);
      se = seen_lower_bound(a.seen_idx, sb, hi, a.item_offset + it1);
    }
    Sb[i] = sb;
    Se[i] = se;
  }
  __syncthreads();

  const int nrc = (H + CH - 1) / CH;
  for (int c0 = it0; c0 < it1; c0 += CH) {
    const int ncols = min(CH, it1 - c0);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
    stage_chunk<true, CHP>(Ws, a.E, H, c0, 0, ncols, min(CH, H));
    cp_async_commit();
    for (int rc = 0; rc < nrc; ++rc) {
      if (rc + 1 < nrc) {
        stage_chunk<true, CHP>(Ws + ((rc + 1) & 1) * WS_SLOT, a.E, H, c0, (rc + 1) * CH, ncols, min(CH, H - (rc + 1) * CH));
        cp_async_commit();
        cp_async_wait<1>();
      } else {
        cp_async_wait<0>();
      }
      __syncthreads();
      mma_nt<4>(acc, Fs, ld, rc * CH, Ws + (rc & 1) * WS_SLOT, min(CH, H - rc * CH));
      __syncthreads();
    }
    if constexpr (BIAS) {
      float b[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = c0 + 4 * tx + j < it1 ? __ldg(a.bias + c0 + 4 * tx + j) : 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] += b[j];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
      *reinterpret_cast<float4*>(Sc + (ty + 16 * i) * CHP + 4 * tx) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    __syncthreads();
    if constexpr (WRITE_ALL) {     // predict(full=True): the score tile goes straight to HBM, coalesced along the item axis
      for (int i = threadIdx.x; i < UT * CH; i += NT) {
        const int r = i / CH, c = i - r * CH;
        if (u0 + r < a.U && c < ncols) a.dense_out[(long long)(u0 + r) * a.dense_ld + a.item_offset + c0 + c] = Sc[r * CHP + c];
      }
      __syncthreads();
      continue;
    }
    // selection: warp per user row.  Lanes filter their two columns against the row's K-th best (and the seen list); the
    // survivors are merged into the sorted list IN PARALLEL by rank counting -- every survivor and every list entry
    // computes its position in the merged order ((score desc, id asc) is a strict total order, so positions are unique)
    // and writes itself there.  Cost per merge ~ (#survivors + K) short steps instead of #survivors serial insertions,
    // which matters because a split of a small catalog never gets a warm list.
    for (int r = w; r < UT; r += NT / 32) {
      const int u = u0 + r;
      if (u >= a.U) continue;
      float* ls = Ls + r * K;
      int* li = Li + r * K;
      const int sb = Sb[r], se = Se[r];
#pragma unroll 1
      for (int half = 0; half < 2; ++half) {
        const int col = l + 32 * half;
        const float s = Sc[r * CHP + col];
        const int item = a.item_offset + c0 + col;
        const int n = Ln[r];
        const bool cand = col < ncols && (n < K || better(s, item, ls[K - 1], li[K - 1])) && !is_seen(a, sb, se, item);
        const unsigned ballot = __ballot_sync(0xffffffffu, cand);
        if (ballot == 0u) continue;
        // this lane's list entries (K <= 64: slots l and l + 32), read before anything is overwritten
        const bool h0 = l < n, h1 = l + 32 < n;
        const float e0s = h0 ? ls[l] : 0.f, e1s = h1 ? ls[l + 32] : 0.f;
        const int e0i = h0 ? li[l] : 0, e1i = h1 ? li[l + 32] : 0;
        int pc = 0, p0 = l, p1 = l + 32;      // merged positions of: my survivor, my two list entries
        for (unsigned b = ballot; b; b &= b - 1) {
          const int src = __ffs(b) - 1;
          const float cs = __shfl_sync(0xffffffffu, s, src);
          const int ci = __shfl_sync(0xffffffffu, item, src);
          pc += better(cs, ci, s, item) ? 1 : 0;
          p0 += better(cs, ci, e0s, e0i) ? 1 : 0;
          p1 += better(cs, ci, e1s, e1i) ? 1 : 0;
        }
        if (cand)
          for (int j = 0; j < n; ++j) pc += better(ls[j], li[j], s, item) ? 1 : 0;   // same address in all lanes: broadcast
        __syncwarp();
        if (h0 && p0 < K) { ls[p0] = e0s; li[p0] = e0i; }
        if (h1 && p1 < K) { ls[p1] = e1s; li[p1] = e1i; }
        if (cand && pc < K) { ls[pc] = s; li[pc] = item; }
        if (l == 0) Ln[r] = min(K, n + __popc(ballot));
        __syncwarp();
      }
    }
    __syncthreads();
  }
  if constexpr (WRITE_ALL) return;
  // write this split's lists (sorted, padded with -inf / -1)
  for (int i = threadIdx.x; i < UT * K; i += NT) {
    const int r = i / K, k = i - r * K;
    if (u0 + r < a.U) {
      const bool ok = k < Ln[r];
      const long long o = ((long long)split * a.U + (u0 + r)) * K + k;
      a.part_scores[o] = ok ? Ls[r * K + k] : -INFINITY;
      a.part_ids[o] = ok ? Li[r * K + k] : -1;
    }
  }
}

// warp per user: K-way selection over the n_splits sorted partial lists
__global__ void __launch_bounds__(256) topk_merge_kernel(TopkArgs a) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int u = blockIdx.x * 8 + w;
  if (u >= a.U) return;
  if (a.user_mask && a.user_mask[u] == 0) return;
  const int K = a.K, S = a.n_splits;
  // lane owns splits l, l+32, ... ; head pointer per owned split (S <= 32*8)
  int hp[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) hp[j] = 0;
  const int answer = a.answers ? a.answers[u] : -1;
  int first = -1;
  for (int k = 0; k < K; ++k) {
    float bs = -INFINITY;
    int bi = 0x7fffffff, bj = -1;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int sp = l + 32 * j;
      if (sp < S && hp[j] < K) {
        const long long o = (long long)sp * a.part_stride + (long long)u * K + hp[j];
        const float s = a.part_scores[o];
        const int id = a.part_ids[o];
        if (id >= 0 && better(s, id, bs, bi)) { bs = s; bi = id; bj = j; }
      }
    }
    // warp argmax
    float ws = bs; int wi = bi; int wl = bj >= 0 ? l : -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float os = __shfl_xor_sync(0xffffffffu, ws, o);
      const int oi = __shfl_xor_sync(0xffffffffu, wi, o);
      const int ol = __shfl_xor_sync(0xffffffffu, wl, o);
      if (ol >= 0 && (wl < 0 || better(os, oi, ws, wi))) { ws = os; wi = oi; wl = ol; }
    }
    if (wl == l && bj >= 0) {
#pragma unroll
      for (int j = 0; j < 8; ++j) if (j == bj) hp[j]++;
    }
    if (l == 0) {
      a.out_scores[(long long)u * K + k] = wl >= 0 ? ws : -INFINITY;
      a.out_ids[(long long)u * K + k] = wl >= 0 ? wi : -1;
      if (wl >= 0 && wi == answer && first < 0) first = k;
    }
  }
  if (l == 0 && a.answers && a.metric_acc) metric_accumulate(a.metric_acc, first);
}

// evaluate_loader's candidate ranking (sasrec/utils.py:407-410) without materialising item_embs [U,C,H] or sorting:
// scores[u][c] = <feats[u], E[idx[u][c]]> (idx_stride = 0: one candidate list shared by all users, the 1-D `item_idx` of
// utils.evaluate / evaluate_valid), rank[u] = #{c > 0 : s_c > s_0} = position of column 0 under a stable descending sort.
// Warp per user; lanes stride over the candidates, 128-bit row loads.
struct CandArgs {
  const float* feats; const float* E; const int* idx; float* scores; int* rank; long long idx_stride; int U, H, C, n_rows;
};
__global__ void __launch_bounds__(256) candidate_scores_kernel(CandArgs a) {
  extern __shared__ __align__(16) float cs_smem[];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  const int u = blockIdx.x * 8 + w;
  if (u >= a.U) return;
  float* f = cs_smem + w * a.H;
  for (int h = l; h < a.H; h += 32) f[h] = a.feats[(long long)u * a.H + h];
  __syncwarp();
  const int* ix = a.idx + (long long)u * a.idx_stride;
  float s0 = 0.f;
  int cnt = 0;
  for (int c0 = 0; c0 < a.C; c0 += 32) {
    const int c = c0 + l;
    float s = -INFINITY;
    if (c < a.C) {
      int id = ix[c];
      id = id < 0 ? 0 : (id >= a.n_rows ? a.n_rows - 1 : id);     // ids are validated on the host; never read out of bounds
      const float* e = a.E + (long long)id * a.H;
      float acc = 0.f;
      for (int h = 0; h < a.H; h += 4) {
        const float4 ev = *reinterpret_cast<const float4*>(e + h);
        const float4 fv = *reinterpret_cast<const float4*>(f + h);
        acc = fmaf(fv.x, ev.x, acc); acc = fmaf(fv.y, ev.y, acc); acc = fmaf(fv.z, ev.z, acc); acc = fmaf(fv.w, ev.w, acc);
      }
      s = acc;
      if (a.scores) a.scores[(long long)u * a.C + c] = s;
    }
    if (c0 == 0) s0 = __shfl_sync(0xffffffffu, s, 0);
    cnt += __popc(__ballot_sync(0xffffffffu, c < a.C && c > 0 && s > s0));
  }
  if (l == 0 && a.rank) a.rank[u] = cnt;
}

// sampled-candidate metrics (utils.py:411-427) from the ranks: acc[0] HR@5, [1] NDCG@5, [2] HR@10, [3] NDCG@10, [4] sum 1/(rank+1),
// [5] #users, [6] sum of (C1 - (rank+1)) / (C1 - 1) with the reference's C1 = 1 + C (quirk B7)
__global__ void __launch_bounds__(256) rank_metrics_kernel(const int* __restrict__ rank, int U, int C, double* __restrict__ acc) {
  double v[7] = {0, 0, 0, 0, 0, 0, 0};
  for (int u = blockIdx.x * blockDim.x + threadIdx.x; u < U; u += gridDim.x * blockDim.x) {
    const int r = rank[u];
    const double g = 1.0 / log2((double)r + 2.0);
    if (r < 5) { v[0] += 1.0; v[1] += g; }
    if (r < 10) { v[2] += 1.0; v[3] += g; }
    v[4] += 1.0 / ((double)r + 1.0);
    v[5] += 1.0;
    v[6] += ((double)(1 + C) - (double)(r + 1)) / (double)C;
  }
#pragma unroll
  for (int j = 0; j < 7; ++j) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[j] += __shfl_xor_sync(0xffffffffu, v[j], o);
    if ((threadIdx.x & 31) == 0 && v[j] != 0.0) atomicAdd(acc + j, v[j]);
  }
}

}  // namespace

extern "C" int adt_score_topk(const adt_score_topk_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (a->K <= 0 || a->K > KMAX || a->H > 256 || (a->H & 3) || a->n_splits <= 0 || a->n_splits > 256 || a->U <= 0) return ADT_E_SHAPE;
  TopkArgs k;
  k.feats = a->feats; k.E = a->item_emb; k.seen_indptr = a->seen_indptr; k.seen_idx = a->seen_idx;
  k.part_scores = a->part_scores; k.part_ids = a->part_ids; k.out_scores = a->out_scores; k.out_ids = a->out_ids;
  k.U = a->U; k.H = a->H; k.n_items = a->n_items; k.item_offset = a->item_offset; k.K = a->K; k.n_splits = a->n_splits;
  k.answers = a->answers; k.metric_acc = a->metric_acc; k.dense_out = nullptr; k.dense_ld = 0; k.user_mask = a->user_mask;
  k.part_stride = (long long)a->U * a->K;
  k.bias = a->item_bias;
  const size_t smem = ((size_t)UT * (a->H + 4) + (size_t)UT * CHP + WS_FLOATS + (size_t)UT * a->K * 2 + 3 * UT) * sizeof(float);
  dim3 grid(a->n_splits, (a->U + UT - 1) / UT);
  if (a->item_bias) {
    cudaFuncSetAttribute(score_topk_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    score_topk_kernel<false, true><<<grid, NT, smem, s>>>(k);
  } else {
    cudaFuncSetAttribute(score_topk_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    score_topk_kernel<false, false><<<grid, NT, smem, s>>>(k);
  }
  if (a->out_ids) topk_merge_kernel<<<(a->U + 7) / 8, 256, 0, s>>>(k);
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}

// predict(full=True) (sasrec/model.py:91-96): the whole fp32 score row, same FFMA tiles as the top-K path
extern "C" int adt_score_full(const float* feats, int32_t U, int32_t H, const float* item_emb, int32_t n_items, int32_t item_offset,
                              float* out, int64_t ld, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (H > 256 || (H & 3) || U <= 0 || n_items <= 0 || ld < (int64_t)item_offset + n_items) return ADT_E_SHAPE;
  TopkArgs k;
  memset(&k, 0, sizeof(k));
  k.feats = feats; k.E = item_emb; k.U = U; k.H = H; k.n_items = n_items; k.item_offset = item_offset; k.K = 1;
  const int tiles = (U + UT - 1) / UT;
  int splits = (4 * 148 + tiles - 1) / tiles;
  const int max_splits = (n_items + CH - 1) / CH;
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  // splits must start on a CH boundary only for efficiency, not correctness: `per` is rounded up to CH
  int per = (n_items + splits - 1) / splits;
  per = (per + CH - 1) / CH * CH;
  splits = (n_items + per - 1) / per;
  k.n_splits = splits; k.dense_out = out; k.dense_ld = ld;
  const size_t smem = ((size_t)UT * (H + 4) + (size_t)UT * CHP + WS_FLOATS + (size_t)UT * 2 + 3 * UT) * sizeof(float);
  cudaFuncSetAttribute(score_topk_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  score_topk_kernel<true, false><<<dim3(splits, tiles), NT, smem, s>>>(k);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}

extern "C" int adt_candidate_scores(const adt_candidate_scores_args* a, adt_stream_t s_) {
  if (a->U <= 0 || a->C <= 0 || a->H <= 0 || (a->H & 3) || a->H > 1024 || a->n_rows <= 0) return ADT_E_SHAPE;
  CandArgs c;
  c.feats = a->feats; c.E = a->item_emb; c.idx = a->idx; c.scores = a->scores; c.rank = a->rank;
  c.idx_stride = a->idx_stride; c.U = a->U; c.H = a->H; c.C = a->C; c.n_rows = a->n_rows;
  candidate_scores_kernel<<<(a->U + 7) / 8, 256, (size_t)8 * a->H * sizeof(float), (cudaStream_t)s_>>>(c);
  if (a->rank && a->metric_acc) rank_metrics_kernel<<<min((a->U + 255) / 256, 148), 256, 0, (cudaStream_t)s_>>>(a->rank, a->U, a->C, a->metric_acc);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}

// item-sharded evaluation: merge the all-gathered per-shard lists [n_lists][U][K] (each best first, -1 ids = padding) into the global
// top-K, order (score desc, id asc), with the same fused metric epilogue as adt_score_topk.  list_stride = elements between lists.
extern "C" int adt_topk_merge(const float* scores, const int32_t* ids, int32_t n_lists, int64_t list_stride, int32_t U, int32_t K,
                              float* out_scores, int32_t* out_ids, const int32_t* answers, double* metric_acc, adt_stream_t s_) {
  if (K <= 0 || K > KMAX || n_lists <= 0 || n_lists > 256 || U <= 0) return ADT_E_SHAPE;
  TopkArgs k;
  memset(&k, 0, sizeof(k));
  k.part_scores = const_cast<float*>(scores); k.part_ids = const_cast<int*>(ids); k.out_scores = out_scores; k.out_ids = out_ids;
  k.answers = answers; k.metric_acc = metric_acc; k.part_stride = list_stride; k.U = U; k.K = K; k.n_splits = n_lists;
  topk_merge_kernel<<<(U + 7) / 8, 256, 0, (cudaStream_t)s_>>>(k);
  return cudaGetLastError() == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}
