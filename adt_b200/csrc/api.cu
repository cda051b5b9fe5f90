// C-ABI entry points of libadt_b200.so (see include/adt_b200.h).  Host-side launch logic only.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/adt_b200.h"
#include "kernels_bwd.cuh"
#include "kernels_embed_opt.cuh"
#include "kernels_fwd.cuh"
#include "kernels_generic.cuh"
#include "kernels_stosa.cuh"
#include "kernels_attn_small.cuh"
#include "kernels_rowtile_small.cuh"
#include "kernels_seq.cuh"
#include "block_tc.cuh"

using namespace adt;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, const char* what) {
  snprintf(g_err, sizeof(g_err), fmt, what);
  return code;
}
// the same message slot for the entry points of the other translation units
namespace adt {
int set_error(int code, const char* msg) { return fail(code, "%s", msg); }
}
static int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return ADT_E_CUDA;
  }
  return ADT_OK;
}

// ---- optional per-kernel CUDA-event timing (bench.py's live roofline measurement) -------------------------
namespace {
constexpr int TIMING_MAX = 8192;
struct TimingRec { const char* name; cudaEvent_t a, b; };
bool g_timing_on = false;
int g_timing_n = 0;
TimingRec g_timing[TIMING_MAX];
struct TimingScope {
  int idx; cudaStream_t s;
  TimingScope(const char* name, cudaStream_t s_) : idx(-1), s(s_) {
    if (!g_timing_on || g_timing_n >= TIMING_MAX) return;
    idx = g_timing_n++;
    TimingRec& r = g_timing[idx];
    r.name = name;
    if (!r.a) { cudaEventCreate(&r.a); cudaEventCreate(&r.b); }
    cudaEventRecord(r.a, s);
  }
  ~TimingScope() { if (idx >= 0) cudaEventRecord(g_timing[idx].b, s); }
};
}  // namespace
#define TIMED(name, stream) TimingScope _ts(name, stream)

extern "C" int adt_timing_enable(int on) { g_timing_on = on != 0; g_timing_n = 0; return ADT_OK; }

// Synchronises the device, aggregates the recorded launches by kernel name.  names: '\n'-separated list written into
// names_buf; total_ms[i] / counts[i] per name.  Returns the number of distinct names (<= max_names).
extern "C" int adt_timing_collect(char* names_buf, int buf_len, float* total_ms, int* counts, int max_names) {
  cudaDeviceSynchronize();
  const char* uniq[64];
  int nu = 0;
  for (int i = 0; i < g_timing_n; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g_timing[i].a, g_timing[i].b) != cudaSuccess) continue;
    int j = 0;
    for (; j < nu; ++j) if (uniq[j] == g_timing[i].name || !strcmp(uniq[j], g_timing[i].name)) break;
    if (j == nu) {
      if (nu >= max_names || nu >= 64) continue;
      uniq[nu] = g_timing[i].name; total_ms[nu] = 0.f; counts[nu] = 0; ++nu;
    }
    total_ms[j] += ms; counts[j] += 1;
  }
  int off = 0;
  for (int j = 0; j < nu; ++j) off += snprintf(names_buf + off, off < buf_len ? buf_len - off : 0, "%s\n", uniq[j]);
  g_timing_n = 0;
  return nu;
}

static DropDesc mk_drop(const adt_dropout& d) {
  DropDesc r;
  memset(&r, 0, sizeof(r));
  r.enabled = (d.enabled && d.p > 0.f) ? 1u : 0u;
  double t = floor((double)d.p * 4294967296.0 + 0.5);
  if (t < 0) t = 0;
  if (t > 4294967295.0) t = 4294967295.0;
  r.thr = (uint32_t)t;
  double t16 = floor((double)d.p * 65536.0 + 0.5);
  r.thr16 = (uint32_t)(t16 < 0 ? 0 : (t16 > 65535.0 ? 65535.0 : t16));
  r.scale = 1.0f / (1.0f - d.p);
  r.seed_lo = (uint32_t)(d.seed & 0xffffffffull);
  r.seed_hi = (uint32_t)(d.seed >> 32);
  r.step = d.step;
  r.site = d.site;
  r.base = d.base;
  r.step_dev = d.step_dev;
  return r;
}

static const size_t SMEM_MAX = 227 * 1024 - 2048;   // leave room for the kernels' small static arrays

// rows-per-CTA choice: the preferred tile height (ADT_TM = 32 / 64 / 128, default 64) when the tile set fits, else the next smaller
// `tuned`: per-kernel measured preference used when ADT_TM is not set (C2 shape: mid_bwd is 20 % faster with 128-row tiles -- half
// the weight-gradient atomics -- every other kernel is fastest at 64)
static int pick_tm(size_t row_floats, size_t* bytes, int max_tm = 128, int tuned = 0) {
  static int pref = -1;
  if (pref < 0) { const char* e = getenv("ADT_TM"); pref = e ? atoi(e) : 0; if (pref != 32 && pref != 64 && pref != 128) pref = 0; }
  const int want = pref ? pref : (tuned ? tuned : 64);
  for (int tm = want < max_tm ? want : max_tm; tm >= 32; tm >>= 1) {
    const size_t b = ((size_t)tm * row_floats + WS_FLOATS) * sizeof(float);
    if (b <= SMEM_MAX) {
      *bytes = b;
      return tm;
    }
  }
  return 0;
}

template <class K>
static cudaError_t set_smem(K kern, size_t bytes) {
  return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// Sequences longer than ATTN_TILE_L positions are served by the fused flash attention (flash_tc.cu) alone, up to FLASH_MAX_L
static const int ATTN_TILE_L = 256, FLASH_MAX_L = 2048;
static int check_dims(int B, int L, int H, int nh) {
  if (L > FLASH_MAX_L) return fail(ADT_E_SHAPE, "%s", "unsupported shape: L > 2048 (the longest sequence the fused flash attention serves)");
  if (B <= 0 || L <= 0 || H <= 0 || H > 256 || (H & 3) || nh <= 0 || nh > 8 || H % nh || ((H / nh) & 3))
    return fail(ADT_E_SHAPE, "%s", "unsupported shape: need 0<L<=2048, H%4==0, H<=256, nh<=8, (H/nh)%4==0");
  return ADT_OK;
}
// shapes of an attention core or a block: beyond 256 positions only the flash kernels serve (bf16, head size 16, 32, ..., 128)
static int check_attn_dims(int B, int L, int H, int nh, int precision) {
  if (int e = check_dims(B, L, H, nh)) return e;
  if (L <= ATTN_TILE_L) return ADT_OK;
  if (!precision)
    return fail(ADT_E_SHAPE, "%s", "unsupported shape: L > 256 needs precision 1 (the fp32 attention cores keep whole score rows in shared "
                                  "memory and stop at 256 positions)");
  if ((H / nh) % 16 || H / nh > 128)
    return fail(ADT_E_SHAPE, "%s", "unsupported shape: L > 256 needs a head size H/nh that is a multiple of 16 and at most 128 (fused flash "
                                  "attention)");
  return ADT_OK;
}

// ---- fused flash attention (flash_tc.cu) --------------------------------------------------------------
namespace adt {
int flash_attn_fwd(const __nv_bfloat16* qkv, float* ctx, float* lse, const int* key_ids, int B, int L, int H, int nh, int mask_mode,
                   const DropDesc& d, cudaStream_t s);
int flash_attn_bwd(const __nv_bfloat16* qkv, const __nv_bfloat16* dcb, const float* ctx, const float* dctx, float* delta, const float* lse,
                   const int* key_ids, float* dq, float* dk, float* dv, int B, int L, int H, int nh, int mask_mode, const DropDesc& d,
                   cudaStream_t s);
}
// its area: bf16 [q | k | v] [M][3H] ; backward: + bf16 dctx [M][H] + delta [B][nh][L] fp32.  0 where the flash kernels do not serve
static long long flash_scratch_bytes(int B, int L, int H, int nh, bool bwd) {
  if (L <= ATTN_TILE_L) return 0;
  const long long M = (long long)B * L;
  return 256 + M * 3 * H * 2 + (bwd ? M * H * 2 + M * nh * 4 : 0);
}

// Row-tile kernels are launched with programmatic stream serialization (opt-in with ADT_PDL=1: measured neutral at the C2 shape): each of them calls
// griddepcontrol.launch_dependents on entry and griddepcontrol.wait before it touches activations, so the next kernel's
// prologue (shared-memory carve-up, weight-ring prefetch) overlaps the tail of the current one.
static bool use_pdl() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("ADT_PDL"); v = e ? (atoi(e) != 0) : 0; }
  return v != 0;
}
template <class... Exp, class... Act>
static void launch_pdl(void (*kern)(Exp...), dim3 grid, size_t smem, cudaStream_t stream, Act&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = dim3(NT); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = use_pdl() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kern, static_cast<Exp>(args)...);
}
#define LAUNCH_ONE(K, grid, smem, stream, ...) \
  do { set_smem(K, smem); launch_pdl(K, dim3(grid), smem, stream, __VA_ARGS__); } while (0)

#define LAUNCH_TM(tm, mma, KERN, grid, smem, stream, ...)                                        \
  do {                                                                                           \
    if ((tm) == 128 && !(mma)) LAUNCH_ONE((KERN<128, false>), grid, smem, stream, __VA_ARGS__);   \
    else if ((tm) == 128) LAUNCH_ONE((KERN<128, true>), grid, smem, stream, __VA_ARGS__);         \
    else if ((tm) == 64 && !(mma)) LAUNCH_ONE((KERN<64, false>), grid, smem, stream, __VA_ARGS__); \
    else if ((tm) == 64) LAUNCH_ONE((KERN<64, true>), grid, smem, stream, __VA_ARGS__);           \
    else if (!(mma)) LAUNCH_ONE((KERN<32, false>), grid, smem, stream, __VA_ARGS__);              \
    else LAUNCH_ONE((KERN<32, true>), grid, smem, stream, __VA_ARGS__);                           \
  } while (0)

#define LAUNCH_TM2(tm, mma, KERN, FLAG, grid, smem, stream, ...)                                 \
  do {                                                                                           \
    if ((tm) == 128 && !(mma)) LAUNCH_ONE((KERN<128, FLAG, false>), grid, smem, stream, __VA_ARGS__); \
    else if ((tm) == 128) LAUNCH_ONE((KERN<128, FLAG, true>), grid, smem, stream, __VA_ARGS__);   \
    else if ((tm) == 64 && !(mma)) LAUNCH_ONE((KERN<64, FLAG, false>), grid, smem, stream, __VA_ARGS__); \
    else if ((tm) == 64) LAUNCH_ONE((KERN<64, FLAG, true>), grid, smem, stream, __VA_ARGS__);     \
    else if (!(mma)) LAUNCH_ONE((KERN<32, FLAG, false>), grid, smem, stream, __VA_ARGS__);        \
    else LAUNCH_ONE((KERN<32, FLAG, true>), grid, smem, stream, __VA_ARGS__);                     \
  } while (0)

extern "C" int adt_version(void) { return 200; }

// sizes of every buffer the caller allocates for one training step (the library allocates nothing); see include/adt_b200.h
extern "C" int adt_workspace_bytes(const adt_workspace_query* q, adt_workspace_sizes* out) {
  if (!q || !out) return fail(ADT_E_SHAPE, "%s", "workspace_bytes: null argument");
  if (int e = check_attn_dims(q->B, q->L, q->H, q->nh > 0 ? q->nh : 1, 1)) return e;
  const long long M = (long long)q->B * q->L, H = q->H, nh = q->nh > 0 ? q->nh : 1, nl = q->nl > 0 ? q->nl : 1, f = sizeof(float);
  const long long MH = M * H * f, lse = (long long)q->B * nh * q->L * f;
  // encoder block: q,k,v,ctx,y,h1 + lse + rec ; decoder block: d,q1,k1,v1,ctx1,a,q2,k2,v2,ctx2,c,h1 + 2 lse ; streams x[nl+1], xd[nl+1]
  out->saved = nl * (6 * MH + lse + M * nh * nh * f) + nl * (12 * MH + 2 * lse) + 2 * (nl + 1) * MH + MH /*feats*/ + 2 * M * f;
  // backward: dk,dv,dk2,dv2 + 10 row buffers + denc[nl] + 5 side buffers + cpos,cneg
  out->scratch = 4 * MH + 10 * MH + nl * MH + 5 * MH + 2 * M * f;
  const long long N = 4 * M;
  out->sort_keys = 4 * N * (long long)sizeof(int);                       // keys, vals, keys_tmp, vals_tmp
  out->sort_hist = 256 * ((N + 255) / 256) * (long long)sizeof(int);
  const long long nb = (N + 31) / 32;
  out->scatter_rows = 2 * nb * H * f;                                    // head, tail
  out->scatter_flags = nb * (long long)sizeof(int);
  out->score_part = (long long)(q->n_splits > 0 ? q->n_splits : 1) * q->B * (q->K > 0 ? q->K : 1) * 8;
  // + the attention area of long sequences: packed bf16 [q|k|v] (+ dctx), scores (+ dP) in fp32 and P (+ dS) in bf16, [B*nh][L][Lp]
  // (sequences beyond 256 positions use the flash kernels and their own O(M H) area instead: no L^2 term)
  const long long Lp = (q->L + 7) / 8 * 8, zll = q->L > ATTN_TILE_L ? 0 : M * nh * Lp;
  out->attn_scratch = flash_scratch_bytes(q->B, q->L, q->H, nh, true);
  out->wgrad_scratch = H >= 128 ? 12 * M * H * 2 + 10 * H * H * 2 + 1024 + 4 * M * H * 2 + zll * 12 : 0;   // tcgen05 backward: <= 10 operand slots + weights
  out->fwd_scratch = H >= 128 ? 9 * M * H * 2 + 10 * H * H * 2 + 1024 + 3 * M * H * 2 + zll * 6 : 0;       // decoder block: 7 operands + fp32 h2 + weights
  return ADT_OK;
}
extern "C" const char* adt_last_error(void) { return g_err; }

// ---------------------------------------------------------------------------------------------------------
extern "C" int adt_embed_fwd(const adt_embed_fwd_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (int e = check_dims(a->B, a->L, a->H, 1)) return e;
  const int M = a->B * a->L;
  const long long n = (long long)M * (a->H / 4);
  if (n >= (1ll << 31)) return fail(ADT_E_SHAPE, "%s", "embed_fwd: B*L*H/4 must be < 2^31");
  const long long blocks = (n + 255) / 256;
  const int grid = (int)(blocks < 148 * 32 ? blocks : 148 * 32);
  TIMED("embed_fwd", s);
  embed_fwd_kernel<<<grid, 256, 0, s>>>(a->ids, a->item_emb, a->pos_emb, a->x, M, a->L, a->H, (float)sqrt((double)a->H), mk_drop(a->drop));
  return check_launch("adt_embed_fwd");
}

// shared launch helpers -------------------------------------------------------------------------------------
static bool use_row_small(int H, int mma) {
  static int small = -1;
  if (small < 0) { const char* e = getenv("ADT_ROW_SMALL"); small = e ? (atoi(e) != 0) : 1; }
  return small && mma && H == RS_H;
}

static int launch_pre_fwd(const float* x, const float* ln_w, const float* ln_b, const adt_mha_w& w, float* q, float* k, float* v,
                          float* norm_out, int M, int H, int nh, int kv_from_norm, int mma, cudaStream_t s) {
  if (use_row_small(H, mma)) {
    const size_t sm = PreFwdSmallSmem::TOTAL_BYTES;
    cudaFuncSetAttribute(pre_fwd_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    TIMED("pre_fwd", s);
    pre_fwd_small_kernel<<<(M + 63) / 64, AS_NT, sm, s>>>(x, ln_w, ln_b, w.in_w, w.in_b, q, k, v, norm_out, M, 1.0f / sqrtf((float)(H / nh)),
                                                        kv_from_norm);
    return check_launch("pre_fwd_small");
  }
  size_t smem;
  const int pad = mma ? 8 : 4;
  const int tm = pick_tm(2 * (size_t)(H + pad), &smem);
  if (!tm) return fail(ADT_E_SHAPE, "%s", "pre_fwd: tile does not fit shared memory");
  const float qscale = 1.0f / sqrtf((float)(H / nh));
  const int grid = (M + tm - 1) / tm;
  TIMED("pre_fwd", s);
  LAUNCH_TM(tm, mma, pre_fwd_kernel, grid, smem, s, x, ln_w, ln_b, w.in_w, w.in_b, q, k, v, norm_out, M, H, qscale, kv_from_norm);
  return check_launch("pre_fwd");
}

// short sequences in the bf16 tensor-core mode: one small CTA per (sequence, head) (kernels_attn_small.cuh); ADT_ATTN_SMALL=0 disables
static bool use_attn_small(int L, int hd, int mma) {
  static int v = -1;
  if (v < 0) { const char* e = getenv("ADT_ATTN_SMALL"); v = e ? (atoi(e) != 0) : 1; }
  return v && mma && L <= 64 && (hd == 16 || hd == 32 || hd == 64);
}

static int launch_attn_fwd(const float* q, const float* k, const float* v, float* ctx, float* lse, const int* key_ids, int B, int L,
                           int H, int nh, int mask_mode, const adt_dropout& d, int training, int mma, cudaStream_t s) {
  const int hd = H / nh;
  if (use_attn_small(L, hd, mma)) {
    adt_dropout dd = d;
    if (!training) dd.enabled = 0;
    const DropDesc dr = mk_drop(dd);
    TIMED("attn_fwd", s);
    if (hd == 16) attn_small_fwd_kernel<16><<<B * nh, AS_NT, 0, s>>>(q, k, v, ctx, lse, key_ids, L, H, nh, mask_mode, dr);
    else if (hd == 32) attn_small_fwd_kernel<32><<<B * nh, AS_NT, 0, s>>>(q, k, v, ctx, lse, key_ids, L, H, nh, mask_mode, dr);
    else attn_small_fwd_kernel<64><<<B * nh, AS_NT, 0, s>>>(q, k, v, ctx, lse, key_ids, L, H, nh, mask_mode, dr);
    return check_launch("attn_small_fwd");
  }
  const int pad = mma ? 8 : 4;
  const size_t rowf = (size_t)(hd + pad) + (size_t)(((L + 3) & ~3) + pad);
  size_t smem;
  int tm = pick_tm(rowf, &smem, 64, L > 128 ? 32 : 0);      // long sequences: 32-query tiles measured 24 % faster at L = 200 (C1)
  if (!tm) return fail(ADT_E_SHAPE, "%s", "attn_fwd: tile does not fit shared memory");
  if (L <= 32 && tm == 64) { tm = 32; smem = ((size_t)tm * rowf + WS_FLOATS) * sizeof(float); }
  adt_dropout dd = d;
  if (!training) dd.enabled = 0;
  dim3 grid((L + tm - 1) / tm, nh, B);
  TIMED("attn_fwd", s);
  LAUNCH_TM(tm, mma, attn_fwd_kernel, grid, smem, s, q, k, v, ctx, lse, key_ids, L, H, nh, mask_mode, mk_drop(dd));
  return check_launch("attn_fwd");
}

static int launch_attn_bwd(const float* q, const float* k, const float* v, const float* dctx, const float* lse, const int* key_ids,
                           float* dq, float* dk, float* dv, int B, int L, int H, int nh, int mask_mode, const adt_dropout& d,
                           int mma, cudaStream_t s) {
  const int hd = H / nh;
  if (use_attn_small(L, hd, mma)) {
    const DropDesc dr = mk_drop(d);
    TIMED("attn_bwd", s);
#define ADT_AS_BWD(HD)                                                                                                   \
    do {                                                                                                                 \
      const size_t sm = (size_t)AsBwdSmem<HD>::TOTAL * 2;                                                                \
      cudaFuncSetAttribute(attn_small_bwd_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);             \
      attn_small_bwd_kernel<HD><<<B * nh, AS_NT, sm, s>>>(q, k, v, dctx, lse, key_ids, dq, dk, dv, L, H, nh, mask_mode, dr); \
    } while (0)
    if (hd == 16) ADT_AS_BWD(16);
    else if (hd == 32) ADT_AS_BWD(32);
    else ADT_AS_BWD(64);
#undef ADT_AS_BWD
    return check_launch("attn_small_bwd");
  }
  const int pad = mma ? 8 : 4;
  const size_t rowf = 2 * (size_t)(hd + pad) + 2 * (size_t)(((L + 3) & ~3) + pad);
  size_t smem;
  int tm = pick_tm(rowf, &smem, 64);
  if (!tm) return fail(ADT_E_SHAPE, "%s", "attn_bwd: tile does not fit shared memory");
  if (L <= 32 && tm == 64) { tm = 32; smem = ((size_t)tm * rowf + WS_FLOATS) * sizeof(float); }
  dim3 grid((L + tm - 1) / tm, nh, B);
  if (grid.x > 1) {   // several query tiles accumulate into the same keys -> atomics on zeroed buffers
    cudaMemsetAsync(dk, 0, (size_t)B * L * H * sizeof(float), s);
    cudaMemsetAsync(dv, 0, (size_t)B * L * H * sizeof(float), s);
  }
  TIMED("attn_bwd", s);
  LAUNCH_TM(tm, mma, attn_bwd_kernel, grid, smem, s, q, k, v, dctx, lse, key_ids, dq, dk, dv, L, H, nh, mask_mode, mk_drop(d));
  return check_launch("attn_bwd");
}

// pre_bwd: narrow models (H == 64) in the bf16 mode take the weights-resident 256-thread kernel (ADT_ROW_SMALL=0 disables)
static int launch_pre_bwd(const PreBwdArgs& r, int mma, cudaStream_t s) {
  TIMED("pre_bwd", s);
  if (use_row_small(r.H, mma)) {
    const size_t sm = PreBwdSmall2Smem::TOTAL_BYTES;
    cudaFuncSetAttribute(pre_bwd_small2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    pre_bwd_small2_kernel<<<(r.M + 63) / 64, RS_BWD_NT, sm, s>>>(r);
    return check_launch("pre_bwd_small");
  }
  const int pad = mma ? 8 : 4;
  size_t smem;
  const int tm = pick_tm(4 * (size_t)(r.H + pad), &smem);
  if (!tm) return fail(ADT_E_SHAPE, "%s", "pre_bwd: tile does not fit shared memory");
  LAUNCH_TM(tm, mma, pre_bwd_kernel, (r.M + tm - 1) / tm, smem, s, r);
  return check_launch("pre_bwd");
}

// ---- hoisted weight gradients (H >= 128, bf16 mode): see emit_bf16_tile in common.cuh; ADT_WGRAD_HOIST=0 keeps the in-kernel atomics
static __nv_bfloat16* hoist_ptr(void* scratch, int H, int mma) {
  static int v = -1;
  if (v < 0) { const char* e = getenv("ADT_WGRAD_HOIST"); v = e ? (atoi(e) != 0) : 1; }
  return (v && mma && scratch && H >= 128 && (H & 7) == 0) ? reinterpret_cast<__nv_bfloat16*>(scratch) : nullptr;
}
// gW[n_out][k_out] += dY^T X over M rows; dY = [M][ldy] (first n_out columns), X = [M][ldx] bf16 row-major
static int hoisted_wgrad(const __nv_bfloat16* dy, long long ldy, int n_out, const __nv_bfloat16* x, long long ldx, int k_out, int M, float* gW,
                         cudaStream_t s) {
  adt_gemm_tc_args g;
  memset(&g, 0, sizeof(g));
  g.a_bf16 = dy; g.lda = ldy; g.b_bf16 = x; g.ldb = ldx; g.c = gW; g.ldc = k_out;
  g.M = n_out; g.N = k_out; g.K = M; g.accumulate = 1; g.scale = 1.f; g.a_mn = 1; g.b_mn = 1;
  const int tiles = ((n_out + 127) / 128) * ((k_out + 127) / 128);
  g.split_k = tiles >= 296 ? 1 : 296 / tiles;     // two CTAs per SM (11 K slabs each at C1: the 3-stage ring)
  TIMED("wgrad_tc", s);
  if (int e = adt_gemm_tc(&g, (adt_stream_t)s)) return fail(e, "%s", "hoisted weight gradient (adt_gemm_tc)");
  return ADT_OK;
}

static adt_dropout row_drop(const adt_dropout& d, int training) {
  adt_dropout r = d;
  if (!training) r.enabled = 0;
  return r;
}

// ---- sequence-resident block kernels (kernels_seq.cuh): one CTA per sequence, a whole block per launch ------------------------
// ADT_SEQ_FUSED is a bit mask of the launches served by the sequence-resident kernels: 1 encoder fwd in evaluation mode, 2 decoder
// fwd, 4 encoder bwd, 8 decoder bwd, 16 encoder fwd in training mode too (0 = the row-tile kernels everywhere).  Default = 1: measured
// on B200 at the C2 shape (profiles/r02_seq_kernel_variants.md) the one-launch-per-block kernels win where a block runs alone
// (evaluation: +6 % users/s) but lose inside the training step, whose row-tile kernels overlap across the two streams of the step
// graph while a sequence-resident CTA pins 83-110 KB of shared memory per SM (0.533 ms -> 0.622 ms with all of them on).
enum { SEQ_ENC_FWD = 1, SEQ_DEC_FWD = 2, SEQ_ENC_BWD = 4, SEQ_DEC_BWD = 8, SEQ_ENC_FWD_TRAIN = 16, SEQ_DEFAULT = 1 };
static int seq_mask() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("ADT_SEQ_FUSED"); v = e ? atoi(e) : SEQ_DEFAULT; }
  return v;
}
static bool use_seq(int L, int H, int nh, int mma, int which = SEQ_ENC_FWD) {
  return (seq_mask() & which) && mma && H == RS_H && L <= 64 && (nh == 1 || nh == 2 || nh == 4);
}
extern "C" int adt_seq_kernels_apply(int32_t L, int32_t H, int32_t nh, int32_t precision) { return use_seq(L, H, nh, precision ? 1 : 0) ? 1 : 0; }

static SeqW mk_seqw(const adt_wmirror& m) {
  SeqW w;
  w.base32 = m.base32; w.base16 = reinterpret_cast<const __nv_bfloat16*>(m.bf16);
  return w;
}
#define SEQ_LAUNCH(KERN, nh, grid, smem, stream, arg)                                                                  \
  do {                                                                                                                 \
    if ((nh) == 1) { cudaFuncSetAttribute(KERN<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem)); KERN<64><<<grid, SQ_NT, smem, stream>>>(arg); } \
    else if ((nh) == 2) { cudaFuncSetAttribute(KERN<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem)); KERN<32><<<grid, SQ_NT, smem, stream>>>(arg); } \
    else { cudaFuncSetAttribute(KERN<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem)); KERN<16><<<grid, SQ_NT, smem, stream>>>(arg); } \
  } while (0)

static int seq_enc_fwd(const adt_enc_block_fwd_args* a, cudaStream_t s) {
  EncSeqFwdArgs p;
  memset(&p, 0, sizeof(p));
  p.x = a->x; p.ids = a->ids; p.ln1_g = a->ln1_w; p.ln1_b = a->ln1_b; p.Win = a->attn.in_w; p.bin = a->attn.in_b; p.Wo = a->attn.out_w;
  p.bo = a->attn.out_b; p.ln2_g = a->ln2_w; p.ln2_b = a->ln2_b; p.C1 = a->ffn.w1; p.c1 = a->ffn.b1; p.C2 = a->ffn.w2; p.c2 = a->ffn.b2;
  p.Wsp = a->sparse_w; p.bsp = a->sparse_b;
  const bool save = a->training != 0;
  p.q = save ? a->q : nullptr; p.k = save ? a->k : nullptr; p.v = save ? a->v : nullptr; p.ctx = save ? a->ctx : nullptr;
  p.lse = save ? a->lse : nullptr; p.y = save ? a->y : nullptr; p.h1 = save ? a->h1 : nullptr;
  p.out = a->out; p.out_last = a->out_last; p.rec = a->rec; p.nll_acc = a->nll_acc;
  if (a->nh == 1) { p.rec = nullptr; p.nll_acc = nullptr; }   // a single head has no independence term (main.py:160)
  p.B = a->B; p.L = a->L; p.mask_mode = a->mask_mode; p.qscale = 1.0f / sqrtf((float)(a->H / a->nh));
  adt_dropout da = a->drop_attn;
  if (!a->training) da.enabled = 0;
  p.drop_attn = mk_drop(da); p.drop1 = mk_drop(row_drop(a->drop_ffn1, a->training)); p.drop2 = mk_drop(row_drop(a->drop_ffn2, a->training));
  p.w = mk_seqw(a->wm);
  TIMED("enc_block_fwd", s);
  SEQ_LAUNCH(enc_seq_fwd_kernel, a->nh, a->B, EncSeqFwdSmem::TOTAL_BYTES, s, p);
  return check_launch("enc_seq_fwd");
}

static int seq_enc_bwd(const adt_enc_block_bwd_args* a, cudaStream_t s) {
  EncSeqBwdArgs p;
  memset(&p, 0, sizeof(p));
  p.x = a->x; p.ids = a->ids; p.q = a->q; p.k = a->k; p.v = a->v; p.ctx = a->ctx; p.lse = a->lse; p.y = a->y; p.h1 = a->h1;
  p.ln1_g = a->ln1_w; p.ln1_b = a->ln1_b; p.Win = a->attn.in_w; p.Wo = a->attn.out_w; p.ln2_g = a->ln2_w; p.ln2_b = a->ln2_b;
  p.C1 = a->ffn.w1; p.C2 = a->ffn.w2; p.Wsp = a->sparse_w; p.bsp = a->sparse_b;
  p.dout = a->dout; p.dx_extra = a->dx_extra; p.drec = a->nh > 1 ? a->drec : nullptr; p.nll_coef = a->nh > 1 ? a->nll_coef : 0.f; p.dx = a->dx;
  p.gln1_g = a->g_ln1_w; p.gln1_b = a->g_ln1_b; p.gWin = a->g_attn.in_w; p.gbin = a->g_attn.in_b; p.gWo = a->g_attn.out_w; p.gbo = a->g_attn.out_b;
  p.gln2_g = a->g_ln2_w; p.gln2_b = a->g_ln2_b; p.gC1 = a->g_ffn.w1; p.gc1 = a->g_ffn.b1; p.gC2 = a->g_ffn.w2; p.gc2 = a->g_ffn.b2;
  p.gWsp = a->g_sparse_w; p.gbsp = a->g_sparse_b;
  p.B = a->B; p.L = a->L; p.mask_mode = a->mask_mode; p.qscale = 1.0f / sqrtf((float)(a->H / a->nh));
  p.drop_attn = mk_drop(a->drop_attn); p.drop1 = mk_drop(a->drop_ffn1); p.drop2 = mk_drop(a->drop_ffn2);
  p.w = mk_seqw(a->wm);
  TIMED("enc_block_bwd", s);
  SEQ_LAUNCH(enc_seq_bwd_kernel, a->nh, a->B, SeqBwdSmem::TOTAL_BYTES, s, p);
  return check_launch("enc_seq_bwd");
}

static int seq_dec_fwd(const adt_dec_block_fwd_args* a, cudaStream_t s) {
  DecSeqFwdArgs p;
  memset(&p, 0, sizeof(p));
  p.x = a->x; p.feats = a->feats; p.ids = a->ids; p.ln_g = a->ln_w; p.ln_b = a->ln_b;
  p.Win1 = a->slf.in_w; p.bin1 = a->slf.in_b; p.Wo1 = a->slf.out_w; p.bo1 = a->slf.out_b;
  p.Win2 = a->enc.in_w; p.bin2 = a->enc.in_b; p.Wo2 = a->enc.out_w; p.bo2 = a->enc.out_b;
  p.C1 = a->ffn.w1; p.c1 = a->ffn.b1; p.C2 = a->ffn.w2; p.c2 = a->ffn.b2; p.enc_in = a->enc_in;
  p.d = a->d; p.q1 = a->q1; p.k1 = a->k1; p.v1 = a->v1; p.ctx1 = a->ctx1; p.lse1 = a->lse1; p.a = a->a;
  p.q2 = a->q2; p.k2 = a->k2; p.v2 = a->v2; p.ctx2 = a->ctx2; p.lse2 = a->lse2; p.c = a->c; p.h1 = a->h1;
  p.out = a->out; p.mse_acc = a->mse_acc;
  p.B = a->B; p.L = a->L; p.mask_mode = a->mask_mode; p.qscale = 1.0f / sqrtf((float)(a->H / a->nh));
  adt_dropout ds = a->drop_slf, de = a->drop_enc;
  if (!a->training) { ds.enabled = 0; de.enabled = 0; }
  p.drop_slf = mk_drop(ds); p.drop_enc = mk_drop(de);
  p.drop1 = mk_drop(row_drop(a->drop_ffn1, a->training)); p.drop2 = mk_drop(row_drop(a->drop_ffn2, a->training));
  p.w = mk_seqw(a->wm);
  if (a->phase != 2) {
    TIMED("dec_block_fwd_p1", s);
    SEQ_LAUNCH(dec_seq_fwd1_kernel, a->nh, a->B, DecSeqFwd1Smem::TOTAL_BYTES, s, p);
    if (int e = check_launch("dec_seq_fwd1")) return e;
  }
  if (a->phase != 1) {
    TIMED("dec_block_fwd_p2", s);
    SEQ_LAUNCH(dec_seq_fwd2_kernel, a->nh, a->B, DecSeqFwd2Smem::TOTAL_BYTES, s, p);
    if (int e = check_launch("dec_seq_fwd2")) return e;
  }
  return ADT_OK;
}

static int seq_dec_bwd(const adt_dec_block_bwd_args* a, cudaStream_t s) {
  DecSeqBwdArgs p;
  memset(&p, 0, sizeof(p));
  p.x = a->x; p.feats = a->feats; p.ids = a->ids;
  p.d = a->d; p.q1 = a->q1; p.k1 = a->k1; p.v1 = a->v1; p.ctx1 = a->ctx1; p.lse1 = a->lse1; p.a = a->a;
  p.q2 = a->q2; p.k2 = a->k2; p.v2 = a->v2; p.ctx2 = a->ctx2; p.lse2 = a->lse2; p.c = a->c; p.h1 = a->h1;
  p.out = a->out; p.enc_in = a->enc_in; p.mse_coef = a->mse_coef;
  p.ln_g = a->ln_w; p.ln_b = a->ln_b; p.Win1 = a->slf.in_w; p.Wo1 = a->slf.out_w; p.Win2 = a->enc.in_w; p.Wo2 = a->enc.out_w;
  p.C1 = a->ffn.w1; p.C2 = a->ffn.w2;
  p.dout = a->dout; p.denc = a->denc; p.dd = a->dd; p.dctx1 = a->dctx; p.dfeats = a->dfeats; p.dx = a->dx;
  p.gln_g = a->g_ln_w; p.gln_b = a->g_ln_b; p.gWin1 = a->g_slf.in_w; p.gbin1 = a->g_slf.in_b; p.gWo1 = a->g_slf.out_w; p.gbo1 = a->g_slf.out_b;
  p.gWin2 = a->g_enc.in_w; p.gbin2 = a->g_enc.in_b; p.gWo2 = a->g_enc.out_w; p.gbo2 = a->g_enc.out_b;
  p.gC1 = a->g_ffn.w1; p.gc1 = a->g_ffn.b1; p.gC2 = a->g_ffn.w2; p.gc2 = a->g_ffn.b2;
  p.B = a->B; p.L = a->L; p.mask_mode = a->mask_mode; p.qscale = 1.0f / sqrtf((float)(a->H / a->nh));
  p.drop_slf = mk_drop(a->drop_slf); p.drop_enc = mk_drop(a->drop_enc); p.drop1 = mk_drop(a->drop_ffn1); p.drop2 = mk_drop(a->drop_ffn2);
  p.w = mk_seqw(a->wm);
  if (a->phase != 1) {
    TIMED("dec_block_bwd_p2", s);
    SEQ_LAUNCH(dec_seq_bwd2_kernel, a->nh, a->B, SeqBwdSmem::TOTAL_BYTES, s, p);
    if (int e = check_launch("dec_seq_bwd2")) return e;
  }
  if (a->phase != 2) {
    TIMED("dec_block_bwd_p1", s);
    SEQ_LAUNCH(dec_seq_bwd1_kernel, a->nh, a->B, SeqBwdSmem::TOTAL_BYTES, s, p);
    if (int e = check_launch("dec_seq_bwd1")) return e;
  }
  return ADT_OK;
}


static int blk_attn_fwd(const float* q, const float* k, const float* v, float* ctx, float* lse, const int* ids, int B, int L, int H, int nh,
                        int mask_mode, const adt_dropout& d, int training, int precision, void* area, void* flash, cudaStream_t s);
static int blk_attn_bwd(const float* q, const float* k, const float* v, const float* ctx, const float* dctx, const float* lse, const int* ids,
                        float* dq, float* dk, float* dv, int B, int L, int H, int nh, int mask_mode, const adt_dropout& d, int precision, void* area,
                        void* flash, cudaStream_t s);
// ---- tcgen05 forward path for wide models (block_tc.cuh); ADT_FWD_TC=0 keeps the row-tile kernels ---------------------------------
static bool use_fwd_tc(const void* scratch, int M, int H, int nh, int mma) {
  static int v = -1;
  if (v < 0) { const char* e = getenv("ADT_FWD_TC"); v = e ? (atoi(e) != 0) : 1; }
  return v && mma && scratch && H >= 128 && H <= 256 && (H & 7) == 0 && M >= 512 && nh <= 8;
}
struct TcScratch {
  __nv_bfloat16* base; long long mh; __nv_bfloat16* wb;     // M*H elements per operand; weights after 9 operands
  __nv_bfloat16* op(int i) const { return base + i * mh; }
};
static TcScratch mk_tcs(void* p, int M, int H) {
  TcScratch t;
  t.base = reinterpret_cast<__nv_bfloat16*>(p); t.mh = (long long)M * H; t.wb = t.base + 9 * t.mh;
  return t;
}
static int ew_grid(long long n4) { const long long b = (n4 + 255) / 256; return (int)(b < 148 * 16 ? (b > 0 ? b : 1) : 148 * 16); }
static int row_grid(int M) { const int b = (M + 7) / 8; return b < 148 * 8 ? b : 148 * 8; }
// bf16 copy of a weight: from the mirror when the caller keeps one, else converted into `dst`
static const __nv_bfloat16* tc_weight(const float* W, long long n, const adt_wmirror& wm, __nv_bfloat16* dst, cudaStream_t s) {
  if (wm.bf16 && wm.base32) return reinterpret_cast<const __nv_bfloat16*>(wm.bf16) + (W - wm.base32);
  cast_bf16_kernel<<<ew_grid(n / 4), 256, 0, s>>>(W, dst, n / 4);
  return dst;
}
static void tc_cast(const float* x, __nv_bfloat16* dst, long long n, cudaStream_t s) { cast_bf16_kernel<<<ew_grid(n / 4), 256, 0, s>>>(x, dst, n / 4); }
// c (and c2 for columns >= n_split) = (A W^T + bias) * scale, optionally added to what c holds
static int tc_linear(const __nv_bfloat16* A, const __nv_bfloat16* W, const float* bias, float* c, float* c2, int n_split, int M, int N, int K,
                     float scale, int accumulate, cudaStream_t s) {
  adt_gemm_tc_args g;
  memset(&g, 0, sizeof(g));
  g.a_bf16 = A; g.lda = K; g.b_bf16 = W; g.ldb = K; g.c = c; g.ldc = c2 ? n_split : N; g.bias = bias;
  g.M = M; g.N = N; g.K = K; g.scale = scale; g.accumulate = accumulate; g.c2 = c2; g.n_split = n_split;
  TIMED("linear_tc", s);
  if (int e = adt_gemm_tc(&g, (adt_stream_t)s)) return fail(e, "%s", "tcgen05 forward path (adt_gemm_tc)");
  return ADT_OK;
}
// shared tail of both blocks: h1 = z C1^T + c1 (saved) ; a = relu(h1 m1) ; h2 = a C2^T + c2 ; block output
static int tc_ffn_out(const TcScratch& t, const __nv_bfloat16* zb, int a_op, int h2_op, const adt_ffn_w& ffn, const __nv_bfloat16* C1b,
                      const __nv_bfloat16* C2b, float* h1, const adt_dropout& d1, const adt_dropout& d2, int training, RowOutArgs o, int M,
                      int H, cudaStream_t s) {
  if (int e = tc_linear(zb, C1b, ffn.b1, h1, nullptr, 0, M, H, H, 1.f, 0, s)) return e;
  { TIMED("row_tc", s); relu_drop_cast_kernel<<<ew_grid((long long)M * H / 4), 256, 0, s>>>(h1, t.op(a_op), (long long)M * H / 4, mk_drop(row_drop(d1, training))); }
  float* h2 = reinterpret_cast<float*>(t.op(h2_op));
  if (int e = tc_linear(t.op(a_op), C2b, ffn.b2, h2, nullptr, 0, M, H, H, 1.f, 0, s)) return e;
  o.h2 = h2; o.M = M; o.H = H; o.drop2 = mk_drop(row_drop(d2, training));
  { TIMED("row_tc", s); row_out_kernel<<<row_grid(M), 256, 0, s>>>(o); }
  return check_launch("tcgen05 forward path");
}

static int tc_enc_fwd(const adt_enc_block_fwd_args* a, cudaStream_t s) {
  const int M = a->B * a->L, H = a->H;
  const TcScratch t = mk_tcs(a->tc_scratch, M, H);
  const long long hh = (long long)H * H;
  const float qscale = 1.0f / sqrtf((float)(H / a->nh));
  if (a->phase != 2) {
    const __nv_bfloat16* Winb = tc_weight(a->attn.in_w, 3 * hh, a->wm, t.wb, s);
    RowLnArgs r;
    memset(&r, 0, sizeof(r));
    r.x = a->x; r.g = a->ln1_w; r.b = a->ln1_b; r.yb = t.op(0); r.xb = t.op(1); r.M = M; r.H = H;
    { TIMED("row_tc", s); row_ln_cast_kernel<<<row_grid(M), 256, 0, s>>>(r); }
    // q = (LN1(x) Wq^T + bq) * scale ; [k | v] = x [Wk; Wv]^T + [bk | bv]
    if (int e = tc_linear(t.op(0), Winb, a->attn.in_b, a->q, nullptr, 0, M, H, H, qscale, 0, s)) return e;
    if (int e = tc_linear(t.op(1), Winb + hh, a->attn.in_b + H, a->k, a->v, H, M, 2 * H, H, 1.f, 0, s)) return e;
    if (int e = blk_attn_fwd(a->q, a->k, a->v, a->ctx, a->lse, a->ids, a->B, a->L, H, a->nh, a->mask_mode, a->drop_attn, a->training, a->precision,
                             t.wb + 10 * hh, a->attn_scratch, s))
      return e;
    if (a->phase == 1) return ADT_OK;
  }
  const __nv_bfloat16* Wob = tc_weight(a->attn.out_w, hh, a->wm, t.wb + 3 * hh, s);
  const __nv_bfloat16* C1b = tc_weight(a->ffn.w1, hh, a->wm, t.wb + 4 * hh, s);
  const __nv_bfloat16* C2b = tc_weight(a->ffn.w2, hh, a->wm, t.wb + 5 * hh, s);
  // y = LN1(x) + ctx Wo^T + bo : LN1(x) is written into y, the out-projection accumulates on top
  RowLnArgs r;
  memset(&r, 0, sizeof(r));
  r.x = a->x; r.g = a->ln1_w; r.b = a->ln1_b; r.y = a->y; r.M = M; r.H = H;
  { TIMED("row_tc", s); row_ln_cast_kernel<<<row_grid(M), 256, 0, s>>>(r); }
  tc_cast(a->ctx, t.op(2), (long long)M * H, s);
  if (a->rec || a->nll_acc) {
    TIMED("row_tc", s);
    sparse_head_fwd_kernel<<<row_grid(M), 256, 0, s>>>(a->ctx, a->sparse_w, a->sparse_b, a->rec, a->nll_acc, M, H, a->nh);
  }
  if (int e = tc_linear(t.op(2), Wob, a->attn.out_b, a->y, nullptr, 0, M, H, H, 1.f, 1, s)) return e;
  memset(&r, 0, sizeof(r));
  r.x = a->y; r.g = a->ln2_w; r.b = a->ln2_b; r.yb = t.op(3); r.M = M; r.H = H;
  { TIMED("row_tc", s); row_ln_cast_kernel<<<row_grid(M), 256, 0, s>>>(r); }
  RowOutArgs o;
  memset(&o, 0, sizeof(o));
  o.u = a->y; o.ln_g = a->ln2_w; o.ln_b = a->ln2_b; o.ids = a->ids; o.out = a->out; o.is_dec = 0;
  return tc_ffn_out(t, t.op(3), 4, 5, a->ffn, C1b, C2b, a->h1, a->drop_ffn1, a->drop_ffn2, a->training, o, M, H, s);
}

static int tc_dec_fwd(const adt_dec_block_fwd_args* a, cudaStream_t s) {
  const int M = a->B * a->L, H = a->H;
  const TcScratch t = mk_tcs(a->tc_scratch, M, H);
  const long long hh = (long long)H * H;
  const float qscale = 1.0f / sqrtf((float)(H / a->nh));
  if (a->phase != 2) {
    const __nv_bfloat16* W1b = tc_weight(a->slf.in_w, 3 * hh, a->wm, t.wb, s);
    RowLnArgs r;
    memset(&r, 0, sizeof(r));
    r.x = a->x; r.g = a->ln_w; r.b = a->ln_b; r.y = a->d; r.yb = t.op(0); r.M = M; r.H = H;
    { TIMED("row_tc", s); row_ln_cast_kernel<<<row_grid(M), 256, 0, s>>>(r); }
    if (int e = tc_linear(t.op(0), W1b, a->slf.in_b, a->q1, nullptr, 0, M, H, H, qscale, 0, s)) return e;
    if (int e = tc_linear(t.op(0), W1b + hh, a->slf.in_b + H, a->k1, a->v1, H, M, 2 * H, H, 1.f, 0, s)) return e;
    if (int e = blk_attn_fwd(a->q1, a->k1, a->v1, a->ctx1, a->lse1, a->ids, a->B, a->L, H, a->nh, a->mask_mode, a->drop_slf, a->training, a->precision,
                             t.wb + 10 * hh, a->attn_scratch, s))
      return e;
    if (a->phase == 1) return ADT_OK;
  }
  const __nv_bfloat16* Wo1b = tc_weight(a->slf.out_w, hh, a->wm, t.wb + 3 * hh, s);
  const __nv_bfloat16* W2b = tc_weight(a->enc.in_w, 3 * hh, a->wm, t.wb + 4 * hh, s);
  const __nv_bfloat16* Wo2b = tc_weight(a->enc.out_w, hh, a->wm, t.wb + 7 * hh, s);
  const __nv_bfloat16* C1b = tc_weight(a->ffn.w1, hh, a->wm, t.wb + 8 * hh, s);
  const __nv_bfloat16* C2b = tc_weight(a->ffn.w2, hh, a->wm, t.wb + 9 * hh, s);
  // a = ctx1 Wo1^T + bo1 ; q2 = (a Wq2^T + bq2) * scale ; [k2 | v2] from the encoder features
  tc_cast(a->ctx1, t.op(1), (long long)M * H, s);
  if (int e = tc_linear(t.op(1), Wo1b, a->slf.out_b, a->a, nullptr, 0, M, H, H, 1.f, 0, s)) return e;
  tc_cast(a->a, t.op(2), (long long)M * H, s);
  tc_cast(a->feats, t.op(3), (long long)M * H, s);
  if (int e = tc_linear(t.op(2), W2b, a->enc.in_b, a->q2, nullptr, 0, M, H, H, qscale, 0, s)) return e;
  if (int e = tc_linear(t.op(3), W2b + hh, a->enc.in_b + H, a->k2, a->v2, H, M, 2 * H, H, 1.f, 0, s)) return e;
  if (int e = blk_attn_fwd(a->q2, a->k2, a->v2, a->ctx2, a->lse2, a->ids, a->B, a->L, H, a->nh, a->mask_mode, a->drop_enc, a->training, a->precision,
                           t.wb + 10 * hh, a->attn_scratch, s))
    return e;
  // c = ctx2 Wo2^T + bo2 ; out = (d + FFN(c) + c) * keep
  tc_cast(a->ctx2, t.op(4), (long long)M * H, s);
  if (int e = tc_linear(t.op(4), Wo2b, a->enc.out_b, a->c, nullptr, 0, M, H, H, 1.f, 0, s)) return e;
  tc_cast(a->c, t.op(5), (long long)M * H, s);
  RowOutArgs o;
  memset(&o, 0, sizeof(o));
  o.u = a->c; o.resid = a->d; o.ids = a->ids; o.enc_in = a->enc_in; o.out = a->out; o.acc = a->mse_acc; o.is_dec = 1;
  return tc_ffn_out(t, t.op(5), 6, 7, a->ffn, C1b, C2b, a->h1, a->drop_ffn1, a->drop_ffn2, a->training, o, M, H, s);
}

// ---- tcgen05 backward path for wide models (block_tc.cuh); ADT_BWD_TC=0 keeps the row-tile kernels (with hoisted weight gradients) -----
static bool use_bwd_tc(const void* scratch, int M, int H, int nh, int mma) {
  static int v = -1;
  if (v < 0) { const char* e = getenv("ADT_BWD_TC"); v = e ? (atoi(e) != 0) : 1; }
  return v && mma && scratch && H >= 128 && H <= 256 && (H & 7) == 0 && M >= 512 && nh <= 8 && ((H / nh) & 31) == 0;
}
struct TcBwdScratch {
  __nv_bfloat16* base; long long mh; __nv_bfloat16* wb;     // 12 operand slots of M*H bf16, then the bf16 weights
  __nv_bfloat16* op(int i) const { return base + i * mh; }
  float* f32(int i) const { return reinterpret_cast<float*>(base + i * mh); }   // an fp32 [M,H] matrix takes slots i, i+1
};
static TcBwdScratch mk_tcb(void* p, int M, int H) {
  TcBwdScratch t;
  t.base = reinterpret_cast<__nv_bfloat16*>(p); t.mh = (long long)M * H; t.wb = t.base + 12 * t.mh;
  return t;
}
static int rows_grid2(int M) { const int b = (M + 7) / 8; return b < 148 * 8 ? b : 148 * 8; }
// c (+)= A W : A bf16 [M][lda] (first Kred columns), W bf16 [Kred][N_out] row-major read MN-major
static int tc_dgrad(const __nv_bfloat16* A, long long lda, int Kred, const __nv_bfloat16* W, int N_out, float* c, int accumulate, int M, cudaStream_t s) {
  adt_gemm_tc_args g;
  memset(&g, 0, sizeof(g));
  g.a_bf16 = A; g.lda = lda; g.b_bf16 = W; g.ldb = N_out; g.b_mn = 1; g.c = c; g.ldc = N_out;
  g.M = M; g.N = N_out; g.K = Kred; g.scale = 1.f; g.accumulate = accumulate;
  TIMED("dgrad_tc", s);
  if (int e = adt_gemm_tc(&g, (adt_stream_t)s)) return fail(e, "%s", "tcgen05 backward path (dgrad)");
  return ADT_OK;
}
static void tc_pack(const float* s0, float sc0, float* gb0, const float* s1, float* gb1, const float* s2, float* gb2, __nv_bfloat16* dst, long long ld,
                    int M, int H, cudaStream_t s) {
  RowPackArgs p;
  memset(&p, 0, sizeof(p));
  p.src[0] = s0; p.scale[0] = sc0; p.gb[0] = gb0; p.src[1] = s1; p.scale[1] = 1.f; p.gb[1] = gb1; p.src[2] = s2; p.scale[2] = 1.f; p.gb[2] = gb2;
  p.n = s2 ? 3 : (s1 ? 2 : 1); p.dst = dst; p.ld = ld; p.M = M; p.H = H;
  TIMED("row_tc", s);
  row_pack_kernel<<<rows_grid2(M), 256, 0, s>>>(p);
}
// ---- attention of long sequences as strided-batch tcgen05 GEMMs (block_tc.cuh); ADT_ATTN_TC=0 keeps the generic row-tile attention ------
static bool use_attn_tc(int B, int L, int H, int nh) {
  static int v = -1;
  if (v < 0) { const char* e = getenv("ADT_ATTN_TC"); v = e ? (atoi(e) != 0) : 1; }
  return v && L > 64 && L <= 256 && ((H / nh) & 7) == 0 && (long long)B * nh <= 65535;
}
static int attn_rows_grid(long long rows) { const long long b = (rows + 7) / 8; return (int)(b < 148 * 16 ? b : 148 * 16); }
static uint8_t* align256(void* p) { return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(p) + 255) & ~(uintptr_t)255); }
struct AttnWs {
  __nv_bfloat16* qkv; __nv_bfloat16* dcb; float* S; float* dP; __nv_bfloat16* Pb; __nv_bfloat16* dSb; long long Lp;
};
static AttnWs mk_attn_ws(void* area, int M, int H, int nh, int L, bool bwd) {
  AttnWs w;
  w.Lp = (L + 7) / 8 * 8;
  const long long zll = (long long)M * nh * w.Lp;          // Z * L * Lp
  uint8_t* p = align256(area);
  w.qkv = reinterpret_cast<__nv_bfloat16*>(p); p += (long long)M * 3 * H * 2;
  w.dcb = reinterpret_cast<__nv_bfloat16*>(p); if (bwd) p += (long long)M * H * 2;
  w.S = reinterpret_cast<float*>(p); p += zll * 4;
  w.dP = reinterpret_cast<float*>(p); if (bwd) p += zll * 4;
  w.Pb = reinterpret_cast<__nv_bfloat16*>(p); p += zll * 2;
  w.dSb = reinterpret_cast<__nv_bfloat16*>(p);
  return w;
}
static int tc_bgemm(const __nv_bfloat16* A, long long lda, long long a_so, long long a_si, int a_mn, const __nv_bfloat16* Bm, long long ldb,
                    long long b_so, long long b_si, int b_mn, float* C, long long ldc, long long c_so, long long c_si, int M, int N, int K, int nh,
                    int B, cudaStream_t s, int causal_skip = 0) {
  adt_gemm_tc_args g;
  memset(&g, 0, sizeof(g));
  g.a_bf16 = A; g.lda = lda; g.a_so = a_so; g.a_si = a_si; g.a_mn = a_mn; g.b_bf16 = Bm; g.ldb = ldb; g.b_so = b_so; g.b_si = b_si; g.b_mn = b_mn;
  g.c = C; g.ldc = ldc; g.c_so = c_so; g.c_si = c_si; g.M = M; g.N = N; g.K = K; g.scale = 1.f; g.batch_inner = nh; g.batch_outer = B; g.causal_skip = causal_skip;
  TIMED("attn_gemm_tc", s);
  if (int e = adt_gemm_tc(&g, (adt_stream_t)s)) return fail(e, "%s", "tcgen05 attention (batched adt_gemm_tc)");
  return ADT_OK;
}
static int tc_attn_fwd(const float* q, const float* k, const float* v, float* ctx, float* lse, const int* key_ids, int B, int L, int H, int nh,
                       int mask_mode, const adt_dropout& d, int training, void* area, cudaStream_t s) {
  const int M = B * L, hd = H / nh;
  const AttnWs w = mk_attn_ws(area, M, H, nh, L, false);
  const long long Lp = w.Lp, q_so = (long long)L * 3 * H, s_so = (long long)nh * L * Lp, s_si = (long long)L * Lp;
  tc_pack(q, 1.f, nullptr, k, nullptr, v, nullptr, w.qkv, 3 * H, M, H, s);
  if (int e = tc_bgemm(w.qkv, 3 * H, q_so, hd, 0, w.qkv + H, 3 * H, q_so, hd, 0, w.S, Lp, s_so, s_si, L, L, hd, nh, B, s, mask_mode == 0)) return e;   // S = q k^T
  AttnRowArgs r;
  memset(&r, 0, sizeof(r));
  r.S = w.S; r.lse_out = lse; r.Pb = w.Pb; r.key_ids = key_ids; r.Z = B * nh; r.L = L; r.Lp = (int)Lp; r.nh = nh; r.mask_mode = mask_mode; r.bwd = 0;
  r.drop = mk_drop(row_drop(d, training));
  { TIMED("attn_row_tc", s); attn_row_kernel<<<attn_rows_grid(B * nh * L), 256, 0, s>>>(r); }
  // ctx = P v  (v read MN-major from the packed copy)
  if (int e = tc_bgemm(w.Pb, Lp, s_so, s_si, 0, w.qkv + 2 * H, 3 * H, q_so, hd, 1, ctx, H, (long long)L * H, hd, L, hd, L, nh, B, s)) return e;
  return check_launch("tcgen05 attention fwd");
}
static int tc_attn_bwd(const float* q, const float* k, const float* v, const float* dctx, const float* lse, const int* key_ids, float* dq, float* dk,
                       float* dv, int B, int L, int H, int nh, int mask_mode, const adt_dropout& d, void* area, cudaStream_t s) {
  const int M = B * L, hd = H / nh;
  const AttnWs w = mk_attn_ws(area, M, H, nh, L, true);
  const long long Lp = w.Lp, q_so = (long long)L * 3 * H, s_so = (long long)nh * L * Lp, s_si = (long long)L * Lp, c_so = (long long)L * H;
  tc_pack(q, 1.f, nullptr, k, nullptr, v, nullptr, w.qkv, 3 * H, M, H, s);
  tc_cast(dctx, w.dcb, (long long)M * H, s);
  if (int e = tc_bgemm(w.qkv, 3 * H, q_so, hd, 0, w.qkv + H, 3 * H, q_so, hd, 0, w.S, Lp, s_so, s_si, L, L, hd, nh, B, s, mask_mode == 0)) return e;        // S = q k^T
  if (int e = tc_bgemm(w.dcb, H, c_so, hd, 0, w.qkv + 2 * H, 3 * H, q_so, hd, 0, w.dP, Lp, s_so, s_si, L, L, hd, nh, B, s, mask_mode == 0)) return e;       // dP = dctx v^T
  AttnRowArgs r;
  memset(&r, 0, sizeof(r));
  r.S = w.S; r.dP = w.dP; r.lse_in = lse; r.Pb = w.Pb; r.dSb = w.dSb; r.key_ids = key_ids; r.Z = B * nh; r.L = L; r.Lp = (int)Lp; r.nh = nh;
  r.mask_mode = mask_mode; r.bwd = 1; r.drop = mk_drop(d);
  { TIMED("attn_row_tc", s); attn_row_kernel<<<attn_rows_grid(B * nh * L), 256, 0, s>>>(r); }
  if (int e = tc_bgemm(w.dSb, Lp, s_so, s_si, 0, w.qkv + H, 3 * H, q_so, hd, 1, dq, H, c_so, hd, L, hd, L, nh, B, s)) return e;             // dq = dS k
  if (int e = tc_bgemm(w.dSb, Lp, s_so, s_si, 1, w.qkv, 3 * H, q_so, hd, 1, dk, H, c_so, hd, L, hd, L, nh, B, s)) return e;                 // dk = dS^T q
  if (int e = tc_bgemm(w.Pb, Lp, s_so, s_si, 1, w.dcb, H, c_so, hd, 1, dv, H, c_so, hd, L, hd, L, nh, B, s)) return e;                      // dv = (P m)^T dctx
  return check_launch("tcgen05 attention bwd");
}
// fused flash attention at any L (flash_tc.cu): the only path beyond 256 positions; `area` holds flash_scratch_bytes(B, max(L, 257), ...)
static int fl_attn_fwd(const float* q, const float* k, const float* v, float* ctx, float* lse, const int* key_ids, int B, int L, int H, int nh,
                       int mask_mode, const adt_dropout& d, int training, void* area, cudaStream_t s) {
  if (!area) return fail(ADT_E_SHAPE, "%s", "attention at L > 256: the fused flash kernels need their scratch area (attn_scratch / tc_scratch)");
  const int M = B * L;
  __nv_bfloat16* qkv = reinterpret_cast<__nv_bfloat16*>(align256(area));
  tc_pack(q, 1.f, nullptr, k, nullptr, v, nullptr, qkv, 3 * H, M, H, s);
  TIMED("attn_flash_fwd", s);
  if (int e = flash_attn_fwd(qkv, ctx, lse, key_ids, B, L, H, nh, mask_mode, mk_drop(row_drop(d, training)), s))
    return fail(e, "%s", "fused flash attention fwd (tensor map or launch)");
  return check_launch("fused flash attention fwd");
}
static int fl_attn_bwd(const float* q, const float* k, const float* v, const float* ctx, const float* dctx, const float* lse, const int* key_ids,
                       float* dq, float* dk, float* dv, int B, int L, int H, int nh, int mask_mode, const adt_dropout& d, void* area, cudaStream_t s) {
  if (!area) return fail(ADT_E_SHAPE, "%s", "attention at L > 256: the fused flash kernels need their scratch area (attn_scratch / tc_scratch)");
  if (!ctx) return fail(ADT_E_SHAPE, "%s", "attention backward at L > 256 reads the forward's output: ctx is NULL");
  const long long M = (long long)B * L;
  __nv_bfloat16* qkv = reinterpret_cast<__nv_bfloat16*>(align256(area));
  __nv_bfloat16* dcb = qkv + M * 3 * H;
  float* delta = reinterpret_cast<float*>(dcb + M * H);
  tc_pack(q, 1.f, nullptr, k, nullptr, v, nullptr, qkv, 3 * H, (int)M, H, s);
  tc_cast(dctx, dcb, M * H, s);
  TIMED("attn_flash_bwd", s);
  if (int e = flash_attn_bwd(qkv, dcb, ctx, dctx, delta, lse, key_ids, dq, dk, dv, B, L, H, nh, mask_mode, mk_drop(d), s))
    return fail(e, "%s", "fused flash attention bwd (tensor map or launch)");
  return check_launch("fused flash attention bwd");
}
// attention of every block path: beyond 256 positions the flash kernels (area `flash`); up to 256, long sequences through the batched
// GEMMs when `area` is given, short ones through the row-tile / small kernels
static int blk_attn_fwd(const float* q, const float* k, const float* v, float* ctx, float* lse, const int* ids, int B, int L, int H, int nh,
                        int mask_mode, const adt_dropout& d, int training, int precision, void* area, void* flash, cudaStream_t s) {
  if (L > ATTN_TILE_L) return fl_attn_fwd(q, k, v, ctx, lse, ids, B, L, H, nh, mask_mode, d, training, flash, s);
  if (area && use_attn_tc(B, L, H, nh)) return tc_attn_fwd(q, k, v, ctx, lse, ids, B, L, H, nh, mask_mode, d, training, area, s);
  return launch_attn_fwd(q, k, v, ctx, lse, ids, B, L, H, nh, mask_mode, d, training, precision, s);
}
static int blk_attn_bwd(const float* q, const float* k, const float* v, const float* ctx, const float* dctx, const float* lse, const int* ids,
                        float* dq, float* dk, float* dv, int B, int L, int H, int nh, int mask_mode, const adt_dropout& d, int precision, void* area,
                        void* flash, cudaStream_t s) {
  if (L > ATTN_TILE_L) return fl_attn_bwd(q, k, v, ctx, dctx, lse, ids, dq, dk, dv, B, L, H, nh, mask_mode, d, flash, s);
  if (area && use_attn_tc(B, L, H, nh)) return tc_attn_bwd(q, k, v, dctx, lse, ids, dq, dk, dv, B, L, H, nh, mask_mode, d, area, s);
  return launch_attn_bwd(q, k, v, dctx, lse, ids, dq, dk, dv, B, L, H, nh, mask_mode, d, precision, s);
}
// FFN adjoint shared by both blocks.  In: dO etc. through `pp`.  Out: slots 6-7 hold dz (enc) / dc (dec) = dO + dh1 C1.
static int tc_ffn_bwd(const TcBwdScratch& t, RowPostPrepArgs pp, const adt_ffn_w& ffn, const adt_ffn_g& gf, const __nv_bfloat16* C1b,
                      const __nv_bfloat16* C2b, const __nv_bfloat16* zb, int M, int H, cudaStream_t s) {
  pp.g = t.f32(6); pp.dh2b = t.op(0); pp.ab = t.op(1); pp.gc2 = gf.b2; pp.M = M; pp.H = H;
  { TIMED("row_tc", s); row_post_prep_kernel<<<rows_grid2(M), 256, 0, s>>>(pp); }
  if (int e = hoisted_wgrad(t.op(0), H, H, t.op(1), H, H, M, gf.w2, s)) return e;
  if (int e = tc_dgrad(t.op(0), H, H, C2b, H, t.f32(8), 0, M, s)) return e;                       // da = dh2 C2
  { TIMED("row_tc", s); row_dh1_kernel<<<rows_grid2(M), 256, 0, s>>>(t.f32(8), pp.h1, t.op(2), gf.b1, M, H, pp.drop1); }
  if (int e = hoisted_wgrad(t.op(2), H, H, zb, H, H, M, gf.w1, s)) return e;
  return tc_dgrad(t.op(2), H, H, C1b, H, t.f32(6), 1, M, s);                                      // dz / dc = dO + dh1 C1
}

static int tc_enc_bwd(const adt_enc_block_bwd_args* a, cudaStream_t s) {
  const int M = a->B * a->L, H = a->H;
  const TcBwdScratch t = mk_tcb(a->wgrad_scratch, M, H);
  const long long hh = (long long)H * H;
  const float qscale = 1.0f / sqrtf((float)(H / a->nh));
  const __nv_bfloat16* Winb = tc_weight(a->attn.in_w, 3 * hh, a->wm, t.wb, s);
  const __nv_bfloat16* Wob = tc_weight(a->attn.out_w, hh, a->wm, t.wb + 3 * hh, s);
  const __nv_bfloat16* C1b = tc_weight(a->ffn.w1, hh, a->wm, t.wb + 4 * hh, s);
  const __nv_bfloat16* C2b = tc_weight(a->ffn.w2, hh, a->wm, t.wb + 5 * hh, s);
  // z = LN2(y) as the wgrad operand of C1
  RowLnArgs r;
  memset(&r, 0, sizeof(r));
  r.x = a->y; r.g = a->ln2_w; r.b = a->ln2_b; r.yb = t.op(3); r.M = M; r.H = H;
  { TIMED("row_tc", s); row_ln_cast_kernel<<<row_grid(M), 256, 0, s>>>(r); }
  RowPostPrepArgs pp;
  memset(&pp, 0, sizeof(pp));
  pp.dout = a->dout; pp.ids = a->ids; pp.h1 = a->h1; pp.is_dec = 0;
  pp.drop1 = mk_drop(a->drop_ffn1); pp.drop2 = mk_drop(a->drop_ffn2);
  if (int e = tc_ffn_bwd(t, pp, a->ffn, a->g_ffn, C1b, C2b, t.op(3), M, H, s)) return e;
  // dy = LN2^T(dz) ; gbo += colsum(dy) ; gWo += dy^T ctx ; dctx = dy Wo (+ independence head)
  RowLnBwdArgs lb;
  memset(&lb, 0, sizeof(lb));
  lb.x = a->y; lb.g = t.f32(6); lb.ln_g = a->ln2_w; lb.dx = a->dy; lb.dxb = t.op(4); lb.gln_g = a->g_ln2_w; lb.gln_b = a->g_ln2_b;
  lb.gb = a->g_attn.out_b; lb.M = M; lb.H = H;
  { TIMED("row_tc", s); row_ln_bwd_kernel<<<rows_grid2(M), 256, 0, s>>>(lb); }
  tc_cast(a->ctx, t.op(5), (long long)M * H, s);
  if (int e = hoisted_wgrad(t.op(4), H, H, t.op(5), H, H, M, a->g_attn.out_w, s)) return e;
  if (int e = tc_dgrad(t.op(4), H, H, Wob, H, a->dctx, 0, M, s)) return e;
  if (a->nll_coef != 0.f || a->drec) {
    TIMED("row_tc", s);
    sparse_head_bwd_kernel<<<attn_rows_grid(M), 256, 0, s>>>(a->ctx, a->sparse_w, a->sparse_b, a->drec, a->nll_coef, a->dctx, a->g_sparse_w,
                                                        a->g_sparse_b, M, H, a->nh);
  }
  if (int e = check_launch("tcgen05 backward path (enc post)")) return e;
  if (int e = blk_attn_bwd(a->q, a->k, a->v, a->ctx, a->dctx, a->lse, a->ids, a->dq, a->dk, a->dv, a->B, a->L, H, a->nh, a->mask_mode,
                           a->drop_attn, a->precision, t.wb + 10 * hh, a->attn_scratch, s))
    return e;
  // in-projection: [dq*s | dk | dv] packed ; q rows read LN1(x), k / v rows read x
  tc_pack(a->dq, qscale, a->g_attn.in_b, a->dk, a->g_attn.in_b + H, a->dv, a->g_attn.in_b + 2 * H, t.op(0), 3 * H, M, H, s);
  memset(&r, 0, sizeof(r));
  r.x = a->x; r.g = a->ln1_w; r.b = a->ln1_b; r.yb = t.op(3); r.xb = t.op(4); r.M = M; r.H = H;
  { TIMED("row_tc", s); row_ln_cast_kernel<<<row_grid(M), 256, 0, s>>>(r); }
  if (int e = hoisted_wgrad(t.op(0), 3 * H, H, t.op(3), H, H, M, a->g_attn.in_w, s)) return e;
  if (int e = hoisted_wgrad(t.op(0) + H, 3 * H, 2 * H, t.op(4), H, H, M, a->g_attn.in_w + hh, s)) return e;
  if (int e = tc_dgrad(t.op(0), 3 * H, H, Winb, H, a->dy, 1, M, s)) return e;                    // dN = dy + dq*s Wq
  memset(&lb, 0, sizeof(lb));
  lb.x = a->x; lb.g = a->dy; lb.ln_g = a->ln1_w; lb.extra = a->dx_extra; lb.dx = a->dx; lb.gln_g = a->g_ln1_w; lb.gln_b = a->g_ln1_b;
  lb.M = M; lb.H = H;
  { TIMED("row_tc", s); row_ln_bwd_kernel<<<rows_grid2(M), 256, 0, s>>>(lb); }
  if (int e = tc_dgrad(t.op(0) + H, 3 * H, 2 * H, Winb + hh, H, a->dx, 1, M, s)) return e;       // dx += dk Wk + dv Wv
  return check_launch("tcgen05 backward path (enc pre)");
}

static int tc_dec_bwd(const adt_dec_block_bwd_args* a, cudaStream_t s) {
  const int M = a->B * a->L, H = a->H;
  const TcBwdScratch t = mk_tcb(a->wgrad_scratch, M, H);
  const long long hh = (long long)H * H;
  const float qscale = 1.0f / sqrtf((float)(H / a->nh));
  if (a->phase != 1) {
    const __nv_bfloat16* Wo1b = tc_weight(a->slf.out_w, hh, a->wm, t.wb + 3 * hh, s);
    const __nv_bfloat16* W2b = tc_weight(a->enc.in_w, 3 * hh, a->wm, t.wb + 4 * hh, s);
    const __nv_bfloat16* Wo2b = tc_weight(a->enc.out_w, hh, a->wm, t.wb + 7 * hh, s);
    const __nv_bfloat16* C1b = tc_weight(a->ffn.w1, hh, a->wm, t.wb + 8 * hh, s);
    const __nv_bfloat16* C2b = tc_weight(a->ffn.w2, hh, a->wm, t.wb + 9 * hh, s);
    tc_cast(a->c, t.op(3), (long long)M * H, s);
    RowPostPrepArgs pp;
    memset(&pp, 0, sizeof(pp));
    pp.dout = a->dout; pp.out = a->out; pp.enc_in = a->enc_in; pp.mse_coef = a->mse_coef; pp.denc = a->denc; pp.ids = a->ids; pp.h1 = a->h1;
    pp.g_copy = a->dd; pp.is_dec = 1;
    pp.drop1 = mk_drop(a->drop_ffn1); pp.drop2 = mk_drop(a->drop_ffn2);
    if (int e = tc_ffn_bwd(t, pp, a->ffn, a->g_ffn, C1b, C2b, t.op(3), M, H, s)) return e;
    // dc (slots 6-7): gbo2 += colsum ; gWo2 += dc^T ctx2 ; dctx2 = dc Wo2
    tc_pack(t.f32(6), 1.f, a->g_enc.out_b, nullptr, nullptr, nullptr, nullptr, t.op(4), H, M, H, s);
    tc_cast(a->ctx2, t.op(5), (long long)M * H, s);
    if (int e = hoisted_wgrad(t.op(4), H, H, t.op(5), H, H, M, a->g_enc.out_w, s)) return e;
    if (int e = tc_dgrad(t.op(4), H, H, Wo2b, H, a->dctx2, 0, M, s)) return e;
    if (int e = check_launch("tcgen05 backward path (dec post)")) return e;
    if (int e = blk_attn_bwd(a->q2, a->k2, a->v2, a->ctx2, a->dctx2, a->lse2, a->ids, a->dq2, a->dk2, a->dv2, a->B, a->L, H, a->nh, a->mask_mode,
                             a->drop_enc, a->precision, t.wb + 10 * hh, a->attn_scratch, s))
      return e;
    // cross-attention in-projection (q rows from a, k / v rows from the encoder features), then the self-attention out-projection
    tc_pack(a->dq2, qscale, a->g_enc.in_b, a->dk2, a->g_enc.in_b + H, a->dv2, a->g_enc.in_b + 2 * H, t.op(0), 3 * H, M, H, s);
    tc_cast(a->a, t.op(3), (long long)M * H, s);
    tc_cast(a->feats, t.op(4), (long long)M * H, s);
    if (int e = hoisted_wgrad(t.op(0), 3 * H, H, t.op(3), H, H, M, a->g_enc.in_w, s)) return e;
    if (int e = hoisted_wgrad(t.op(0) + H, 3 * H, 2 * H, t.op(4), H, H, M, a->g_enc.in_w + hh, s)) return e;
    if (int e = tc_dgrad(t.op(0), 3 * H, H, W2b, H, t.f32(8), 0, M, s)) return e;                  // da = dq2*s Wq2
    if (int e = tc_dgrad(t.op(0) + H, 3 * H, 2 * H, W2b + hh, H, a->dfeats, 1, M, s)) return e;    // dfeats += dk2 Wk2 + dv2 Wv2
    tc_pack(t.f32(8), 1.f, a->g_slf.out_b, nullptr, nullptr, nullptr, nullptr, t.op(5), H, M, H, s);
    tc_cast(a->ctx1, t.op(6), (long long)M * H, s);
    if (int e = hoisted_wgrad(t.op(5), H, H, t.op(6), H, H, M, a->g_slf.out_w, s)) return e;
    if (int e = tc_dgrad(t.op(5), H, H, Wo1b, H, a->dctx, 0, M, s)) return e;
    if (int e = check_launch("tcgen05 backward path (dec mid)")) return e;
    if (a->phase == 2) return ADT_OK;
  }
  const __nv_bfloat16* W1b = tc_weight(a->slf.in_w, 3 * hh, a->wm, t.wb, s);
  if (int e = blk_attn_bwd(a->q1, a->k1, a->v1, a->ctx1, a->dctx, a->lse1, a->ids, a->dq, a->dk, a->dv, a->B, a->L, H, a->nh, a->mask_mode,
                           a->drop_slf, a->precision, t.wb + 10 * hh, a->attn_scratch, s))
    return e;
  // q, k and v all read d = LN(x): one [3H x H] weight gradient, one K = 3H dgrad on top of dd
  tc_pack(a->dq, qscale, a->g_slf.in_b, a->dk, a->g_slf.in_b + H, a->dv, a->g_slf.in_b + 2 * H, t.op(0), 3 * H, M, H, s);
  tc_cast(a->d, t.op(3), (long long)M * H, s);
  if (int e = hoisted_wgrad(t.op(0), 3 * H, 3 * H, t.op(3), H, H, M, a->g_slf.in_w, s)) return e;
  if (int e = tc_dgrad(t.op(0), 3 * H, 3 * H, W1b, H, a->dd, 1, M, s)) return e;
  RowLnBwdArgs lb;
  memset(&lb, 0, sizeof(lb));
  lb.x = a->x; lb.g = a->dd; lb.ln_g = a->ln_w; lb.dx = a->dx; lb.gln_g = a->g_ln_w; lb.gln_b = a->g_ln_b; lb.M = M; lb.H = H;
  { TIMED("row_tc", s); row_ln_bwd_kernel<<<rows_grid2(M), 256, 0, s>>>(lb); }
  return check_launch("tcgen05 backward path (dec pre)");
}

// ---------------------------------------------------------------------------------------------------------
extern "C" int adt_enc_block_fwd(const adt_enc_block_fwd_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (int e = check_attn_dims(a->B, a->L, a->H, a->nh, a->precision)) return e;
  const int M = a->B * a->L, H = a->H;
  const int mma = a->precision ? 1 : 0, pad = mma ? 8 : 4;
  if (a->phase < 0 || a->phase > 2) return fail(ADT_E_SHAPE, "%s", "enc_block_fwd: phase must be 0, 1 or 2");
  if (a->phase == 0 && use_seq(a->L, H, a->nh, mma, a->training ? SEQ_ENC_FWD_TRAIN : SEQ_ENC_FWD)) return seq_enc_fwd(a, s);
  if (a->y && a->h1 && a->out && use_fwd_tc(a->tc_scratch, M, H, a->nh, mma)) return tc_enc_fwd(a, s);
  if (a->phase != 2) {
    if (int e = launch_pre_fwd(a->x, a->ln1_w, a->ln1_b, a->attn, a->q, a->k, a->v, nullptr, M, H, a->nh, 0, a->precision, s)) return e;
    if (int e = blk_attn_fwd(a->q, a->k, a->v, a->ctx, a->lse, a->ids, a->B, a->L, H, a->nh, a->mask_mode, a->drop_attn, a->training, a->precision,
                             nullptr, a->attn_scratch, s))
      return e;
    if (a->phase == 1) return ADT_OK;
  }
  PostFwdArgs p;
  memset(&p, 0, sizeof(p));
  p.ctx = a->ctx; p.resid = a->x; p.ids = a->ids; p.Wo = a->attn.out_w; p.bo = a->attn.out_b;
  p.ln1_g = a->ln1_w; p.ln1_b = a->ln1_b; p.ln2_g = a->ln2_w; p.ln2_b = a->ln2_b;
  p.C1 = a->ffn.w1; p.c1 = a->ffn.b1; p.C2 = a->ffn.w2; p.c2 = a->ffn.b2;
  p.Wsp = a->sparse_w; p.bsp = a->sparse_b;
  p.u_save = a->y; p.h1_save = a->h1; p.out = a->out; p.rec = a->rec; p.acc = a->nll_acc;
  p.M = M; p.H = H; p.nh = a->nh;
  p.drop1 = mk_drop(row_drop(a->drop_ffn1, a->training));
  p.drop2 = mk_drop(row_drop(a->drop_ffn2, a->training));
  size_t smem;
  const int tm = pick_tm(3 * (size_t)(H + pad), &smem);
  if (!tm) return fail(ADT_E_SHAPE, "%s", "post_fwd: tile does not fit shared memory");
  if (use_row_small(H, mma) && a->nh <= 8) {
    const size_t sm = PostFwdSmallSmem::TOTAL_BYTES;
    cudaFuncSetAttribute(post_fwd_small_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    TIMED("enc_post_fwd", s);
    post_fwd_small_kernel<false><<<(M + 63) / 64, AS_NT, sm, s>>>(p);
    return check_launch("enc post_fwd_small");
  }
  { TIMED("enc_post_fwd", s); LAUNCH_TM2(tm, mma, post_fwd_kernel, false, (M + tm - 1) / tm, smem, s, p); }
  return check_launch("enc post_fwd");
}

extern "C" int adt_enc_block_bwd(const adt_enc_block_bwd_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (int e = check_attn_dims(a->B, a->L, a->H, a->nh, a->precision)) return e;
  const int M = a->B * a->L, H = a->H;
  const int mma = a->precision ? 1 : 0, pad = mma ? 8 : 4;
  if (use_seq(a->L, H, a->nh, mma, SEQ_ENC_BWD)) return seq_enc_bwd(a, s);
  if (use_bwd_tc(a->wgrad_scratch, M, H, a->nh, mma)) return tc_enc_bwd(a, s);
  PostBwdArgs p;
  memset(&p, 0, sizeof(p));
  p.dout = a->dout; p.ids = a->ids; p.ctx = a->ctx; p.u = a->y; p.h1 = a->h1;
  p.Wo = a->attn.out_w; p.ln2_g = a->ln2_w; p.ln2_b = a->ln2_b; p.C1 = a->ffn.w1; p.C2 = a->ffn.w2;
  p.Wsp = a->sparse_w; p.bsp = a->sparse_b; p.nll_coef = a->nll_coef; p.drec = a->drec;
  p.dctx = a->dctx; p.dres = a->dy;
  p.gWo = a->g_attn.out_w; p.gbo = a->g_attn.out_b; p.gln2_g = a->g_ln2_w; p.gln2_b = a->g_ln2_b;
  p.gC1 = a->g_ffn.w1; p.gc1 = a->g_ffn.b1; p.gC2 = a->g_ffn.w2; p.gc2 = a->g_ffn.b2;
  p.gWsp = a->g_sparse_w; p.gbsp = a->g_sparse_b;
  p.M = M; p.H = H; p.nh = a->nh;
  p.drop1 = mk_drop(a->drop_ffn1); p.drop2 = mk_drop(a->drop_ffn2);
  __nv_bfloat16* hz = hoist_ptr(a->wgrad_scratch, H, mma);
  const long long hu = (long long)M * H;
  p.hoist = hz;
  size_t smem;
  int tm = pick_tm(4 * (size_t)(H + pad), &smem);
  if (!tm) return fail(ADT_E_SHAPE, "%s", "post_bwd: tile does not fit shared memory");
  if (use_row_small(H, mma) && a->nh <= 8) {
    const size_t sm = PostBwdSmallSmem::TOTAL_BYTES;
    cudaFuncSetAttribute(post_bwd_small_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    TIMED("enc_post_bwd", s);
    post_bwd_small_kernel<false><<<(M + 63) / 64, RS_BWD_NT, sm, s>>>(p);
  } else {
    TIMED("enc_post_bwd", s); LAUNCH_TM2(tm, mma, post_bwd_kernel, false, (M + tm - 1) / tm, smem, s, p);
  }
  if (int e = check_launch("enc post_bwd")) return e;
  if (hz) {
    if (int e = hoisted_wgrad(hz, H, H, hz + hu, H, H, M, a->g_ffn.w2, s)) return e;
    if (int e = hoisted_wgrad(hz + 2 * hu, H, H, hz + 3 * hu, H, H, M, a->g_ffn.w1, s)) return e;
    if (int e = hoisted_wgrad(hz + 4 * hu, H, H, hz + 5 * hu, H, H, M, a->g_attn.out_w, s)) return e;
  }
  if (int e = blk_attn_bwd(a->q, a->k, a->v, a->ctx, a->dctx, a->lse, a->ids, a->dq, a->dk, a->dv, a->B, a->L, H, a->nh, a->mask_mode,
                           a->drop_attn, a->precision, nullptr, a->attn_scratch, s))
    return e;
  PreBwdArgs r;
  memset(&r, 0, sizeof(r));
  r.dq = a->dq; r.dk = a->dk; r.dv = a->dv; r.x = a->x; r.dnorm_extra = a->dy; r.dx_extra = a->dx_extra;
  r.ln_g = a->ln1_w; r.ln_b = a->ln1_b; r.Win = a->attn.in_w; r.dx = a->dx;
  r.gWin = a->g_attn.in_w; r.gbin = a->g_attn.in_b; r.gln_g = a->g_ln1_w; r.gln_b = a->g_ln1_b;
  r.M = M; r.H = H; r.qscale = 1.0f / sqrtf((float)(H / a->nh)); r.kv_from_norm = 0;
  r.hoist = hz;
  if (int e = launch_pre_bwd(r, mma, s)) return e;
  if (hz) {   // Wq from LN(x), [Wk; Wv] from x
    if (int e = hoisted_wgrad(hz, 3 * H, H, hz + 3 * hu, H, H, M, a->g_attn.in_w, s)) return e;
    if (int e = hoisted_wgrad(hz + H, 3 * H, 2 * H, hz + 4 * hu, H, H, M, a->g_attn.in_w + (long long)H * H, s)) return e;
  }
  return ADT_OK;
}

// ---------------------------------------------------------------------------------------------------------
extern "C" int adt_dec_block_fwd(const adt_dec_block_fwd_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (int e = check_attn_dims(a->B, a->L, a->H, a->nh, a->precision)) return e;
  const int M = a->B * a->L, H = a->H;
  const int mma = a->precision ? 1 : 0, pad = mma ? 8 : 4;
  if (use_seq(a->L, H, a->nh, mma, SEQ_DEC_FWD)) return seq_dec_fwd(a, s);
  if (a->d && a->a && a->c && a->h1 && use_fwd_tc(a->tc_scratch, M, H, a->nh, mma)) return tc_dec_fwd(a, s);
  if (a->phase != 2) {
    if (int e = launch_pre_fwd(a->x, a->ln_w, a->ln_b, a->slf, a->q1, a->k1, a->v1, a->d, M, H, a->nh, 1, a->precision, s)) return e;
    if (int e = blk_attn_fwd(a->q1, a->k1, a->v1, a->ctx1, a->lse1, a->ids, a->B, a->L, H, a->nh, a->mask_mode, a->drop_slf, a->training, a->precision,
                             nullptr, a->attn_scratch, s))
      return e;
    if (a->phase == 1) return ADT_OK;
  }
  size_t smem;
  int tm = pick_tm(3 * (size_t)(H + pad), &smem);
  if (!tm) return fail(ADT_E_SHAPE, "%s", "mid_fwd: tile does not fit shared memory");
  const float qscale = 1.0f / sqrtf((float)(H / a->nh));
  if (use_row_small(H, mma)) {
    const size_t sm = MidFwdSmallSmem::TOTAL_BYTES;
    cudaFuncSetAttribute(mid_fwd_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    TIMED("mid_fwd", s);
    mid_fwd_small_kernel<<<(M + 63) / 64, AS_NT, sm, s>>>(a->ctx1, a->feats, a->slf.out_w, a->slf.out_b, a->enc.in_w, a->enc.in_b, a->a,
                                                        a->q2, a->k2, a->v2, M, qscale);
  } else {
    TIMED("mid_fwd", s);
    LAUNCH_TM(tm, mma, mid_fwd_kernel, (M + tm - 1) / tm, smem, s, a->ctx1, a->feats, a->slf.out_w, a->slf.out_b, a->enc.in_w, a->enc.in_b, a->a,
              a->q2, a->k2, a->v2, M, H, qscale);
  }
  if (int e = check_launch("mid_fwd")) return e;
  if (int e = blk_attn_fwd(a->q2, a->k2, a->v2, a->ctx2, a->lse2, a->ids, a->B, a->L, H, a->nh, a->mask_mode, a->drop_enc, a->training, a->precision,
                           nullptr, a->attn_scratch, s))
    return e;
  PostFwdArgs p;
  memset(&p, 0, sizeof(p));
  p.ctx = a->ctx2; p.resid = a->d; p.ids = a->ids; p.Wo = a->enc.out_w; p.bo = a->enc.out_b;
  p.C1 = a->ffn.w1; p.c1 = a->ffn.b1; p.C2 = a->ffn.w2; p.c2 = a->ffn.b2;
  p.enc_in = a->enc_in; p.u_save = a->c; p.h1_save = a->h1; p.out = a->out; p.acc = a->mse_acc;
  p.M = M; p.H = H; p.nh = a->nh;
  p.drop1 = mk_drop(row_drop(a->drop_ffn1, a->training));
  p.drop2 = mk_drop(row_drop(a->drop_ffn2, a->training));
  if (use_row_small(H, mma)) {
    const size_t sm = PostFwdSmallSmem::TOTAL_BYTES;
    cudaFuncSetAttribute(post_fwd_small_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    TIMED("dec_post_fwd", s);
    post_fwd_small_kernel<true><<<(M + 63) / 64, AS_NT, sm, s>>>(p);
    return check_launch("dec post_fwd_small");
  }
  { TIMED("dec_post_fwd", s); LAUNCH_TM2(tm, mma, post_fwd_kernel, true, (M + tm - 1) / tm, smem, s, p); }
  return check_launch("dec post_fwd");
}

extern "C" int adt_dec_block_bwd(const adt_dec_block_bwd_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (int e = check_attn_dims(a->B, a->L, a->H, a->nh, a->precision)) return e;
  const int M = a->B * a->L, H = a->H;
  const int mma = a->precision ? 1 : 0, pad = mma ? 8 : 4;
  const float qscale = 1.0f / sqrtf((float)(H / a->nh));
  if (use_seq(a->L, H, a->nh, mma, SEQ_DEC_BWD)) return seq_dec_bwd(a, s);
  if (use_bwd_tc(a->wgrad_scratch, M, H, a->nh, mma)) return tc_dec_bwd(a, s);
  __nv_bfloat16* hz = hoist_ptr(a->wgrad_scratch, H, mma);
  const long long hu = (long long)M * H;
  size_t smem;
  int tm = pick_tm(4 * (size_t)(H + pad), &smem);
  if (!tm) return fail(ADT_E_SHAPE, "%s", "post_bwd: tile does not fit shared memory");
  if (a->phase != 1) {
  PostBwdArgs p;
  memset(&p, 0, sizeof(p));
  p.dout = a->dout; p.out = a->out; p.enc_in = a->enc_in; p.mse_coef = a->mse_coef; p.denc = a->denc; p.ids = a->ids;
  p.ctx = a->ctx2; p.u = a->c; p.h1 = a->h1; p.Wo = a->enc.out_w; p.C1 = a->ffn.w1; p.C2 = a->ffn.w2;
  p.dctx = a->dctx2; p.dres = a->dd;
  p.gWo = a->g_enc.out_w; p.gbo = a->g_enc.out_b; p.gC1 = a->g_ffn.w1; p.gc1 = a->g_ffn.b1; p.gC2 = a->g_ffn.w2; p.gc2 = a->g_ffn.b2;
  p.M = M; p.H = H; p.nh = a->nh;
  p.drop1 = mk_drop(a->drop_ffn1); p.drop2 = mk_drop(a->drop_ffn2);
  p.hoist = hz;
  if (use_row_small(H, mma)) {
    const size_t sm = PostBwdSmallSmem::TOTAL_BYTES;
    cudaFuncSetAttribute(post_bwd_small_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    TIMED("dec_post_bwd", s);
    post_bwd_small_kernel<true><<<(M + 63) / 64, RS_BWD_NT, sm, s>>>(p);
  } else {
    TIMED("dec_post_bwd", s); LAUNCH_TM2(tm, mma, post_bwd_kernel, true, (M + tm - 1) / tm, smem, s, p);
  }
  if (int e = check_launch("dec post_bwd")) return e;
  if (hz) {
    if (int e = hoisted_wgrad(hz, H, H, hz + hu, H, H, M, a->g_ffn.w2, s)) return e;
    if (int e = hoisted_wgrad(hz + 2 * hu, H, H, hz + 3 * hu, H, H, M, a->g_ffn.w1, s)) return e;
    if (int e = hoisted_wgrad(hz + 4 * hu, H, H, hz + 5 * hu, H, H, M, a->g_enc.out_w, s)) return e;
  }
  // cross attention (keys/values from the encoder features)
  if (int e = blk_attn_bwd(a->q2, a->k2, a->v2, a->ctx2, a->dctx2, a->lse2, a->ids, a->dq2, a->dk2, a->dv2, a->B, a->L, H, a->nh, a->mask_mode,
                           a->drop_enc, a->precision, nullptr, a->attn_scratch, s))
    return e;
  MidBwdArgs m;
  memset(&m, 0, sizeof(m));
  m.dq2 = a->dq2; m.dk2 = a->dk2; m.dv2 = a->dv2; m.a = a->a; m.feats = a->feats; m.ctx1 = a->ctx1;
  m.Wo1 = a->slf.out_w; m.Win2 = a->enc.in_w; m.dfeats = a->dfeats; m.dctx1 = a->dctx;
  m.gWo1 = a->g_slf.out_w; m.gbo1 = a->g_slf.out_b; m.gWin2 = a->g_enc.in_w; m.gbin2 = a->g_enc.in_b;
  m.M = M; m.H = H; m.qscale = qscale;
  m.hoist = hz;
  if (use_row_small(H, mma)) {
    const size_t sm = MidBwdSmallSmem::TOTAL_BYTES;
    cudaFuncSetAttribute(mid_bwd_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    TIMED("mid_bwd", s);
    mid_bwd_small_kernel<<<(M + 63) / 64, RS_BWD_NT, sm, s>>>(m);
  } else {
  tm = pick_tm(3 * (size_t)(H + pad) + (size_t)(2 * H + pad), &smem, 128, M >= 148 * 64 ? 128 : 64);
  if (!tm) return fail(ADT_E_SHAPE, "%s", "mid_bwd: tile does not fit shared memory");
  { TIMED("mid_bwd", s); LAUNCH_TM(tm, mma, mid_bwd_kernel, (M + tm - 1) / tm, smem, s, m); }
  }
  if (int e = check_launch("mid_bwd")) return e;
  if (hz) {   // cross-attention in-projection (q rows from a, [k; v] rows from the encoder features) and the self-attention out-projection
    if (int e = hoisted_wgrad(hz, H, H, hz + hu, H, H, M, a->g_enc.in_w, s)) return e;
    if (int e = hoisted_wgrad(hz + 2 * hu, 2 * H, 2 * H, hz + 4 * hu, H, H, M, a->g_enc.in_w + (long long)H * H, s)) return e;
    if (int e = hoisted_wgrad(hz + 5 * hu, H, H, hz + 6 * hu, H, H, M, a->g_slf.out_w, s)) return e;
  }
  if (a->phase == 2) return ADT_OK;
  }
  if (int e = blk_attn_bwd(a->q1, a->k1, a->v1, a->ctx1, a->dctx, a->lse1, a->ids, a->dq, a->dk, a->dv, a->B, a->L, H, a->nh, a->mask_mode,
                           a->drop_slf, a->precision, nullptr, a->attn_scratch, s))
    return e;
  PreBwdArgs r;
  memset(&r, 0, sizeof(r));
  r.dq = a->dq; r.dk = a->dk; r.dv = a->dv; r.x = a->x; r.dnorm_extra = a->dd; r.dx_extra = nullptr;
  r.ln_g = a->ln_w; r.ln_b = a->ln_b; r.Win = a->slf.in_w; r.dx = a->dx;
  r.gWin = a->g_slf.in_w; r.gbin = a->g_slf.in_b; r.gln_g = a->g_ln_w; r.gln_b = a->g_ln_b;
  r.M = M; r.H = H; r.qscale = qscale; r.kv_from_norm = 1;
  r.hoist = hz;
  if (int e = launch_pre_bwd(r, mma, s)) return e;
  if (hz) {   // q, k and v all read d = LN(x): one [3H x H] product
    if (int e = hoisted_wgrad(hz, 3 * H, 3 * H, hz + 3 * hu, H, H, M, a->g_slf.in_w, s)) return e;
  }
  return ADT_OK;
}

// ---------------------------------------------------------------------------------------------------------
extern "C" int adt_final_logits_loss_fwd(const adt_final_fwd_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (a->H > 256 || (a->H & 3)) return fail(ADT_E_SHAPE, "%s", "final_fwd: H");
  const int grid = min((a->M + 7) / 8, 148 * 8);
  TIMED("final_fwd", s);
  final_fwd_kernel<<<grid, NT, 0, s>>>(a->x, a->ln_w, a->ln_b, a->item_emb, a->pos, a->neg, a->feats, a->pos_logits, a->neg_logits, a->acc,
                                       a->M, a->H);
  return check_launch("final_fwd");
}

extern "C" int adt_final_logits_loss_bwd(const adt_final_bwd_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (a->H > 256 || (a->H & 3)) return fail(ADT_E_SHAPE, "%s", "final_bwd: H");
  FinalBwdArgs p;
  p.x = a->x; p.ln_g = a->ln_w; p.E = a->item_emb; p.pos = a->pos; p.neg = a->neg;
  p.pos_logits = a->pos_logits; p.neg_logits = a->neg_logits; p.dfeats_in = a->dfeats_in; p.n_valid = a->n_valid;
  p.bce_weight = a->bce_weight; p.dpl_ext = a->dpl_ext; p.dnl_ext = a->dnl_ext;
  p.dx = a->dx; p.cpos = a->cpos; p.cneg = a->cneg; p.gln_g = a->g_ln_w; p.gln_b = a->g_ln_b; p.M = a->M; p.H = a->H;
  const int grid = min((a->M + 7) / 8, 148 * 4);
  TIMED("final_bwd", s);
  final_bwd_kernel<<<grid, NT, 0, s>>>(p);
  return check_launch("final_bwd");
}

// ---------------------------------------------------------------------------------------------------------
extern "C" int adt_embed_sort(const adt_embed_sort_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  const int N = 4 * a->M;
  const int nW = (N + SORT_WCH - 1) / SORT_WCH;
  int bits = 1;
  while ((1ll << bits) <= (long long)a->max_id) ++bits;
  const int passes = (bits + 7) / 8;
  SortSrc src;
  src.ids[0] = a->seq; src.ids[1] = a->dec; src.ids[2] = a->pos; src.ids[3] = a->neg; src.M = a->M;
  const int grid = (nW + 7) / 8;
  // ping-pong so that the last pass lands in (keys, vals)
  int* kbuf[2] = {a->keys, a->keys_tmp};
  int* vbuf[2] = {a->vals, a->vals_tmp};
  int cur = (passes & 1) ? 0 : 1;   // buffer written by pass 0
  const int* kin = nullptr;
  const int* vin = nullptr;
  TIMED("embed_sort", s);
  // offsets: exclusive scan of the 256*nW digit counters.  Small inputs: one CTA.  Large inputs: per-tile scans + a scan of
  // the tile totals kept in the unused upper part of `hist` (its size is 256*ceil(N/256) >= 256*nW + tiles there).
  const int nh = 256 * nW, tiles = (nh + 4095) / 4096;
  const long long room = 256ll * ((N + 255) / 256) - nh;
  const bool tiled = tiles > 2 && room >= tiles;
  int* tsum = tiled ? a->hist + nh : nullptr;
  for (int p = 0; p < passes; ++p) {
    const int shift = 8 * p;
    if (p == 0) radix_hist_kernel<true><<<grid, 256, 0, s>>>(src, nullptr, N, shift, a->hist, nW);
    else radix_hist_kernel<false><<<grid, 256, 0, s>>>(src, kin, N, shift, a->hist, nW);
    if (tiled) {
      scan_tiles_kernel<<<tiles, 1024, 0, s>>>(a->hist, nh, tsum);
      exclusive_scan_kernel<<<1, 1024, 0, s>>>(tsum, tiles);
    } else {
      exclusive_scan_kernel<<<1, 1024, 0, s>>>(a->hist, nh);
    }
    if (p == 0) radix_scatter_kernel<true><<<grid, 256, 0, s>>>(src, nullptr, nullptr, N, shift, a->hist, nW, kbuf[cur], vbuf[cur], tsum);
    else radix_scatter_kernel<false><<<grid, 256, 0, s>>>(src, kin, vin, N, shift, a->hist, nW, kbuf[cur], vbuf[cur], tsum);
    kin = kbuf[cur];
    vin = vbuf[cur];
    cur ^= 1;
  }
  return check_launch("adt_embed_sort");
}

extern "C" int adt_embed_bwd(const adt_embed_bwd_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (int e = check_dims(a->B, a->L, a->H, 1)) return e;
  const int M = a->B * a->L;
  if (NT / (a->H / 4) < 1) return fail(ADT_E_SHAPE, "%s", "embed_bwd: H");
  TIMED("embed_bwd", s);
  if (a->d_pos_emb) {
    const int BS = (a->B + 148 * 4 - 1) / (148 * 4), pg = (a->B + BS - 1) / BS;   // sequences per CTA / CTAs
    if (a->dx_enc || a->dx_dec)
      posgrad_kernel<<<dim3(pg, 2), NT, 0, s>>>(a->dx_enc, a->seq, mk_drop(a->drop_enc), a->dx_dec, a->dec, mk_drop(a->drop_dec), a->d_pos_emb,
                                                a->B, a->L, a->H, BS);
  }
  ScatterArgs sa;
  memset(&sa, 0, sizeof(sa));
  sa.keys = a->keys; sa.vals = a->vals; sa.N = 4 * M; sa.M = M; sa.H = a->H;
  sa.dx_enc = a->dx_enc; sa.dx_dec = a->dx_dec; sa.feats = a->feats; sa.cpos = a->cpos; sa.cneg = a->cneg;
  sa.scale = a->emb_scale != 0.f ? a->emb_scale : (float)sqrt((double)a->H);
  sa.drop_enc = mk_drop(a->drop_enc); sa.drop_dec = mk_drop(a->drop_dec);
  sa.dE = a->d_item_emb; sa.head = a->head; sa.tail = a->tail; sa.has_tail = a->has_tail;
  const int nb = (sa.N + 31) / 32;
  if (a->H <= 128) scatter_phase1_kernel<1><<<(nb + 7) / 8, 256, 0, s>>>(sa);
  else scatter_phase1_kernel<2><<<(nb + 7) / 8, 256, 0, s>>>(sa);
  scatter_phase2_kernel<<<(nb + 7) / 8, 256, 0, s>>>(sa);
  return check_launch("adt_embed_bwd");
}

// ---------------------------------------------------------------------------------------------------------
extern "C" int adt_sumsq(const float* x, int64_t n, double* out, adt_stream_t s_) {
  const int grid = (int)((n / 4 + 255) / 256 < 148 * 8 ? ((n / 4 + 255) / 256 > 0 ? (n / 4 + 255) / 256 : 1) : 148 * 8);
  TIMED("sumsq", (cudaStream_t)s_);
  sumsq_kernel<<<grid, 256, 0, (cudaStream_t)s_>>>(x, (long long)n, out);
  return check_launch("adt_sumsq");
}

extern "C" int adt_sumsq_decay(float* g, const float* w, int64_t n, int64_t decay_off, float wd, const double* normsq, double* out,
                               adt_stream_t s_) {
  if (decay_off & 3) return fail(ADT_E_ALIGN, "%s", "sumsq_decay: decay_off must be a multiple of 4");
  const int grid = (int)((n / 4 + 255) / 256 < 148 * 8 ? ((n / 4 + 255) / 256 > 0 ? (n / 4 + 255) / 256 : 1) : 148 * 8);
  TIMED("sumsq", (cudaStream_t)s_);
  sumsq_decay_kernel<<<grid, 256, 0, (cudaStream_t)s_>>>(g, w, (long long)n, (long long)decay_off, wd, normsq, out);
  return check_launch("adt_sumsq_decay");
}

extern "C" int adt_norm_decay_grad(float* g, const float* w, int64_t n, float wd, const double* normsq, adt_stream_t s_) {
  const long long blocks = (n + 255) / 256;
  norm_decay_grad_kernel<<<(int)(blocks < 148 * 8 ? blocks : 148 * 8), 256, 0, (cudaStream_t)s_>>>(g, w, (long long)n, wd, normsq);
  return check_launch("adt_norm_decay_grad");
}

extern "C" int adt_adam(const adt_adam_args* a, adt_stream_t s_) {
  AdamArgs k;
  k.p = a->p; k.g = a->g; k.m = a->m; k.v = a->v; k.n = a->n;
  k.lr = a->lr; k.beta1 = a->beta1; k.beta2 = a->beta2; k.eps = a->eps; k.weight_decay = a->weight_decay;
  k.bc1 = (float)(1.0 - pow((double)a->beta1, (double)a->step));
  k.bc2 = (float)(1.0 - pow((double)a->beta2, (double)a->step));
  k.max_norm = a->max_norm; k.gnormsq = a->gnormsq; k.step_dev = a->step_dev;
  k.mirror = reinterpret_cast<__nv_bfloat16*>(a->mirror); k.mirror_n = a->mirror ? (a->mirror_n & ~3ll) : 0;
  if ((((uintptr_t)a->p | (uintptr_t)a->g | (uintptr_t)a->m | (uintptr_t)a->v) & 15) != 0)
    return fail(ADT_E_ALIGN, "%s", "adam: buffers must be 16-byte aligned");
  const long long blocks = (a->n / 4 + 255) / 256 + 1;
  TIMED("adam", (cudaStream_t)s_);
  adam_kernel<<<(int)(blocks < 148 * 8 ? blocks : 148 * 8), 256, 0, (cudaStream_t)s_>>>(k);
  return check_launch("adt_adam");
}

extern "C" int adt_adam_segmented(const adt_adam_args* a, const adt_adam_segments* g, adt_stream_t s_) {
  if (g->n_chunks <= 0) return ADT_OK;
  AdamSegArgs k;
  k.a.p = a->p; k.a.g = a->g; k.a.m = a->m; k.a.v = a->v; k.a.n = a->n;
  k.a.lr = a->lr; k.a.beta1 = a->beta1; k.a.beta2 = a->beta2; k.a.eps = a->eps; k.a.weight_decay = a->weight_decay;
  k.a.bc1 = k.a.bc2 = 1.f; k.a.max_norm = a->max_norm; k.a.gnormsq = a->gnormsq; k.a.step_dev = nullptr;
  k.a.mirror = nullptr; k.a.mirror_n = 0;
  k.chunk_start = (const long long*)g->chunk_start; k.chunk_len = g->chunk_len; k.chunk_seg = g->chunk_seg; k.n_chunks = g->n_chunks;
  k.seg_step = g->seg_step; k.active_seg = g->active_seg; k.n_active = g->n_active;
  TIMED("adam", (cudaStream_t)s_);
  if (g->n_active > 0) adam_seg_step_kernel<<<(g->n_active + 255) / 256, 256, 0, (cudaStream_t)s_>>>(k);
  adam_seg_kernel<<<g->n_chunks < 148 * 8 ? g->n_chunks : 148 * 8, 256, 0, (cudaStream_t)s_>>>(k);
  return check_launch("adt_adam_segmented");
}

extern "C" int adt_count_nonzero(const int32_t* ids, int32_t n, double* out, adt_stream_t s_) {
  cudaMemsetAsync(out, 0, sizeof(double), (cudaStream_t)s_);
  count_nonzero_kernel<<<min((n + 255) / 256, 148), 256, 0, (cudaStream_t)s_>>>(ids, n, out);
  return check_launch("adt_count_nonzero");
}

extern "C" int adt_philox_mask(float* out, int64_t n, const adt_dropout* d, adt_stream_t s_) {
  const long long blocks = (n + 255) / 256;
  philox_mask_kernel<<<(int)(blocks < 148 * 8 ? blocks : 148 * 8), 256, 0, (cudaStream_t)s_>>>(out, (long long)n, mk_drop(*d));
  return check_launch("adt_philox_mask");
}

// ---------------------------------------------------------------------------------------------------------
// generic ops
extern "C" int adt_linear_fwd(const adt_linear_fwd_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (a->M <= 0 || (a->K & 3) || a->N <= 0 || a->K > 2048) return fail(ADT_E_SHAPE, "%s", "linear_fwd: K must be a multiple of 4, K <= 2048");
  const int mma = a->precision ? 1 : 0, pad = mma ? 8 : 4;
  size_t smem;
  const int tm = pick_tm((size_t)(a->K + pad), &smem);
  if (!tm) return fail(ADT_E_SHAPE, "%s", "linear_fwd: tile does not fit shared memory");
  LinearFwdArgs p;
  p.x = a->x; p.W = a->w; p.b = a->b; p.y = a->y; p.pre = a->pre; p.M = a->M; p.K = a->K; p.N = a->N; p.act = a->act;
  p.scale = a->scale == 0.f ? 1.f : a->scale;
  p.ldy = a->ldy ? a->ldy : a->N;
  TIMED("linear_fwd", s);
  LAUNCH_TM(tm, mma, linear_fwd_kernel, (a->M + tm - 1) / tm, smem, s, p);
  return check_launch("linear_fwd");
}

extern "C" int adt_linear_bwd(const adt_linear_bwd_args* a, adt_stream_t s_) {
  cudaStream_t s = (cudaStream_t)s_;
  if (a->M <= 0 || (a->K & 3) || a->N <= 0) return fail(ADT_E_SHAPE, "%s", "linear_bwd: K must be a multiple of 4");
  const int mma = a->precision ? 1 : 0, pad = mma ? 8 : 4;
  size_t smem;
  const int tm = pick_tm((size_t)(a->K + pad) + (size_t)(((a->N + 3) & ~3) + pad), &smem);
  if (!tm) return fail(ADT_E_SHAPE, "%s", "linear_bwd: tile does not fit shared memory");
  LinearBwdArgs p;
  p.x = a->x; p.W = a->w; p.dy = a->dy; p.dx = a->dx; p.gW = a->g_w; p.gb = a->g_b; p.M = a->M; p.K = a->K; p.N = a->N;
  p.accumulate_dx = a->accumulate_dx; p.scale = a->scale == 0.f ? 1.f : a->scale;
  p.lddy = a->lddy ? a->lddy : a->N;
  TIMED("linear_bwd", s);
  LAUNCH_TM(tm, mma, linear_bwd_kernel, (a->M + tm - 1) / tm, smem, s, p);
  return check_launch("linear_bwd");
}

extern "C" int adt_act_bwd(const float* dy, const float* pre, float* dpre, int64_t n, int32_t act, adt_stream_t s_) {
  if (n & 3) return fail(ADT_E_SHAPE, "%s", "act_bwd: n must be a multiple of 4");
  const long long n4 = n / 4, blocks = (n4 + 255) / 256;
  act_bwd_kernel<<<(int)(blocks < 148 * 16 ? (blocks > 0 ? blocks : 1) : 148 * 16), 256, 0, (cudaStream_t)s_>>>(dy, pre, dpre, n4, act);
  return check_launch("act_bwd");
}

static DrlArgs mk_drl(const adt_drl_args* a) {
  DrlArgs p;
  p.a = a->a; p.r = a->r; p.gamma = a->gamma; p.beta = a->beta; p.y = a->y; p.dy = a->dy; p.da = a->da; p.dr = a->dr;
  p.ggamma = a->g_gamma; p.gbeta = a->g_beta; p.M = a->M; p.H = a->H; p.mode = a->mode; p.eps = a->eps; p.drop = mk_drop(a->drop);
  return p;
}
extern "C" int adt_drop_res_ln_fwd(const adt_drl_args* a, adt_stream_t s_) {
  if (a->H > 256 || a->H <= 0) return fail(ADT_E_SHAPE, "%s", "drop_res_ln: H <= 256");
  const int grid = min((a->M + 7) / 8, 148 * 8);
  drl_fwd_kernel<<<grid, NT, 0, (cudaStream_t)s_>>>(mk_drl(a));
  return check_launch("drop_res_ln_fwd");
}
extern "C" int adt_drop_res_ln_bwd(const adt_drl_args* a, adt_stream_t s_) {
  if (a->H > 256 || a->H <= 0) return fail(ADT_E_SHAPE, "%s", "drop_res_ln: H <= 256");
  const int grid = min((a->M + 7) / 8, 148 * 4);
  drl_bwd_kernel<<<grid, NT, 0, (cudaStream_t)s_>>>(mk_drl(a));
  return check_launch("drop_res_ln_bwd");
}

extern "C" int adt_gather3(const int32_t* ia, const float* A, const int32_t* ib, const float* B, const int32_t* ic, const float* C, float* sdst,
                           int32_t M, int32_t H, adt_stream_t s_) {
  if (H & 3) return fail(ADT_E_SHAPE, "%s", "gather3: H % 4");
  const long long n = (long long)M * (H / 4), blocks = (n + 255) / 256;
  gather3_kernel<<<(int)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, (cudaStream_t)s_>>>(ia, A, ib, B, ic, C, sdst, M, H);
  return check_launch("gather3");
}
extern "C" int adt_small_table_grad(const int32_t* ids, const float* dx, float* g, int32_t M, int32_t H, int32_t padding_idx,
                                    adt_stream_t s_) {
  if (H & 3) return fail(ADT_E_SHAPE, "%s", "small_table_grad: H % 4");
  const long long n = (long long)M * (H / 4), blocks = (n + 255) / 256;
  small_table_grad_kernel<<<(int)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, (cudaStream_t)s_>>>(ids, dx, g, M, H, padding_idx);
  return check_launch("small_table_grad");
}

extern "C" int64_t adt_attention_scratch_bytes(int32_t B, int32_t L, int32_t H, int32_t nh, int32_t backward) {
  if (B <= 0 || L <= 0 || H <= 0 || nh <= 0) return 0;
  if (L > ATTN_TILE_L) return flash_scratch_bytes(B, L, H, nh, backward != 0);
  if (!use_attn_tc(B, L, H, nh)) return 0;
  const long long M = (long long)B * L, Lp = (L + 7) / 8 * 8, zll = M * nh * Lp;
  return 1024 + (backward ? 4 : 3) * M * H * 2 + zll * (backward ? 12 : 6);
}
extern "C" int adt_attention_fwd(const adt_attention_args* a, adt_stream_t s_) {
  if (int e = check_attn_dims(a->B, a->L, a->H, a->nh, a->precision)) return e;
  return blk_attn_fwd(a->q, a->k, a->v, a->ctx, a->lse, a->key_ids, a->B, a->L, a->H, a->nh, a->mask_mode, a->drop, a->training,
                      a->precision ? 1 : 0, a->precision ? a->tc_scratch : nullptr, a->tc_scratch, (cudaStream_t)s_);
}
extern "C" int adt_attention_bwd(const adt_attention_args* a, adt_stream_t s_) {
  if (int e = check_attn_dims(a->B, a->L, a->H, a->nh, a->precision)) return e;
  return blk_attn_bwd(a->q, a->k, a->v, a->ctx, a->dctx, a->lse, a->key_ids, a->dq, a->dk, a->dv, a->B, a->L, a->H, a->nh, a->mask_mode, a->drop,
                      a->precision ? 1 : 0, a->precision ? a->tc_scratch : nullptr, a->tc_scratch, (cudaStream_t)s_);
}
// the flash kernels at any L <= 2048 (for L <= 256 a test / comparison entry: the dispatch above never takes them there)
static int check_flash(const adt_attention_args* a) {
  if (int e = check_attn_dims(a->B, a->L > ATTN_TILE_L ? a->L : ATTN_TILE_L + 1, a->H, a->nh, a->precision)) return e;
  return check_dims(a->B, a->L, a->H, a->nh);
}
extern "C" int adt_attention_flash_fwd(const adt_attention_args* a, adt_stream_t s_) {
  if (int e = check_flash(a)) return e;
  return fl_attn_fwd(a->q, a->k, a->v, a->ctx, a->lse, a->key_ids, a->B, a->L, a->H, a->nh, a->mask_mode, a->drop, a->training, a->tc_scratch,
                     (cudaStream_t)s_);
}
extern "C" int adt_attention_flash_bwd(const adt_attention_args* a, adt_stream_t s_) {
  if (int e = check_flash(a)) return e;
  return fl_attn_bwd(a->q, a->k, a->v, a->ctx, a->dctx, a->lse, a->key_ids, a->dq, a->dk, a->dv, a->B, a->L, a->H, a->nh, a->mask_mode, a->drop,
                     a->tc_scratch, (cudaStream_t)s_);
}

extern "C" int adt_softmax_ce_fwd(const float* logits, const int32_t* labels, float* lse, double* loss_acc, int32_t R, int32_t V,
                                  adt_stream_t s_) {
  softmax_ce_kernel<<<min(R, 148 * 8), NT, 0, (cudaStream_t)s_>>>(const_cast<float*>(logits), labels, lse, loss_acc, R, V, 0, 0.f);
  return check_launch("softmax_ce_fwd");
}
extern "C" int adt_softmax_ce_bwd(float* logits, const int32_t* labels, const float* lse, float coef, int32_t R, int32_t V, adt_stream_t s_) {
  softmax_ce_kernel<<<min(R, 148 * 8), NT, 0, (cudaStream_t)s_>>>(logits, labels, const_cast<float*>(lse), nullptr, R, V, 1, coef);
  return check_launch("softmax_ce_bwd");
}

// ---- STOSA-ADT -------------------------------------------------------------------------------------------------
extern "C" int adt_act_fwd(const float* x, float* y, int64_t n, int32_t act, adt_stream_t s_) {
  if (n & 3) return fail(ADT_E_SHAPE, "%s", "act_fwd: n must be a multiple of 4");
  const long long n4 = n / 4, blocks = (n4 + 255) / 256;
  act_fwd_kernel<<<(int)(blocks < 148 * 16 ? (blocks > 0 ? blocks : 1) : 148 * 16), 256, 0, (cudaStream_t)s_>>>(x, y, n4, act);
  return check_launch("act_fwd");
}
static int launch_wattn(const adt_wattention_args* a, bool bwd, cudaStream_t s) {
  if (a->B <= 0 || a->L <= 0 || a->nh <= 0 || a->H % a->nh || ((a->H / a->nh) & 3)) return fail(ADT_E_SHAPE, "%s", "wattention: dims");
  const int hd = a->H / a->nh;
  const size_t smem = wattn_smem_floats(a->L, hd, bwd) * sizeof(float);
  if (smem > 220 * 1024) return fail(ADT_E_SHAPE, "%s", "wattention: (L, H/nh) tile does not fit shared memory");
  WAttnArgs p;
  p.mq = a->mq; p.cq = a->cq; p.mk = a->mk; p.ck = a->ck; p.mv = a->mv; p.cv = a->cv; p.mctx = a->mctx; p.cctx = a->cctx; p.lse = a->lse;
  p.key_ids = a->key_ids; p.dmctx = a->dmctx; p.dcctx = a->dcctx; p.dmq = a->dmq; p.dcq = a->dcq; p.dmk = a->dmk; p.dck = a->dck;
  p.dmv = a->dmv; p.dcv = a->dcv; p.B = a->B; p.L = a->L; p.H = a->H; p.nh = a->nh; p.inv_sqrt_hd = 1.0f / sqrtf((float)hd);
  p.drop = mk_drop(a->drop);
  const int grid = min(a->B * a->nh, 148 * 8);
  if (bwd) {
    cudaFuncSetAttribute(wattn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    wattn_bwd_kernel<<<grid, NT, smem, s>>>(p);
  } else {
    cudaFuncSetAttribute(wattn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    wattn_fwd_kernel<<<grid, NT, smem, s>>>(p);
  }
  return check_launch(bwd ? "wattention_bwd" : "wattention_fwd");
}
extern "C" int adt_wattention_fwd(const adt_wattention_args* a, adt_stream_t s_) { return launch_wattn(a, false, (cudaStream_t)s_); }
extern "C" int adt_wattention_bwd(const adt_wattention_args* a, adt_stream_t s_) { return launch_wattn(a, true, (cudaStream_t)s_); }

static WBprArgs mk_wbpr(const adt_wbpr_args* a) {
  WBprArgs p;
  p.sm = a->seq_mean; p.sc = a->seq_cov; p.Em = a->item_mean; p.Ec = a->item_cov; p.pos = a->pos; p.neg = a->neg; p.acc = a->acc;
  p.gcoef = a->gcoef; p.dsm = a->d_seq_mean; p.dsc = a->d_seq_cov; p.gpm = a->g_pos_mean; p.gpc = a->g_pos_cov; p.gnm = a->g_neg_mean;
  p.gnc = a->g_neg_cov; p.M = a->M; p.H = a->H;
  return p;
}
extern "C" int adt_wbpr_fwd(const adt_wbpr_args* a, adt_stream_t s_) {
  if (a->M <= 0 || a->H <= 0) return fail(ADT_E_SHAPE, "%s", "wbpr: dims");
  wbpr_fwd_kernel<<<min((a->M + 7) / 8, 148 * 8), NT, 0, (cudaStream_t)s_>>>(mk_wbpr(a));
  return check_launch("wbpr_fwd");
}
extern "C" int adt_wbpr_bwd(const adt_wbpr_args* a, adt_stream_t s_) {
  if (a->M <= 0 || a->H <= 0) return fail(ADT_E_SHAPE, "%s", "wbpr: dims");
  wbpr_bwd_kernel<<<min((a->M + 7) / 8, 148 * 8), NT, 0, (cudaStream_t)s_>>>(mk_wbpr(a));
  return check_launch("wbpr_bwd");
}
extern "C" int adt_sqdiff_fwd(const float* a, const float* b, int64_t n, double* acc, adt_stream_t s_) {
  if (n & 3) return fail(ADT_E_SHAPE, "%s", "sqdiff: n must be a multiple of 4");
  const long long n4 = n / 4, blocks = (n4 + 255) / 256;
  sqdiff_fwd_kernel<<<(int)(blocks < 148 * 8 ? (blocks > 0 ? blocks : 1) : 148 * 8), 256, 0, (cudaStream_t)s_>>>(a, b, n4, acc);
  return check_launch("sqdiff_fwd");
}
extern "C" int adt_sqdiff_bwd(const float* a, const float* b, const float* g, float scale, float* da, float* db, int64_t n, adt_stream_t s_) {
  if (n & 3) return fail(ADT_E_SHAPE, "%s", "sqdiff: n must be a multiple of 4");
  const long long n4 = n / 4, blocks = (n4 + 255) / 256;
  sqdiff_bwd_kernel<<<(int)(blocks < 148 * 8 ? (blocks > 0 ? blocks : 1) : 148 * 8), 256, 0, (cudaStream_t)s_>>>(a, b, g, scale, da, db, n4);
  return check_launch("sqdiff_bwd");
}
extern "C" int adt_wcatalog_rows(const float* mean, const float* cov, float* out, int32_t n, int32_t H, int32_t is_user, adt_stream_t s_) {
  if (n <= 0 || H <= 0) return fail(ADT_E_SHAPE, "%s", "wcatalog_rows: dims");
  wcatalog_kernel<<<min((n + 7) / 8, 148 * 8), NT, 0, (cudaStream_t)s_>>>(mean, cov, out, n, H, is_user);
  return check_launch("wcatalog_rows");
}
extern "C" int adt_wcatalog_work_bytes(int32_t H, int64_t* bytes) {
  if (H <= 0 || 2 * H > NT) return fail(ADT_E_SHAPE, "%s", "wcatalog_work_bytes: H must be 1..128");
  *bytes = (int64_t)WCAT_PARTS * 2 * H * (int64_t)sizeof(double) + 16;
  return ADT_OK;
}
extern "C" int adt_wcatalog_build(const float* mean, const float* cov, int32_t n, int32_t H, float* mu, float* rows, float* bias, void* work,
                                  adt_stream_t s_) {
  if (n <= 0 || H <= 0 || 2 * H > NT) return fail(ADT_E_SHAPE, "%s", "wcatalog_build: dims (n >= 1, H must be 1..128)");
  const cudaStream_t s = (cudaStream_t)s_;
  double* part = (double*)work;
  unsigned int* counter = (unsigned int*)(part + (int64_t)WCAT_PARTS * 2 * H);
  wcat_mean_kernel<<<WCAT_PARTS, NT, 0, s>>>(mean, cov, n, H, part, counter, mu);
  wcat_rows_kernel<<<min((n + 7) / 8, 148 * 8), NT, 0, s>>>(mean, cov, mu, n, H, rows, bias);
  return check_launch("wcatalog_build");
}
extern "C" int adt_wcatalog_user(const float* mean, const float* cov, const float* mu, float* out, int32_t U, int32_t H, adt_stream_t s_) {
  if (U <= 0 || H <= 0) return fail(ADT_E_SHAPE, "%s", "wcatalog_user: dims");
  const long long blocks = ((long long)U * 2 * H + NT - 1) / NT;
  wcat_user_kernel<<<(int)min(blocks, 148LL * 8), NT, 0, (cudaStream_t)s_>>>(mean, cov, mu, U, H, out);
  return check_launch("wcatalog_user");
}

extern "C" int adt_debug_read(long long* out, int n) {
  cudaDeviceSynchronize();
  return cudaMemcpyFromSymbol(out, g_dbg_clock, sizeof(long long) * (n < 64 ? n : 64)) == cudaSuccess ? ADT_OK : ADT_E_CUDA;
}
