"""torch.autograd bridges over the generic C-ABI ops (include/adt_b200.h "generic ops"): linear, dropout+residual+
LayerNorm, attention core, three-table embedding sum.  Used to compose the post-LN backbones on the host
(bert4rec.py); every device op is a libadt_b200.so kernel."""
import ctypes
import torch

from . import _lib as L
from .blocks import _scatter


def _st(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


NBLK = 1024   # column block of wide linear layers


def no_drop():
    return L.adt_dropout()


SM_COUNT = 148
TC_MIN_WORK = 1 << 22     # M*N*K below this: the row-tile kernel's single launch beats convert + GEMM


def _ceil8(n):
    return (n + 7) // 8 * 8


def _bf16(x, transpose=False):
    """bf16 operand copy of a contiguous fp32 matrix [R, C] (leading dimension padded to a multiple of 8 for TMA), or of its transpose"""
    lib = L.lib()
    R, C = x.shape
    st = _st(x.device)
    if transpose:
        ld = _ceil8(R)
        y = torch.empty(C, ld, dtype=torch.bfloat16, device=x.device)
        if ld != R:
            y[:, R:].zero_()
        L.check(lib.adt_to_bf16_t(L.ptr(x), ctypes.c_int64(x.stride(0)), L.ptr(y), ctypes.c_int64(ld), ctypes.c_int32(R), ctypes.c_int32(C), st),
                "adt_to_bf16_t")
        return y, ld
    ld = _ceil8(C)
    y = torch.empty(R, ld, dtype=torch.bfloat16, device=x.device)
    if ld != C:
        y[:, C:].zero_()
    L.check(lib.adt_to_bf16_ld(L.ptr(x), ctypes.c_int64(x.stride(0)), L.ptr(y), ctypes.c_int64(ld), ctypes.c_int64(R), ctypes.c_int32(C), st),
            "adt_to_bf16_ld")
    return y, ld


def _gemm_tc(a16, lda, b16, ldb, c, M, N, K, bias=None, act=0, scale=1.0, pre=None, accumulate=False, a_mn=False, b_mn=False, split_k=1):
    a = L.fill(L.adt_gemm_tc_args(), a_bf16=a16, b_bf16=b16, lda=lda, ldb=ldb, c=c, pre=pre, bias=bias, ldc=c.stride(0), M=M, N=N, K=K,
               act=act, accumulate=int(accumulate), scale=scale, a_mn=int(a_mn), b_mn=int(b_mn), split_k=split_k)
    L.check(L.lib().adt_gemm_tc(ctypes.byref(a), _st(c.device)), "adt_gemm_tc")


def _use_tc(precision, M, N, K):
    return bool(precision) and M >= 128 and M * N * K >= TC_MIN_WORK and torch.cuda.get_device_capability()[0] >= 10


FLASH_MIN_L = 257   # sequences at least this long run in the fused flash attention kernels (adt_attention_fwd / _bwd dispatch)


def _attn_scratch(ref, B, Lq, H, nh, precision, backward):
    """scratch of the tcgen05 attention paths (bf16 mode): at 65..256 positions the batched path's packed bf16 operands, scores and
    probabilities in HBM; at 257..2048 positions the fused flash kernels' packed bf16 operands (+ bf16 dctx and the row sums of
    dctx * ctx in the backward), O(B L H) with no L^2 term"""
    if not precision or torch.cuda.get_device_capability()[0] < 10:
        return None
    f = L.lib().adt_attention_scratch_bytes
    f.restype = ctypes.c_int64
    n = int(f(ctypes.c_int32(B), ctypes.c_int32(Lq), ctypes.c_int32(H), ctypes.c_int32(nh), ctypes.c_int32(backward)))
    return torch.empty(n, dtype=torch.uint8, device=ref.device) if n else None


class LinearFn(torch.autograd.Function):
    """y = act((x W^T + b) * scale), x [M,K], W [N,K]  (act: 0 none, 1 relu, 2 gelu)."""

    @staticmethod
    def forward(ctx, x, W, b, act, scale, precision):
        x = x.contiguous()
        M, K = x.shape
        N = W.shape[0]
        y = torch.empty(M, N, dtype=torch.float32, device=x.device)
        pre = torch.empty_like(y) if act else None
        if _use_tc(precision, M, N, K):   # tcgen05 GEMM on bf16 operand copies (fp32 accumulate, fp32 bias / activation epilogue)
            x16, lda = _bf16(x)
            w16, ldb = _bf16(W)
            _gemm_tc(x16, lda, w16, ldb, y, M, N, K, bias=b, act=act, scale=scale, pre=pre)
            ctx.save_for_backward(x, W, pre if pre is not None else y)
            ctx.cfg = (act, scale, precision, b is not None)
            return y
        for n0 in range(0, N, NBLK):      # wide outputs (the vocabulary head) are produced in column blocks
            n1 = min(N, n0 + NBLK)
            a = L.fill(L.adt_linear_fwd_args(), x=x, w=W[n0:n1], b=b[n0:n1] if b is not None else None, y=y[:, n0:n1],
                       pre=pre[:, n0:n1] if pre is not None else None, M=M, K=K, N=n1 - n0, act=act, scale=scale, precision=precision, ldy=N)
            L.check(L.lib().adt_linear_fwd(ctypes.byref(a), _st(x.device)), "adt_linear_fwd")
        ctx.save_for_backward(x, W, pre if pre is not None else y)
        ctx.cfg = (act, scale, precision, b is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, W, pre = ctx.saved_tensors
        act, scale, precision, has_b = ctx.cfg
        M, K = x.shape
        N = W.shape[0]
        dy = dy.contiguous()
        lib = L.lib()
        if act:
            dpre = torch.empty_like(dy)
            L.check(lib.adt_act_bwd(L.ptr(dy), L.ptr(pre), L.ptr(dpre), ctypes.c_int64(dy.numel()), ctypes.c_int32(act), _st(x.device)),
                    "adt_act_bwd")
            dy = dpre
        dx = torch.empty_like(x)
        gW = torch.zeros_like(W)
        gb = torch.zeros(N, dtype=torch.float32, device=x.device) if has_b else None
        if _use_tc(precision, M, N, K):
            # dx = scale * dy W ; dW = scale * dy^T x ; db = scale * colsum(dy): three more products on the tensor cores
            # (W, dy and x are read MN-major where the product needs their transpose: no transposed copies)
            dy16, ldd = _bf16(dy)
            w16, ldw = _bf16(W)
            x16, ldx = _bf16(x)
            _gemm_tc(dy16, ldd, w16, ldw, dx, M, K, N, scale=scale, b_mn=True)
            tiles = ((N + 127) // 128) * ((K + 127) // 128)
            _gemm_tc(dy16, ldd, x16, ldx, gW, N, K, M, scale=scale, a_mn=True, b_mn=True, accumulate=True,
                     split_k=max(1, min((M + 63) // 64, SM_COUNT // tiles)))
            if has_b:
                L.check(lib.adt_colsum(L.ptr(dy), ctypes.c_int64(dy.stride(0)), ctypes.c_int32(M), ctypes.c_int32(N), L.ptr(gb), _st(x.device)),
                        "adt_colsum")
                if scale != 1.0:
                    gb.mul_(scale)
            return dx, gW, gb, None, None, None
        for n0 in range(0, N, NBLK):
            n1 = min(N, n0 + NBLK)
            a = L.fill(L.adt_linear_bwd_args(), x=x, w=W[n0:n1], dy=dy[:, n0:n1], dx=dx, g_w=gW[n0:n1], g_b=gb[n0:n1] if has_b else None,
                       M=M, K=K, N=n1 - n0, accumulate_dx=1 if n0 else 0, scale=scale, precision=precision, lddy=N)
            L.check(lib.adt_linear_bwd(ctypes.byref(a), _st(x.device)), "adt_linear_bwd")
        return dx, gW, gb, None, None, None


def linear(x, W, b=None, act=0, scale=1.0, precision=0):
    return LinearFn.apply(x, W, b, act, scale, precision)


LINEAR_CE_SCRATCH = 256 << 20   # bytes of the fused head's vocabulary-chunk scratch (bf16 dS [R, Vc] + the forward's per-tile partials)


def linear_ce_plan(R, V, H, scratch_bytes):
    """(vocab_chunk, min_scratch_bytes) of adt_linear_ce_plan; raises when scratch_bytes is below the minimum."""
    vc, mn = ctypes.c_int32(0), ctypes.c_int64(0)
    L.check(L.lib().adt_linear_ce_plan(ctypes.c_int32(R), ctypes.c_int32(V), ctypes.c_int32(H), ctypes.c_int64(scratch_bytes), ctypes.byref(vc),
                                       ctypes.byref(mn)), "adt_linear_ce_plan")
    return vc.value, mn.value


def linear_ce_scratch_bytes(R, V, H, budget=None):
    """scratch the fused head is given: `budget` (default LINEAR_CE_SCRATCH), at least the planner's minimum, at most what one chunk
    covering all of V needs."""
    budget = LINEAR_CE_SCRATCH if budget is None else budget
    _, mn = linear_ce_plan(R, V, H, 1 << 62)
    # one chunk covering V: 2 R bytes of dS and 8 R / 128 of partials per column, 12 R of row state, 256-byte alignment of four areas
    full = 264 * R * ((V + 127) // 128) + 12 * R + 1024
    return max(mn, min(budget, full))


class LinearCE(torch.autograd.Function):
    """mean over rows of cross_entropy(h W^T + b, labels) on the tcgen05 fused head (adt_linear_ce_fwd / _bwd): the [R, V] logits are
    never materialised.  Saves the bf16 copies of h and W and the per-row log-sum-exp; the backward recomputes the scores chunk by chunk."""

    @staticmethod
    def forward(ctx, h, W, b, labels, scratch_bytes):
        h = h.contiguous()
        R, H = h.shape
        V = W.shape[0]
        dev = h.device
        x16, ldx = _bf16(h)
        w16, ldw = _bf16(W.contiguous())
        b = b.contiguous() if b is not None else None
        labels = labels.to(device=dev, dtype=torch.int32).contiguous()
        nbytes = linear_ce_scratch_bytes(R, V, H, scratch_bytes)
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        lse = torch.empty(R, dtype=torch.float32, device=dev)
        acc = torch.zeros(1, dtype=torch.float64, device=dev)
        a = L.fill(L.adt_linear_ce_args(), x_bf16=x16, w_bf16=w16, ldx=ldx, ldw=ldw, bias=b, labels=labels, R=R, V=V, H=H, lse=lse,
                   loss_acc=acc, scratch=scratch, scratch_bytes=nbytes)
        L.check(L.lib().adt_linear_ce_fwd(ctypes.byref(a), _st(dev)), "adt_linear_ce_fwd")
        ctx.save_for_backward(x16, w16, b, labels, lse)
        ctx.cfg = (ldx, ldw, W.shape, nbytes)
        return (acc / R).float().squeeze(0)

    @staticmethod
    def backward(ctx, g):
        x16, w16, b, labels, lse = ctx.saved_tensors
        ldx, ldw, wshape, nbytes = ctx.cfg
        R, V, H = lse.shape[0], wshape[0], wshape[1]
        dev = lse.device
        g = g.detach().float().reshape(1).contiguous()     # the upstream gradient stays on the device: no host sync
        dx = torch.empty(R, H, dtype=torch.float32, device=dev)
        gW = torch.zeros(wshape, dtype=torch.float32, device=dev)
        gb = torch.zeros(V, dtype=torch.float32, device=dev) if b is not None else None
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        a = L.fill(L.adt_linear_ce_args(), x_bf16=x16, w_bf16=w16, ldx=ldx, ldw=ldw, bias=b, labels=labels, R=R, V=V, H=H,
                   lse=lse, coef=1.0 / R, coef_dev=g, dx=dx, g_w=gW, g_bias=gb, scratch=scratch, scratch_bytes=nbytes)
        L.check(L.lib().adt_linear_ce_bwd(ctypes.byref(a), _st(dev)), "adt_linear_ce_bwd")
        return dx, gW, gb, None, None


def linear_cross_entropy(h, W, b, labels, scratch_bytes=None):
    """mean_r [logsumexp_v(h_r . W_v + b_v) - (h_r . W_{labels[r]} + b_{labels[r]})] with bf16 products and fp32 accumulation, without the
    [R, V] logits: h [R, H] fp32, W [V, H] fp32, b [V] fp32 or None, labels [R] in [0, V).  Differentiable in h, W and b.  Needs sm_100."""
    if h.shape[0] < 1:
        raise L.AdtError("linear_cross_entropy: no rows")
    if torch.cuda.get_device_capability(h.device) != (10, 0):
        raise L.AdtError("linear_cross_entropy runs on the sm_100 tensor cores only")
    return LinearCE.apply(h, W, b, labels, scratch_bytes)


class DrlFn(torch.autograd.Function):
    """mode 0: LN(dropout(a) + r) ; mode 1: dropout(LN(a + r)).  r may be None."""

    @staticmethod
    def forward(ctx, a, r, gamma, beta, mode, eps, drop):
        a = a.contiguous()
        r = r.contiguous() if r is not None else None
        M, H = a.shape
        y = torch.empty_like(a)
        args = L.fill(L.adt_drl_args(), a=a, r=r, gamma=gamma, beta=beta, y=y, dy=None, da=None, dr=None, g_gamma=None, g_beta=None, M=M,
                      H=H, mode=mode, eps=eps, drop=drop)
        L.check(L.lib().adt_drop_res_ln_fwd(ctypes.byref(args), _st(a.device)), "adt_drop_res_ln_fwd")
        ctx.save_for_backward(a, r if r is not None else a, gamma, beta)
        ctx.cfg = (mode, eps, drop, r is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        a, r, gamma, beta = ctx.saved_tensors
        mode, eps, drop, has_r = ctx.cfg
        M, H = a.shape
        dy = dy.contiguous()
        da = torch.empty_like(a)
        dr = torch.empty_like(a) if has_r else None
        gg, gb = torch.zeros_like(gamma), torch.zeros_like(beta)
        args = L.fill(L.adt_drl_args(), a=a, r=r if has_r else None, gamma=gamma, beta=beta, y=None, dy=dy, da=da, dr=dr, g_gamma=gg,
                      g_beta=gb, M=M, H=H, mode=mode, eps=eps, drop=drop)
        L.check(L.lib().adt_drop_res_ln_bwd(ctypes.byref(args), _st(a.device)), "adt_drop_res_ln_bwd")
        return da, dr, gg, gb, None, None, None


class AttnFn(torch.autograd.Function):
    """attention core on projected q (pre-scaled), k, v [B*L, H] -> ctx [B*L, H]."""

    @staticmethod
    def forward(ctx, q, k, v, key_ids, dims, drop, training, precision):
        B, Lq, nh, mask_mode = dims
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        H = q.shape[1]
        out = torch.empty_like(q)
        lse = torch.empty(B, nh, Lq, dtype=torch.float32, device=q.device)
        ws = _attn_scratch(q, B, Lq, H, nh, precision, 0)
        a = L.fill(L.adt_attention_args(), q=q, k=k, v=v, ctx=out, lse=lse, key_ids=key_ids, dctx=None, dq=None, dk=None, dv=None, B=B,
                   L=Lq, H=H, nh=nh, mask_mode=mask_mode, training=int(training), drop=drop, precision=precision, tc_scratch=ws)
        L.check(L.lib().adt_attention_fwd(ctypes.byref(a), _st(q.device)), "adt_attention_fwd")
        # the flash backward (L > 256) reads the forward's output for its row sums of dctx * ctx
        ctx.save_for_backward(q, k, v, lse, out if Lq >= FLASH_MIN_L else None)
        ctx.cfg = (key_ids, dims, drop, training, precision)
        return out

    @staticmethod
    def backward(ctx, dctx):
        q, k, v, lse, out = ctx.saved_tensors
        key_ids, (B, Lq, nh, mask_mode), drop, training, precision = ctx.cfg
        H = q.shape[1]
        dq, dk, dv = torch.empty_like(q), torch.empty_like(q), torch.empty_like(q)
        d = drop
        if not training:
            d = no_drop()
        ws = _attn_scratch(q, B, Lq, H, nh, precision, 1)
        a = L.fill(L.adt_attention_args(), q=q, k=k, v=v, ctx=out, lse=lse, key_ids=key_ids, dctx=dctx.contiguous(), dq=dq, dk=dk, dv=dv,
                   B=B, L=Lq, H=H, nh=nh, mask_mode=mask_mode, training=int(training), drop=d, precision=precision, tc_scratch=ws)
        L.check(L.lib().adt_attention_bwd(ctypes.byref(a), _st(q.device)), "adt_attention_bwd")
        return dq, dk, dv, None, None, None, None, None


class Gather3Fn(torch.autograd.Function):
    """s = word[ids] + pos[pos_ids] + sent[sent_ids]; all three tables have padding_idx=0 (no lookup gradient for row 0)."""

    @staticmethod
    def forward(ctx, ids, pos_ids, sent_ids, word, pos, sent):
        B, Lq = ids.shape
        H = word.shape[1]
        s = torch.empty(B * Lq, H, dtype=torch.float32, device=word.device)
        L.check(L.lib().adt_gather3(L.ptr(ids), L.ptr(word), L.ptr(pos_ids), L.ptr(pos), L.ptr(sent_ids), L.ptr(sent), L.ptr(s),
                                    ctypes.c_int32(B * Lq), ctypes.c_int32(H), _st(word.device)), "adt_gather3")
        ctx.ids = (ids, pos_ids, sent_ids)
        ctx.shapes = (word.shape, pos.shape, sent.shape)
        return s

    @staticmethod
    def backward(ctx, ds):
        ids, pos_ids, sent_ids = ctx.ids
        ws, ps, ss = ctx.shapes
        B, Lq = ids.shape
        H = ws[1]
        dev = ds.device
        ds = ds.contiguous()
        dW = torch.zeros(ws, device=dev)
        _scatter(dev, B * Lq, B, Lq, H, ws[0] - 1, seq=ids, dx_enc=ds, dE=dW, dP=None, emb_scale=1.0)
        dP, dS = torch.zeros(ps, device=dev), torch.zeros(ss, device=dev)
        lib = L.lib()
        for idx, g in ((pos_ids, dP), (sent_ids, dS)):
            L.check(lib.adt_small_table_grad(L.ptr(idx), L.ptr(ds), L.ptr(g), ctypes.c_int32(B * Lq), ctypes.c_int32(H), ctypes.c_int32(0),
                                             _st(dev)), "adt_small_table_grad")
        return None, None, None, dW, dP, dS
