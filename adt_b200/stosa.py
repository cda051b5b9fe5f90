"""STOSA-ADT on B200 (SURVEY 8a row a20): the reference's `DisenDistSAModel` surface composed from libadt_b200.so ops.

Mirrors /root/reference/stosa/models.py:166-270 (constructor reads `args.item_size, hidden_units, maxlen, num_users,
num_layers, num_heads, dropout, attention_dropout, initializer_range`; `finetune(input_ids, dec_ids, user_ids)` -> the
7-tuple; parameter names/shapes identical so reference checkpoints load) and stosa/modules.py (DistAttention,
DistEDAttention, DistIntermediate, DistLayer, DistDecLayer).  Two streams (mean, covariance) run through the generic
linear / dropout+residual+LayerNorm kernels; the Wasserstein attention core (scores in matmul form, additive
padding*causal mask, softmax, dropout, P.v_mean and P^2.v_cov) is one kernel per direction (adt_wattention_fwd/bwd); with
`precision = 1`, shapes whose attention tile does not fit shared memory (up to L 2048, H/nh a multiple of 16 up to 64) run in the
fused tcgen05 flash kernels instead (adt_wattention_flash_fwd/bwd).

`fused_loss` is the B200 training entry (stosa/trainer.py:358-378 + :517-533): BPR + pvn terms on elementwise
Wasserstein distances in one kernel with the four table-row gradients scatter-added through the sorted segmented
scatter, reconstruction and independence terms through the squared-difference / softmax-CE kernels.
`full_sort_topk` replaces `dist_predict_full` + the host-side argpartition over the whole [U, I] matrix
(trainer.py:464-479, :604-614) by the shared full-catalog path (adt_b200.evaluate.CatalogScorer): the Wasserstein distance is
ranked as a centred dot product plus a per-item bias (`scoring_catalog`, `final_feats`).
"""
import ctypes
import math
import numpy as np
import torch
import torch.nn as nn

from . import _lib as L
from .blocks import DropCfg, _scatter
from .ops import DrlFn, linear, no_drop, _st
from .bert4rec import MaskedCE, _ids

ELU, ELU1 = 3, 4   # activation codes of adt_linear_fwd / adt_act_fwd
MAX_CATALOG_HIDDEN = 128   # full-catalog ranking: rows [mean | sqrt cov] of 2H floats, at most 256 for the K7 kernels


class _LN(nn.Module):
    """stosa/modules.py:88-101 (TF-style LayerNorm, eps inside the square root)."""

    def __init__(self, H):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(H))
        self.bias = nn.Parameter(torch.zeros(H))


class _DistAttention(nn.Module):
    def __init__(self, H):
        super().__init__()
        for n in ("mean_query", "cov_query", "mean_key", "cov_key", "mean_value", "cov_value"):
            setattr(self, n, nn.Linear(H, H))
        self.mean_dense, self.cov_dense = nn.Linear(H, H), nn.Linear(H, H)
        self.LayerNorm = _LN(H)


class _DistIntermediate(nn.Module):
    def __init__(self, H):
        super().__init__()
        self.dense_1, self.dense_2 = nn.Linear(H, 4 * H), nn.Linear(4 * H, H)
        self.LayerNorm = _LN(H)


class _DistLayer(nn.Module):
    def __init__(self, H, nh):
        super().__init__()
        self.attention = _DistAttention(H)
        self.mean_intermediate, self.cov_intermediate = _DistIntermediate(H), _DistIntermediate(H)
        self.mean_independence_layer, self.cov_independence_layer = nn.Linear(H // nh, nh), nn.Linear(H // nh, nh)


class _DistDecLayer(nn.Module):
    def __init__(self, H):
        super().__init__()
        self.dec_attention = _DistAttention(H)     # evaluated and discarded by the reference (modules.py:537-538): parameters only
        self.enc_attention = _DistAttention(H)
        self.mean_intermediate, self.cov_intermediate = _DistIntermediate(H), _DistIntermediate(H)


class _Stack(nn.Module):
    def __init__(self, layers):
        super().__init__()
        self.layer = nn.ModuleList(layers)


# ---- autograd bridges ------------------------------------------------------------------------------------------------
class ActFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, act):
        x = x.contiguous()
        y = torch.empty_like(x)
        L.check(L.lib().adt_act_fwd(L.ptr(x), L.ptr(y), ctypes.c_int64(x.numel()), ctypes.c_int32(act), _st(x.device)), "adt_act_fwd")
        ctx.save_for_backward(x)
        ctx.act = act
        return y

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        dy = dy.contiguous()
        dx = torch.empty_like(x)
        L.check(L.lib().adt_act_bwd(L.ptr(dy), L.ptr(x), L.ptr(dx), ctypes.c_int64(x.numel()), ctypes.c_int32(ctx.act), _st(x.device)),
                "adt_act_bwd")
        return dx, None


def _embed_rows(ids, pos_ids, E, P):
    """E[ids] + P[pos_ids] -> [B*L, H]"""
    B, Lq = ids.shape
    H = E.shape[1]
    s = torch.empty(B * Lq, H, dtype=torch.float32, device=E.device)
    L.check(L.lib().adt_gather3(L.ptr(ids), L.ptr(E), L.ptr(pos_ids), L.ptr(P), None, None, L.ptr(s), ctypes.c_int32(B * Lq),
                                ctypes.c_int32(H), _st(E.device)), "adt_gather3")
    return s


class EmbedPairFn(torch.autograd.Function):
    """(E[ids] + P[0..L-1], E[dec_ids] + P[0..L-1]) for one (item, position) table pair; item table has padding_idx=0
    (models.py:169-172), the position table does not."""

    @staticmethod
    def forward(ctx, ids, dec_ids, pos_ids, E, P):
        ctx.ids = (ids, dec_ids, pos_ids)
        ctx.shapes = (E.shape, P.shape)
        return _embed_rows(ids, pos_ids, E, P), _embed_rows(dec_ids, pos_ids, E, P)

    @staticmethod
    def backward(ctx, d_enc, d_dec):
        ids, dec_ids, pos_ids = ctx.ids
        es, ps = ctx.shapes
        B, Lq = ids.shape
        H = es[1]
        dev = d_enc.device
        d_enc, d_dec = d_enc.contiguous(), d_dec.contiguous()
        dE = torch.zeros(es, device=dev)
        _scatter(dev, B * Lq, B, Lq, H, es[0] - 1, seq=ids, dx_enc=d_enc, dec=dec_ids, dx_dec=d_dec, dE=dE, dP=None, emb_scale=1.0)
        dP = torch.zeros(ps, device=dev)
        for d in (d_enc, d_dec):
            L.check(L.lib().adt_small_table_grad(L.ptr(pos_ids), L.ptr(d), L.ptr(dP), ctypes.c_int32(B * Lq), ctypes.c_int32(H),
                                                 ctypes.c_int32(-1), _st(dev)), "adt_small_table_grad")
        return None, None, None, dE, dP


def _resident_fits(Lq, H, nh, backward):
    """the resident (fp32, shared-memory) Wasserstein attention kernels serve this shape; False also for dims they refuse outright"""
    return L.lib().adt_wattention_resident_fits(ctypes.c_int32(Lq), ctypes.c_int32(H), ctypes.c_int32(nh), ctypes.c_int32(int(backward))) == 1


def _wflash_scratch(ref, B, Lq, H, nh, backward):
    f = L.lib().adt_wattention_scratch_bytes
    f.restype = ctypes.c_int64
    n = int(f(ctypes.c_int32(B), ctypes.c_int32(Lq), ctypes.c_int32(H), ctypes.c_int32(nh), ctypes.c_int32(int(backward))))
    return torch.empty(n, dtype=torch.uint8, device=ref.device) if n > 0 else None    # n < 0: refused shape, the launch names why


class WAttnFn(torch.autograd.Function):
    """Wasserstein attention core (modules.py:240-254): six projected streams [B*L,H] -> (mean ctx, cov ctx).

    precision 0 runs the resident fp32 kernels (adt_wattention_fwd/bwd), which refuse shapes whose tile does not fit shared memory.
    precision 1 runs the same kernels where they fit and the tcgen05 flash kernels (adt_wattention_flash_fwd/bwd: bf16 operands, L up to
    2048, H/nh a multiple of 16 up to 64) where they do not: the backward tile decides when a gradient will be needed, else the forward
    tile, so a forward and its backward always take the same path."""

    @staticmethod
    def forward(ctx, mq, cq, mk, ck, mv, cv, key_ids, dims, drop, precision=0):
        B, Lq, nh = dims
        t = [x.contiguous() for x in (mq, cq, mk, ck, mv, cv)]
        H = t[0].shape[1]
        mctx, cctx = torch.empty_like(t[0]), torch.empty_like(t[0])
        lse = torch.empty(B, nh, Lq, 2, dtype=torch.float32, device=mctx.device)
        ctx.flash = precision == 1 and not _resident_fits(Lq, H, nh, any(ctx.needs_input_grad[:6]))
        a = L.fill(L.adt_wattention_args(), mq=t[0], cq=t[1], mk=t[2], ck=t[3], mv=t[4], cv=t[5], mctx=mctx, cctx=cctx, lse=lse,
                   key_ids=key_ids, dmctx=None, dcctx=None, dmq=None, dcq=None, dmk=None, dck=None, dmv=None, dcv=None, B=B, L=Lq, H=H,
                   nh=nh, drop=drop)
        if ctx.flash:
            ws = _wflash_scratch(mctx, B, Lq, H, nh, 0)
            a.tc_scratch = None if ws is None else ws.data_ptr()
            L.check(L.lib().adt_wattention_flash_fwd(ctypes.byref(a), _st(mctx.device)), "adt_wattention_flash_fwd")
            ctx.save_for_backward(*t, lse, mctx, cctx)
        else:
            L.check(L.lib().adt_wattention_fwd(ctypes.byref(a), _st(mctx.device)), "adt_wattention_fwd")
            ctx.save_for_backward(*t, lse)
        ctx.cfg = (key_ids, dims, drop)
        return mctx, cctx

    @staticmethod
    def backward(ctx, dm, dc):
        mq, cq, mk, ck, mv, cv, lse = ctx.saved_tensors[:7]
        key_ids, (B, Lq, nh), drop = ctx.cfg
        H = mq.shape[1]
        g = [torch.empty_like(mq) for _ in range(6)]
        a = L.fill(L.adt_wattention_args(), mq=mq, cq=cq, mk=mk, ck=ck, mv=mv, cv=cv, mctx=None, cctx=None, lse=lse, key_ids=key_ids,
                   dmctx=dm.contiguous(), dcctx=dc.contiguous(), dmq=g[0], dcq=g[1], dmk=g[2], dck=g[3], dmv=g[4], dcv=g[5], B=B, L=Lq,
                   H=H, nh=nh, drop=drop)
        if ctx.flash:
            ws = _wflash_scratch(mq, B, Lq, H, nh, 1)
            a.tc_scratch = None if ws is None else ws.data_ptr()
            a.mctx_in, a.cctx_in = ctx.saved_tensors[7].data_ptr(), ctx.saved_tensors[8].data_ptr()
            L.check(L.lib().adt_wattention_flash_bwd(ctypes.byref(a), _st(mq.device)), "adt_wattention_flash_bwd")
        else:
            L.check(L.lib().adt_wattention_bwd(ctypes.byref(a), _st(mq.device)), "adt_wattention_bwd")
        return (*g, None, None, None, None)


class WBprFn(torch.autograd.Function):
    """trainer.py:358-378 -> (bpr, mean clamp(d_pos - d_pn, 0), auc), each averaged over the target positions."""

    @staticmethod
    def forward(ctx, sm, sc, Em, Ec, pos, neg):
        sm, sc = sm.contiguous(), sc.contiguous()
        M, H = sm.shape
        acc = torch.zeros(4, dtype=torch.float64, device=sm.device)
        a = L.fill(L.adt_wbpr_args(), seq_mean=sm, seq_cov=sc, item_mean=Em, item_cov=Ec, pos=pos, neg=neg, acc=acc, gcoef=None,
                   d_seq_mean=None, d_seq_cov=None, g_pos_mean=None, g_pos_cov=None, g_neg_mean=None, g_neg_cov=None, M=M, H=H)
        L.check(L.lib().adt_wbpr_fwd(ctypes.byref(a), _st(sm.device)), "adt_wbpr_fwd")
        ctx.save_for_backward(sm, sc, Em, Ec, acc)
        ctx.ids = (pos, neg)
        out = (acc[:3] / acc[3]).float()
        return out[0], out[1], out[2]

    @staticmethod
    def backward(ctx, g_bpr, g_pvn, g_auc):
        sm, sc, Em, Ec, acc = ctx.saved_tensors
        pos, neg = ctx.ids
        M, H = sm.shape
        dev = sm.device
        gcoef = (torch.stack([g_bpr, g_pvn]).double() / acc[3]).float().contiguous()
        o = [torch.empty_like(sm) for _ in range(6)]
        a = L.fill(L.adt_wbpr_args(), seq_mean=sm, seq_cov=sc, item_mean=Em, item_cov=Ec, pos=pos, neg=neg, acc=acc, gcoef=gcoef,
                   d_seq_mean=o[0], d_seq_cov=o[1], g_pos_mean=o[2], g_pos_cov=o[3], g_neg_mean=o[4], g_neg_cov=o[5], M=M, H=H)
        L.check(L.lib().adt_wbpr_bwd(ctypes.byref(a), _st(dev)), "adt_wbpr_bwd")
        B, Lq = pos.shape
        dEm, dEc = torch.zeros_like(Em), torch.zeros_like(Ec)
        _scatter(dev, M, B, Lq, H, Em.shape[0] - 1, seq=pos, dx_enc=o[2], dec=neg, dx_dec=o[4], dE=dEm, dP=None, emb_scale=1.0)
        _scatter(dev, M, B, Lq, H, Em.shape[0] - 1, seq=pos, dx_enc=o[3], dec=neg, dx_dec=o[5], dE=dEc, dP=None, emb_scale=1.0)
        return o[0], o[1], dEm, dEc, None, None


class MseFn(torch.autograd.Function):
    """F.mse_loss(a, b) with gradients to both sides (trainer.py:519-520)."""

    @staticmethod
    def forward(ctx, a, b):
        a, b = a.contiguous(), b.contiguous()
        acc = torch.zeros(1, dtype=torch.float64, device=a.device)
        L.check(L.lib().adt_sqdiff_fwd(L.ptr(a), L.ptr(b), ctypes.c_int64(a.numel()), L.ptr(acc), _st(a.device)), "adt_sqdiff_fwd")
        ctx.save_for_backward(a, b)
        return (acc / a.numel()).float().squeeze(0)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        da, db = torch.empty_like(a), torch.empty_like(b)
        g = g.float().reshape(1).contiguous()
        L.check(L.lib().adt_sqdiff_bwd(L.ptr(a), L.ptr(b), L.ptr(g), ctypes.c_float(1.0 / a.numel()), L.ptr(da), L.ptr(db),
                                       ctypes.c_int64(a.numel()), _st(a.device)), "adt_sqdiff_bwd")
        return da, db


# ---- the model -------------------------------------------------------------------------------------------------------
class DisenDistSAModel(nn.Module):
    def __init__(self, args):
        super().__init__()
        H, nh = args.hidden_units, args.num_heads
        if H % nh != 0:
            raise ValueError("The hidden size (%d) is not a multiple of the number of attention heads (%d)" % (H, nh))
        self.args = args
        self.item_mean_embeddings = nn.Embedding(args.item_size, H, padding_idx=0)
        self.item_cov_embeddings = nn.Embedding(args.item_size, H, padding_idx=0)
        self.position_mean_embeddings = nn.Embedding(args.maxlen, H)
        self.position_cov_embeddings = nn.Embedding(args.maxlen, H)
        self.user_margins = nn.Embedding(args.num_users, 1)
        self.item_encoder = _Stack([_DistLayer(H, nh) for _ in range(args.num_layers)])
        self.item_decoder = _Stack([_DistDecLayer(H) for _ in range(args.num_layers)])
        self.LayerNorm = _LN(H)
        self.decLayerNorm = _LN(H)       # present in the reference, never applied
        self.hidden_units, self.num_heads, self.num_layers, self.maxlen = H, nh, args.num_layers, args.maxlen
        self.dropout_p, self.attention_dropout_p = float(args.dropout), float(args.attention_dropout)
        self.pvn_weight = float(getattr(args, "pvn_weight", 0.005))
        self.drop_seed, self.drop_step, self.precision = 0, 0, 0
        self.step_dev = None      # optional device-side dropout step counter (adt_b200.dp.GraphedStep)
        self._wcat, self._wcat_key = None, None   # ranked catalog (mu, rows, bias, scratch) and the _catalog_key it was built from
        self._scorers = {}        # (K, device) -> CatalogScorer of full_sort_topk (keeps its bf16 table and scratch between calls)
        self.apply(self.init_weights)
        L.lib()

    def init_weights(self, module):
        """models.py:262-270."""
        std = float(getattr(self.args, "initializer_range", 0.02))
        if isinstance(module, (nn.Linear, nn.Embedding)):
            module.weight.data.normal_(mean=0.01, std=std)
        elif isinstance(module, _LN):
            module.bias.data.zero_()
            module.weight.data.fill_(1.0)
        if isinstance(module, nn.Linear) and module.bias is not None:
            module.bias.data.zero_()

    # ------------------------------------------------------------------------------------------
    def _check(self):
        if self.LayerNorm.weight.device.type != "cuda":
            raise L.AdtError("adt_b200.DisenDistSAModel runs on CUDA only (no CPU fallback): call .to('cuda') first")

    def _drop(self, dc, kind, p, Lq):
        old = dc.p
        dc.p = p
        d = dc.next(kind, self.num_heads, Lq, self.hidden_units)
        dc.p = old
        return d

    def _embed(self, ids, dec_ids, pos_ids, dc, Lq):
        """models.py:183-210 for both sequences: -> ((mean, cov) of input_ids, (mean, cov) of dec_ids)."""
        ln = self.LayerNorm
        me, md = EmbedPairFn.apply(ids, dec_ids, pos_ids, self.item_mean_embeddings.weight, self.position_mean_embeddings.weight)
        ce, cd = EmbedPairFn.apply(ids, dec_ids, pos_ids, self.item_cov_embeddings.weight, self.position_cov_embeddings.weight)
        out = []
        for s, act in ((me, ELU), (ce, ELU1), (md, ELU), (cd, ELU1)):     # the reference's call order: mean, cov, dec mean, dec cov
            d = self._drop(dc, "row", self.dropout_p, Lq)
            out.append(ActFn.apply(DrlFn.apply(s, None, ln.weight, ln.bias, 1, 1e-12, d), act))
        return (out[0], out[1]), (out[2], out[3])

    def _attention(self, m, qm, qc, km, kc, key_ids, B, Lq, dc):
        """DistAttention / DistEDAttention.forward (modules.py:222-275, :312-361) -> (mean', cov', mean ctx, cov ctx)."""
        pr = self.precision
        lin = lambda mod, x, act=0: linear(x, mod.weight, mod.bias, act, 1.0, pr)
        mq, mk, mv = lin(m.mean_query, qm), lin(m.mean_key, km), lin(m.mean_value, km)
        cq, ck, cv = lin(m.cov_query, qc, ELU1), lin(m.cov_key, kc, ELU1), lin(m.cov_value, kc, ELU1)
        d = self._drop(dc, "attn", self.attention_dropout_p, Lq)
        mctx, cctx = WAttnFn.apply(mq, cq, mk, ck, mv, cv, key_ids, (B, Lq, self.num_heads), d, self.precision)
        ln = m.LayerNorm
        mh = DrlFn.apply(lin(m.mean_dense, mctx), qm, ln.weight, ln.bias, 0, 1e-12, self._drop(dc, "row", self.dropout_p, Lq))
        ch = DrlFn.apply(lin(m.cov_dense, cctx), qc, ln.weight, ln.bias, 0, 1e-12, self._drop(dc, "row", self.dropout_p, Lq))
        return mh, ch, mctx, cctx

    def _intermediate(self, m, x, dc, Lq):
        """DistIntermediate.forward (modules.py:484-494)."""
        h = linear(x, m.dense_1.weight, m.dense_1.bias, ELU, 1.0, self.precision)
        h = linear(h, m.dense_2.weight, m.dense_2.bias, 0, 1.0, self.precision)
        return DrlFn.apply(h, x, m.LayerNorm.weight, m.LayerNorm.bias, 0, 1e-12, self._drop(dc, "row", self.dropout_p, Lq))

    def _encode(self, ids, m, c, dc):
        """the encoder stack (models.py:236-241) on the embedded (mean, cov) streams -> (mean, cov, encoder inputs, independence logits)."""
        B, Lq = ids.shape
        nh, H = self.num_heads, self.hidden_units
        enc_inputs, rec_logits = [], []
        for layer in self.item_encoder.layer:
            enc_inputs.append((m, c))
            am, ac, rm, rc = self._attention(layer.attention, m, c, m, c, ids, B, Lq, dc)
            m = self._intermediate(layer.mean_intermediate, am, dc, Lq)
            c = ActFn.apply(self._intermediate(layer.cov_intermediate, ac, dc, Lq), ELU1)
            mi, ci = layer.mean_independence_layer, layer.cov_independence_layer
            rec_logits.append((linear(rm.view(B * Lq * nh, H // nh), mi.weight, mi.bias, 0, 1.0, 0),
                               linear(rc.view(B * Lq * nh, H // nh), ci.weight, ci.bias, 0, 1.0, 0)))
        return m, c, enc_inputs, rec_logits

    def _body(self, input_ids, dec_ids):
        self._check()
        dev = self.LayerNorm.weight.device
        ids, dec = _ids(input_ids, dev), _ids(dec_ids, dev)
        B, Lq = ids.shape
        pos_ids = torch.arange(Lq, dtype=torch.int32, device=dev).repeat(B, 1)
        dc = DropCfg(self.dropout_p, self.drop_seed, self.drop_step, self.training, step_dev=self.step_dev)
        (m, c), (dm, dcv) = self._embed(ids, dec, pos_ids, dc, Lq)
        m, c, enc_inputs, rec_logits = self._encode(ids, m, c, dc)
        dec_outs = []
        for layer in self.item_decoder.layer:
            # the reference evaluates dec_attention and discards it (modules.py:537-538): only its three dropout sites are consumed
            self._drop(dc, "attn", self.attention_dropout_p, Lq)
            self._drop(dc, "row", self.dropout_p, Lq)
            self._drop(dc, "row", self.dropout_p, Lq)
            am, ac, _, _ = self._attention(layer.enc_attention, dm, dcv, m, c, ids, B, Lq, dc)
            dm = self._intermediate(layer.mean_intermediate, am, dc, Lq)
            dcv = ActFn.apply(self._intermediate(layer.cov_intermediate, ac, dc, Lq), ELU1)
            dec_outs.append((dm, dcv))
        if self.training:
            self.drop_step += 1
        return m, c, enc_inputs, rec_logits, dec_outs, (B, Lq)

    def finetune(self, input_ids, dec_ids, user_ids):
        """models.py:212-260 -> (mean [B,L,H], cov, att_scores, margins, encoder inputs, encoder recs, decoder outputs).
        `att_scores` (the last layer's [B,nh,L,L] probabilities, read by nobody) is not materialised: None."""
        m, c, enc_inputs, rec_logits, dec_outs, (B, Lq) = self._body(input_ids, dec_ids)
        H, nh = self.hidden_units, self.num_heads
        v = lambda t: t.view(B, Lq, H)
        recs = [[torch.log_softmax(a.view(B, Lq, nh, nh), dim=3), torch.log_softmax(b.view(B, Lq, nh, nh), dim=3)] for a, b in rec_logits]
        margins = self.user_margins.weight[torch.as_tensor(np.asarray(user_ids.cpu() if isinstance(user_ids, torch.Tensor) else user_ids))
                                           .to(self.user_margins.weight.device).long()]
        return v(m), v(c), None, margins, [[v(a), v(b)] for a, b in enc_inputs], recs, [[v(a), v(b)] for a, b in dec_outs]

    def fused_loss(self, input_ids, dec_ids, pos_ids, neg_ids, lambda1, lambda2):
        """trainer.py:512-534 -> (loss, bpr, pvn_loss, auc); `loss.backward()` runs the CUDA adjoints."""
        m, c, enc_inputs, rec_logits, dec_outs, (B, Lq) = self._body(input_ids, dec_ids)
        dev = m.device
        pos, neg = _ids(pos_ids, dev), _ids(neg_ids, dev)
        bpr, pvn_raw, auc = WBprFn.apply(m, c, self.item_mean_embeddings.weight, self.item_cov_embeddings.weight, pos, neg)
        pvn = self.pvn_weight * pvn_raw
        total = bpr
        dec_rev = list(reversed(dec_outs))
        for l in range(self.num_layers):
            if lambda1[l] != 0:
                total = total + lambda1[l] * (MseFn.apply(enc_inputs[l][0], dec_rev[l][0]) + MseFn.apply(enc_inputs[l][1], dec_rev[l][1]))
        nh = self.num_heads
        label = torch.arange(nh, dtype=torch.int32, device=dev).repeat(B * Lq)
        for l in range(self.num_layers):
            if lambda2[l] != 0:
                total = total + lambda2[l] * (MaskedCE.apply(rec_logits[l][0], label) + MaskedCE.apply(rec_logits[l][1], label))
        return total + pvn, bpr, pvn, auc

    # ---- evaluation ---------------------------------------------------------------------------
    @torch.no_grad()
    def _last_states(self, input_ids):
        """(mean, cov) [U, H] of the last position in evaluation mode: embedding + encoder only (the decoder does not feed the
        ranking)."""
        self._check()
        dev = self.LayerNorm.weight.device
        ids = _ids(input_ids, dev)
        B, Lq = ids.shape
        H, ln = self.hidden_units, self.LayerNorm
        pos_ids = torch.arange(Lq, dtype=torch.int32, device=dev).repeat(B, 1)
        mc = []
        for E, P, act in ((self.item_mean_embeddings, self.position_mean_embeddings, ELU),
                          (self.item_cov_embeddings, self.position_cov_embeddings, ELU1)):
            s = _embed_rows(ids, pos_ids, E.weight, P.weight)
            mc.append(ActFn.apply(DrlFn.apply(s, None, ln.weight, ln.bias, 1, 1e-12, no_drop()), act))
        m, c, _, _ = self._encode(ids, mc[0], mc[1], DropCfg(0.0, 0, 0, False))
        return m.view(B, Lq, H)[:, -1, :].contiguous(), c.view(B, Lq, H)[:, -1, :].contiguous()

    def _rows(self, mean, cov, is_user):
        n, H = mean.shape
        out = torch.empty(n, 2 * H + 4, dtype=torch.float32, device=mean.device)
        L.check(L.lib().adt_wcatalog_rows(L.ptr(mean), L.ptr(cov), L.ptr(out), ctypes.c_int32(n), ctypes.c_int32(H), ctypes.c_int32(is_user),
                                          _st(mean.device)), "adt_wcatalog_rows")
        return out

    @torch.no_grad()
    def dist_predict_full(self, seq_mean_out, seq_cov_out):
        """trainer.py:464-479: Wasserstein distance matrix [U, item_size] (smaller is better)."""
        u = self._rows(seq_mean_out.contiguous(), seq_cov_out.contiguous(), 1)
        cat = self._rows(self.item_mean_embeddings.weight, self.item_cov_embeddings.weight, 0)
        neg = linear(u, cat, None, 0, 1.0, 0)                                   # = -distance + (|mean_u|^2 + sum cov_u)
        const = (seq_mean_out ** 2).sum(-1, keepdim=True) + seq_cov_out.sum(-1, keepdim=True)
        return const - neg

    def _catalog_key(self):
        """what the ranked catalog is derived from, read on the host (launches nothing): storage and in-place version of both item
        tables, and this package's optimisers' raw-pointer writes (_adt_param_version)."""
        Em, Ec = self.item_mean_embeddings.weight, self.item_cov_embeddings.weight
        return (Em.data_ptr(), Em._version, Ec.data_ptr(), Ec._version, getattr(self, "_adt_param_version", 0))

    def _build_catalog(self):
        """(re)build mu, the centred rows and their bias from the current item tables, in place when the shapes are unchanged so that a
        captured evaluation graph keeps reading the same buffers."""
        key = self._catalog_key()
        Em, Ec = self.item_mean_embeddings.weight.detach(), self.item_cov_embeddings.weight.detach()
        n, H = Em.shape
        if H > MAX_CATALOG_HIDDEN or H % 2:
            raise L.AdtError(f"STOSA full-catalog ranking needs an even hidden size <= {MAX_CATALOG_HIDDEN} (rows of 2H <= 256 floats); "
                             f"got hidden_units = {H}")
        self._check()
        dev = Em.device
        if self._wcat is None or self._wcat[1].shape != (n, 2 * H) or self._wcat[1].device != dev:
            nb = ctypes.c_int64(0)
            L.check(L.lib().adt_wcatalog_work_bytes(ctypes.c_int32(H), ctypes.byref(nb)), "adt_wcatalog_work_bytes")
            self._wcat = (torch.empty(2 * H, device=dev), torch.empty(n, 2 * H, device=dev), torch.empty(n, device=dev),
                          torch.zeros(nb.value, dtype=torch.uint8, device=dev))
        mu, e, b, work = self._wcat
        L.check(L.lib().adt_wcatalog_build(L.ptr(Em), L.ptr(Ec), ctypes.c_int32(n), ctypes.c_int32(H), L.ptr(mu), L.ptr(e), L.ptr(b),
                                           L.ptr(work), _st(dev)), "adt_wcatalog_build")
        self._wcat_key = key

    def scoring_catalog(self):
        """what full-catalog ranking scores (adt_b200.evaluate.catalog_of): -distance(u, i) + const(u) = <final_feats[u], e_i> + b_i with
        e_i = y_i - mu, b_i = -|e_i|^2 over all item_size rows from id 0 (y_i = [mean_i | sqrt(elu(cov_i)+1)], mu their column mean).
        The model-owned rows are rebuilt here, in place, whenever an item table changed since the last build (never during stream
        capture: a captured graph reads the buffers as they stand).  `version` tells CatalogScorer when its bf16 copy is stale."""
        from .evaluate import Catalog
        if self._wcat_key != self._catalog_key():
            if not (self.item_mean_embeddings.weight.is_cuda and torch.cuda.is_current_stream_capturing()):
                self._build_catalog()
            elif self._wcat is None:
                raise L.AdtError("the STOSA catalog is built outside stream capture: rank once (or call scoring_catalog()) before capturing")
        _, e, b, _ = self._wcat
        return Catalog(e, b, 0, e.shape[1], self._wcat_key)

    @torch.no_grad()
    def final_feats(self, seqs):
        """[U, 2H] rows the catalog is scored against: 2 ([mean_u | sqrt(cov_u)] - mu) of the last position, encoder in evaluation
        mode.  No host synchronisation, so a CUDA graph can capture it (GraphedScorer)."""
        return self.user_feats(*self._last_states(seqs))

    @torch.no_grad()
    def user_feats(self, mean, cov):
        """last-position (mean, cov) [U, H] (cov already ELU+1) -> the [U, 2H] rows 2 ([mean | sqrt(cov)] - mu)."""
        self.scoring_catalog()
        mu = self._wcat[0]
        mean, cov = mean.contiguous(), cov.contiguous()
        U, H = mean.shape
        f = torch.empty(U, 2 * H, dtype=torch.float32, device=mean.device)
        L.check(L.lib().adt_wcatalog_user(L.ptr(mean), L.ptr(cov), L.ptr(mu), L.ptr(f), ctypes.c_int32(U), ctypes.c_int32(H),
                                          _st(mean.device)), "adt_wcatalog_user")
        return f

    @torch.no_grad()
    def full_sort_topk(self, input_ids, seen_indptr=None, seen_idx=None, K=40, answers=None, metric_acc=None):
        """trainer.py:596-614 -> ids [U, K] of the K nearest unseen items, nearest first (ties by ascending id).  Seen ids: CSR, ascending
        per user.  answers [U] + metric_acc (float64 device tensor [6]): fused HIT/NDCG@5,10 + MRR sums, as in CatalogScorer.topk."""
        from .evaluate import CatalogScorer
        key = (int(K), self.item_mean_embeddings.weight.device)
        if key not in self._scorers:
            self._scorers[key] = CatalogScorer(self, K=K)
        return self._scorers[key].topk(input_ids, seen_indptr, seen_idx, answers, metric_acc)[1]
