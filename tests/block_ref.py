"""fp64 references of one SASRec-ADT encoder or decoder block, forward and backward, for the block C ABI tests.

The block is oracle.sasrec_oracle.encoder_layer / decoder_layer.  Its matrix products go through an oracle.Products hook:
  - PLAIN evaluates every product in fp64 on the operands as they are;
  - BF16 rounds every operand of every product to bf16 (round to nearest even) and accumulates in fp64, in the forward and in both
    backward products (dgrad rb(g) rb(W), wgrad rb(g)^T rb(x)), as the tensor-core kernels feed their MMAs.
LayerNorm, biases, residuals, dropout, the pad mask and the independence head stay the oracle's own, in fp64, on either hook.

Rounding plan (the points where a bf16 route rounds, read from the kernels; the BF16 hook follows the default column):

  point                          default (BF16 hook)                       routes that depart
  weights                        rb(W): RN cast (cast_bf16_kernel) or the  --
                                 adt_wmirror copy, which holds the same RN
                                 bits (adt_adam / adt_to_bf16)
  q operand of q k^T             rb(q) after the 1/sqrt(hd) scale: the     --
                                 saved q is scaled (kernels_fwd.cuh:79)
  P~ operand of P~ v             rb(P * m / l): normalised, then rounded   flash (L > 256): rb(exp(s - m_run) m) against the
                                 (kernels_attn_small.cuh:264-276,          running max, ctx = O / l at the end
                                 block_tc.cuh:539-542)                     (flash_tc.cu:14-15, :129, :159)
  backward P                     exp(s - lse) with the fp32 lse            --
                                 (kernels_attn_small.cuh:350)
  delta = rowsum(dP P)           fp64 sum of dP P                          flash: rowsum(dctx ctx) in fp32 (flash_tc.cu:17)
  dS, P~, dctx operands          rb(dS), rb(P m), rb(dctx)                 --
                                 (kernels_attn_small.cuh:371-374)
  masked keys, mask mode 1       s = -1e9, dS flows back into q and k as   --
                                 if s were q k^T (the fp32 lse of a fully
                                 padded row is -1e9, so P = 1 there)
  bias and LayerNorm gradients   fp32 sums of the unrounded adjoint        --
  in-projection adjoint operand   rb(dq * qscale), rb(dk), rb(dv): the      --
                                 H = 64 backward stages dq scaled by qscale
                                 as a bf16 tile (kernels_rowtile_small.cuh:
                                 838, :911); the BF16 hook's dgrad rounds
                                 the same scaled adjoint
  independence head              fp32 on the fp32 ctx                      H = 64 row kernels: bf16 ctx tile
                                 (block_tc.cuh:81, kernels_fwd.cuh:314)    (kernels_rowtile_small.cuh:427, :777)
The departures are left to the measured bounds of tests/test_block_fp64_gpu.py; DESIGN.md section 5 lists what they cost.

Two kinds of ties are not departures and are not modelled.  A value that lies on a bf16 rounding boundary can round up in one
evaluation and down in the other, because fp32 and fp64 sums differ in their last bits.  For example, LN(x) feeding the encoder's q
projection does this: one such element moves q by about 4e-4 of its max, while k and v, which round the fp32 input x itself, agree
to 1e-7.  Second, an FFN pre-activation close to zero can take different signs in the two evaluations (see follow_relu_signs).
"""
import numpy as np
import torch

from oracle import sasrec_oracle as O


def rb(t):
    """round to bf16 (nearest even) and back to fp64"""
    return t.to(torch.bfloat16).double()


def _ident(t):
    return t


class _Bf16Linear(torch.autograd.Function):
    """x W^T on bf16-rounded operands with fp64 accumulation; both backward products on bf16-rounded operands"""

    @staticmethod
    def forward(ctx, x, w):
        ctx.save_for_backward(x, w)
        return rb(x) @ rb(w).T

    @staticmethod
    def backward(ctx, g):
        x, w = ctx.saved_tensors
        gr = rb(g)
        return gr @ rb(w), gr.reshape(-1, g.shape[-1]).T @ rb(x).reshape(-1, x.shape[-1])


class _Attention(torch.autograd.Function):
    """attention core of the kernels: scores on rounded q, k; masked scores replaced (-inf causal, -1e9 key padding); P~ = r(P m);
    the backward takes P = exp(s - lse) with the fp32-rounded lse and feeds r(dctx), r(dS), r(P m) to its products"""

    @staticmethod
    def forward(ctx, q, k, v, m, masked, fill, r, lse_out):
        Q, K, V = r(q), r(k), r(v)
        S = torch.where(masked, torch.full_like(q[..., :1], fill), Q @ K.transpose(-1, -2))
        lse = torch.logsumexp(S, -1)
        P = torch.exp(S - lse[..., None])
        out = r(P * m) @ V
        lse_out.append(lse)
        ctx.save_for_backward(Q, K, V, S, lse, m)
        ctx.r = r
        return out

    @staticmethod
    def backward(ctx, dO):
        Q, K, V, S, lse, m = ctx.saved_tensors
        r = ctx.r
        P = torch.exp(S - lse.float().double()[..., None])
        dOr = r(dO)
        dP = (dOr @ V.transpose(-1, -2)) * m
        dS = P * (dP - (dP * P).sum(-1, keepdim=True))
        dSr = r(dS)
        return dSr @ K, dSr.transpose(-1, -2) @ Q, r(P * m).transpose(-1, -2) @ dOr, None, None, None, None, None


# ReLU ties: an FFN pre-activation within KINK_TOL * max |h1| of zero may come out with the other sign in the kernel's fp32 sums than
# in the fp64 reference.  The forward barely notices (relu(h) ~ 0 either way), but the backward's relu'(h) switches a whole element of
# dh1 on or off, and that element reaches dctx, dx and every weight gradient upstream of it.  Given the kernel's saved h1, the
# reference follows the kernel's sign at such ties (h -> -h, with the gradient passing through unchanged); a sign that differs on a
# larger pre-activation is a kernel error and fails the comparison.
KINK_TOL = 1e-2


def follow_relu_signs(y, kernel_h1):
    """y: reference FFN pre-activation; kernel_h1: the kernel's, same shape -> y with the kernel's sign at ties (see KINK_TOL)"""
    k = torch.as_tensor(kernel_h1, dtype=torch.float64).view(y.shape)
    flip = (k > 0) != (y.detach() > 0)
    big = flip & (y.detach().abs() > KINK_TOL * float(y.detach().abs().max()))
    assert not bool(big.any()), f"FFN pre-activation of the other sign beyond a rounding tie at {int(big.sum())} elements"
    return y - (2 * y.detach()) * flip


class Products(O.Products):
    """product hook of one block call: bf16 or plain operands, the mask mode, and a record of every product's operands and result
    (the saved activations of the kernels are read from it).  relu_from = (index of the FFN's first linear among the block's
    products, the kernel's saved h1) makes the reference follow the kernel's sign at ReLU ties (follow_relu_signs)."""

    def __init__(self, bf16, mask_mode, ids, relu_from=None):
        self.bf16, self.mask_mode, self.ids, self.relu_from = bf16, mask_mode, ids, relu_from
        self.lin, self.att = [], []

    def linear(self, x, w, b):
        y = (_Bf16Linear.apply(x, w) if self.bf16 else x @ w.T) + b
        if self.relu_from is not None and len(self.lin) == self.relu_from[0]:
            y = follow_relu_signs(y, self.relu_from[1])
        self.lin.append((x, y))
        return y

    def attention(self, q, k, v, drop, site, causal=True):
        B, nh, L, _ = q.shape
        m = drop.mask(site, (B, nh, L, L), torch.float64) if drop.active() else torch.ones(B, nh, L, L, dtype=torch.float64)
        if self.mask_mode == 0:
            masked, fill = torch.ones(L, L, dtype=torch.bool).triu(1).expand(B, nh, L, L), float("-inf")
        else:
            masked, fill = (self.ids == 0).view(B, 1, 1, L).expand(B, nh, L, L), -1e9
        lse = []
        ctx = _Attention.apply(q, k, v, m, masked, fill, rb if self.bf16 else _ident, lse)
        ctx.retain_grad()
        self.att.append((q, k, v, ctx, lse[0]))
        return ctx


def attention_core(q, k, v, dctx, ids, B, L, H, nh, mask_mode, p, seed, step, base):
    """fp64 attention core on bf16-rounded q / k / v (rows [B*L, H]) with the Philox keep masks of dropout site 5, and its backward
    for the adjoint dctx: returns ctx, lse [B, nh, L], dq, dk, dv.  dctx enters unrounded (the flash kernels' own test compares
    their attention core with it at a bound that leaves room for that)."""
    from oracle.philox import keep_mask_attn
    hd = H // nh
    r = lambda t: t.to(torch.bfloat16).double().view(B, L, nh, hd).permute(0, 2, 1, 3)
    Q, K, V = r(q), r(k), r(v)
    dO = dctx.double().view(B, L, nh, hd).permute(0, 2, 1, 3)
    S = Q @ K.transpose(-1, -2)
    if mask_mode == 0:
        S = S.masked_fill(torch.ones(L, L, dtype=torch.bool).triu(1), float("-inf"))
    else:
        S = torch.where((ids == 0).view(B, 1, 1, L), torch.full_like(S, -1e9), S)
    lse = torch.logsumexp(S, -1)
    P = torch.exp(S - lse[..., None])
    if p > 0:
        keep = keep_mask_attn(B * nh * L, L, p, seed, step, 5, row_offset=base)
        m = torch.from_numpy(keep.astype(np.float64)).view(B, nh, L, L) / (1.0 - np.float32(p))
    else:
        m = torch.ones_like(P)
    ctx = (P * m) @ V
    Pb = torch.exp(S - lse.float().double()[..., None])
    dPd = dO @ V.transpose(-1, -2)
    delta = (dO * ctx).sum(-1, keepdim=True)
    dS = Pb * (dPd * m - delta)
    back = lambda t: t.permute(0, 2, 1, 3).reshape(B * L, H)
    return back(ctx), lse, back(dS @ K), back(dS.transpose(-1, -2) @ Q), back((Pb * m).transpose(-1, -2) @ dO)


# ---- whole blocks -----------------------------------------------------------------------------------------------------------------
ENC_PARAMS = ("ln1_w", "ln1_b", "in_w", "in_b", "out_w", "out_b", "ln2_w", "ln2_b", "w1", "b1", "w2", "b2", "sp_w", "sp_b")
DEC_PARAMS = ("ln_w", "ln_b", "s_in_w", "s_in_b", "s_out_w", "s_out_b", "e_in_w", "e_in_b", "e_out_w", "e_out_b", "w1", "b1", "w2", "b2")
_ENC_SD = dict(zip(ENC_PARAMS, ("attention_layernorm.weight", "attention_layernorm.bias", "attention_layer.in_proj_weight",
                                "attention_layer.in_proj_bias", "attention_layer.out_proj.weight", "attention_layer.out_proj.bias",
                                "forward_layernorm.weight", "forward_layernorm.bias", "forward_layer.conv1.weight",
                                "forward_layer.conv1.bias", "forward_layer.conv2.weight", "forward_layer.conv2.bias", "sparse.weight",
                                "sparse.bias")))
_DEC_SD = dict(zip(DEC_PARAMS, ("layer_norm.weight", "layer_norm.bias", "slf_attn.in_proj_weight", "slf_attn.in_proj_bias",
                                "slf_attn.out_proj.weight", "slf_attn.out_proj.bias", "enc_attn.in_proj_weight", "enc_attn.in_proj_bias",
                                "enc_attn.out_proj.weight", "enc_attn.out_proj.bias", "pos_ffn.conv1.weight", "pos_ffn.conv1.bias",
                                "pos_ffn.conv2.weight", "pos_ffn.conv2.bias")))


def _leaf(t):
    return t.detach().double().clone().requires_grad_(True)


def _rows(t):
    """[B, nh, L, hd] -> [B*L, H]"""
    B, nh, L, hd = t.shape
    return t.permute(0, 2, 1, 3).reshape(B * L, nh * hd)


def enc_block(inp, bf16, encoder_layer=O.encoder_layer, kernel_h1=None, prod=Products):
    """encoder block forward + backward on block_harness.inputs(case)["enc"] -> {name: fp64 tensor} with the names of the C ABI: the
    saved activations, out, rec, the nll_acc contribution, dx, dctx and g_<param> (the gradient contributions).  kernel_h1: the
    kernel's saved h1, whose signs the reference follows at ReLU ties (follow_relu_signs)."""
    B, L, H, nh = inp["B"], inp["L"], inp["H"], inp["nh"]
    ids = inp["ids"].long()
    prm = {k: _leaf(inp[k]) for k in ENC_PARAMS}
    x = _leaf(inp["x"])
    pr = prod(bf16, inp["mask_mode"], ids, None if kernel_h1 is None else (4, kernel_h1))
    sd = {"e." + _ENC_SD[k]: v for k, v in prm.items()}
    keep = (ids != 0).unsqueeze(-1).double()
    sites = {"enc0_attn": inp["sites"][0], "enc0_ffn1": inp["sites"][1], "enc0_ffn2": inp["sites"][2]}
    out, rec, _ = encoder_layer(sd, "e.", x.view(B, L, H), keep, nh, inp["drop"], sites, 0, prod=pr)
    diag = torch.diagonal(rec, dim1=-2, dim2=-1).sum()
    J = (out.reshape(-1, H) * inp["dout"].double()).sum() - inp["nll_coef"] * diag
    if inp.get("drec") is not None:
        J = J + (rec.reshape(-1, nh, nh) * inp["drec"].double()).sum()
    J.backward()
    q, k, v, ctx, lse = pr.att[0]
    res = {"q": _rows(q), "k": _rows(k), "v": _rows(v), "ctx": _rows(ctx), "lse": lse,
           "y": (pr.lin[0][0] + pr.lin[3][1]).reshape(-1, H), "h1": pr.lin[4][1].reshape(-1, H), "out": out.reshape(-1, H),
           "rec": rec.reshape(-1, nh, nh), "nll_acc": -diag, "dctx": _rows(ctx.grad),
           "dx": x.grad + (inp["dx_extra"].double() if inp.get("dx_extra") is not None else 0.0)}
    res.update({"g_" + k: v.grad for k, v in prm.items()})
    return {k: v.detach() for k, v in res.items()}


def dec_block(inp, bf16, decoder_layer=O.decoder_layer, kernel_h1=None, prod=Products):
    """decoder block forward + backward on block_harness.inputs(case)["dec"] -> saved activations, out, the mse_acc contribution, dx,
    dfeats, denc, dctx, dctx2, g_<param>; kernel_h1 as in enc_block"""
    B, L, H, nh = inp["B"], inp["L"], inp["H"], inp["nh"]
    ids = inp["ids"].long()
    prm = {k: _leaf(inp[k]) for k in DEC_PARAMS}
    x, feats = _leaf(inp["x"]), _leaf(inp["feats"])
    enc_in = _leaf(inp["enc_in"]) if inp.get("enc_in") is not None else None
    pr = prod(bf16, inp["mask_mode"], ids, None if kernel_h1 is None else (8, kernel_h1))
    sd = {"d." + _DEC_SD[k]: v for k, v in prm.items()}
    keep = (ids != 0).unsqueeze(-1).double()
    s = inp["sites"]
    sites = {"dec0_self": s[0], "dec0_cross": s[1], "dec0_ffn1": s[2], "dec0_ffn2": s[3]}
    out = decoder_layer(sd, "d.", x.view(B, L, H), feats.view(B, L, H), keep, nh, inp["drop"], sites, 0, prod=pr).reshape(-1, H)
    J = (out * inp["dout"].double()).sum()
    mse = None
    if enc_in is not None:
        mse = ((enc_in - out) ** 2).sum()
        J = J + 0.5 * inp["mse_coef"] * mse
    J.backward()
    q1, k1, v1, ctx1, lse1 = pr.att[0]
    q2, k2, v2, ctx2, lse2 = pr.att[1]
    res = {"d": pr.lin[0][0].reshape(-1, H), "q1": _rows(q1), "k1": _rows(k1), "v1": _rows(v1), "ctx1": _rows(ctx1), "lse1": lse1,
           "a": pr.lin[3][1].reshape(-1, H), "q2": _rows(q2), "k2": _rows(k2), "v2": _rows(v2), "ctx2": _rows(ctx2), "lse2": lse2,
           "c": pr.lin[7][1].reshape(-1, H), "h1": pr.lin[8][1].reshape(-1, H), "out": out,
           "dx": x.grad, "dfeats": feats.grad, "dctx": _rows(ctx1.grad), "dctx2": _rows(ctx2.grad)}
    if enc_in is not None:
        res.update(mse_acc=mse, denc=enc_in.grad)
    res.update({"g_" + k: v.grad for k, v in prm.items()})
    return {k: v.detach() for k, v in res.items()}


def err(a, b):
    """(max |a - b| / max |b|, cosine) in fp64"""
    a, b = torch.as_tensor(a).double().ravel(), torch.as_tensor(b).double().ravel()
    den = b.abs().max().clamp_min(1e-30)
    return float((a - b).abs().max() / den), float(a @ b / (a.norm() * b.norm()).clamp_min(1e-30))
