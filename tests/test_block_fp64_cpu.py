"""The fp64 block references of block_ref.py on the host.

The default product hook reproduces the pre-hook oracle formulas bit for bit; the BF16 hook's products and their adjoints are the
bf16-operand products; and the bounds of test_block_fp64_gpu.py reject realistic bugs of a block on every bf16 route: each perturbation
below moves some tensor by more than twice the loosest bf16 bound.  The independence-head adjoint left out of dctx does so while every
parameter gradient keeps a cosine above 0.99 with the right one, which the whole-step checks (cosine 0.99 per parameter) accept."""
import math

import pytest
import torch
import torch.nn.functional as F

import block_harness as BH
import block_ref as R
from oracle import sasrec_oracle as O
from test_block_fp64_gpu import BOUNDS, ROUTES


def _c2():
    return BH.inputs(ROUTES["h64_fused_c2"][0])


def _old_mha(q_in, kv_in, w_in, b_in, w_o, b_o, nh, drop, site):
    """mha as the oracle wrote it before the product hook"""
    B, L, H = q_in.shape
    hd = H // nh
    q = F.linear(q_in, w_in[:H], b_in[:H])
    k = F.linear(kv_in, w_in[H:2 * H], b_in[H:2 * H])
    v = F.linear(kv_in, w_in[2 * H:], b_in[2 * H:])
    q = q.view(B, L, nh, hd).transpose(1, 2) / math.sqrt(hd)
    k = k.view(B, L, nh, hd).transpose(1, 2)
    v = v.view(B, L, nh, hd).transpose(1, 2)
    s = q @ k.transpose(-1, -2) + torch.full((L, L), float("-inf"), dtype=q.dtype).triu(1)
    p = drop.apply(torch.softmax(s, dim=-1), site)
    ctx = (p @ v).transpose(1, 2).reshape(B, L, H)
    return F.linear(ctx, w_o, b_o), ctx


def _old_ffn(x, w1, b1, w2, b2, drop, s1, s2):
    h = torch.relu(drop.apply(F.linear(x, w1, b1), s1))
    return drop.apply(F.linear(h, w2, b2), s2) + x


def test_default_hook_is_the_oracle():
    """encoder and decoder layer through the default Products hook against the pre-hook formulas: identical bits in fp32"""
    inp = _c2()
    e, d = inp["enc"], inp["dec"]
    B, L, H, nh = e["B"], e["L"], e["H"], e["nh"]
    keep = (e["ids"] != 0).unsqueeze(-1).float()
    sd = {"e." + R._ENC_SD[k]: e[k] for k in R.ENC_PARAMS}
    x = e["x"].view(B, L, H)
    out, rec, ctx = O.encoder_layer(sd, "e.", x, keep, nh, e["drop"], {"enc0_attn": 0, "enc0_ffn1": 1, "enc0_ffn2": 2}, 0)
    Qn = O.layer_norm(x, e["ln1_w"], e["ln1_b"])
    mo, c0 = _old_mha(Qn, x, e["in_w"], e["in_b"], e["out_w"], e["out_b"], nh, e["drop"], 0)
    z = O.layer_norm(Qn + mo, e["ln2_w"], e["ln2_b"])
    assert torch.equal(ctx, c0)
    assert torch.equal(out, _old_ffn(z, e["w1"], e["b1"], e["w2"], e["b2"], e["drop"], 1, 2) * keep)
    sd = {"d." + R._DEC_SD[k]: d[k] for k in R.DEC_PARAMS}
    xd, feats = d["x"].view(B, L, H), d["feats"].view(B, L, H)
    sites = {"dec0_self": 3, "dec0_cross": 4, "dec0_ffn1": 5, "dec0_ffn2": 6}
    got = O.decoder_layer(sd, "d.", xd, feats, keep, nh, d["drop"], sites, 0)
    dn = O.layer_norm(xd, d["ln_w"], d["ln_b"])
    a, _ = _old_mha(dn, dn, d["s_in_w"], d["s_in_b"], d["s_out_w"], d["s_out_b"], nh, d["drop"], 3)
    c, _ = _old_mha(a, feats, d["e_in_w"], d["e_in_b"], d["e_out_w"], d["e_out_b"], nh, d["drop"], 4)
    assert torch.equal(got, (dn + _old_ffn(c, d["w1"], d["b1"], d["w2"], d["b2"], d["drop"], 5, 6)) * keep)


def test_bf16_hook_products_and_adjoints():
    """x W^T and its two adjoints on a tiny case against the hand-written bf16-operand formulas"""
    g = torch.Generator().manual_seed(0)
    x, w, dy = (torch.randn(*s, generator=g, dtype=torch.float64) for s in ((5, 8), (3, 8), (5, 3)))
    x.requires_grad_(True)
    w.requires_grad_(True)
    y = R._Bf16Linear.apply(x, w)
    y.backward(dy)
    rb = R.rb
    assert torch.equal(y, rb(x) @ rb(w).T)
    assert torch.equal(x.grad, rb(dy) @ rb(w))
    assert torch.equal(w.grad, rb(dy).T @ rb(x))
    assert not torch.equal(x.grad, dy @ w.detach())


class _PadKVNoGrad(R.Products):
    """no gradient through the keys and values of padded positions (causal attention does not mask them)"""

    def attention(self, q, k, v, drop, site, causal=True):
        pad = (self.ids == 0).view(k.shape[0], 1, -1, 1)
        return super().attention(q, torch.where(pad, k.detach(), k), torch.where(pad, v.detach(), v), drop, site, causal)


def _no_head_adjoint(sd, pre, x, keep, nh, drop, sites, l, prod):
    """the independence head's adjoint left out of dctx"""
    out, rec, ctx = O.encoder_layer(sd, pre, x, keep, nh, drop, sites, l, prod=prod)
    B, L, H = x.shape
    logits = F.linear(ctx.detach().view(B, L, nh, H // nh), sd[pre + "sparse.weight"], sd[pre + "sparse.bias"])
    return out, torch.log_softmax(logits, dim=3), ctx


# name -> (block, perturbation, whether every parameter gradient keeps a cosine above 0.99).  The head adjoint is checked at a
# realistic weight of the independence loss (nll_coef 0.03, no external drec), where it is a small part of dctx.
PERTURBATIONS = {
    "enc_pad_kv_no_grad": ("enc", dict(prod=_PadKVNoGrad), False),
    "dec_pad_kv_no_grad": ("dec", dict(prod=_PadKVNoGrad), False),
    "enc_no_head_adjoint": ("enc", dict(encoder_layer=_no_head_adjoint), True),
}


@pytest.mark.parametrize("name", list(PERTURBATIONS))
def test_perturbation_exceeds_every_bf16_bound(name):
    blk, kw, subtle = PERTURBATIONS[name]
    loosest = max(b for r, b in BOUNDS.items() if ROUTES[r][0].precision == 1)
    inp = dict(BH.inputs(BH.Case(7, 50, 64, 2, [0, 2, 1, 0, 3, 1, 4], b0=3, sdev=4))[blk])     # C2 shape, little padding
    if blk == "enc":
        inp.update(nll_coef=0.03, drec=None)
    fn = R.enc_block if blk == "enc" else R.dec_block
    ref, got = fn(inp, True), fn(inp, True, **kw)
    errs = {k: R.err(got[k], ref[k]) for k in ref if float(ref[k].abs().max()) > 0}
    worst = max(errs, key=lambda k: errs[k][0])
    assert errs[worst][0] > 2 * loosest, (name, worst, errs[worst])
    if subtle:
        gcos = {k: c for k, (_, c) in errs.items() if k.startswith("g_")}
        assert min(gcos.values()) > 0.99, (name, gcos)
