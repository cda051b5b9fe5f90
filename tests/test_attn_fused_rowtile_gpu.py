"""Attention fused into the H = 64 projection kernels (ADT_ATTN_FUSED=1, sequences of 33 .. 64 positions) against the separate
attention launches (ADT_ATTN_FUSED=0, separate process: the switch is read once per process), through the block C ABI.  The per-row
arithmetic is the same on both paths, so the forward outputs and the row-wise backward outputs (dx, dfeats, dctx, ...) must agree
bit for bit; the weight gradients are fp32 atomic sums over differently cut row tiles and agree to re-association.  At L <= 32 both
settings run the separate launches."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# (B, L, nh, mask_mode, dropout, left padding of each sequence, data-parallel batch offset)
_CASES = [
    (7, 50, 2, 0, 0.5, [0, 1, 20, 49, 50, 3, 0], 3),      # C2 shape, an empty sequence, non-zero DP offset
    (5, 64, 4, 1, 0.3, [0, 63, 10, 5, 0], 0),            # L = 64, four heads, key-padding mask
    (3, 33, 1, 0, 0.0, [0, 32, 7], 0),                   # L = 33, one head (forward fused, backward separate), no dropout
    (6, 63, 2, 1, 0.0, [1, 0, 62, 30, 8, 0], 11),         # odd L, key-padding mask, no dropout
    (4, 40, 4, 0, 0.5, [39, 0, 3, 12], 1),               # four heads with dropout
    (5, 32, 2, 0, 0.5, [0, 5, 31, 2, 0], 0),             # L = 32: not fused
    (3, 20, 4, 1, 0.3, [0, 19, 4], 2),                   # L = 20: not fused
]
_ROW_OUT = ("enc/q", "enc/k", "enc/v", "enc/ctx", "enc/lse", "enc/y", "enc/h1", "enc/out", "enc/rec", "enc/dx", "enc/dctx", "enc/dy",
            "dec/d", "dec/q1", "dec/k1", "dec/v1", "dec/ctx1", "dec/a", "dec/q2", "dec/k2", "dec/v2", "dec/ctx2", "dec/c", "dec/h1",
            "dec/out", "dec/lse1", "dec/lse2", "dec/dx", "dec/dfeats", "dec/dctx", "dec/dd", "dec/dctx2")


def _run_blocks(case):
    """encoder and decoder block, forward and backward, on seeded inputs -> {name: array}"""
    import torch
    from adt_b200 import _lib as L
    B, Lq, nh, mask_mode, p, pad, b0 = case
    H, M, dev = 64, case[0] * case[1], torch.device("cuda")
    g = torch.Generator(device="cpu").manual_seed(1000 + Lq * 10 + nh)
    rnd = lambda *s, sc=1.0: (sc * torch.randn(*s, generator=g)).to(dev)
    ids = torch.zeros(B, Lq, dtype=torch.int32)
    for b in range(B):
        ids[b, pad[b]:] = torch.randint(1, 100, (Lq - pad[b],), generator=g, dtype=torch.int32)
    ids = ids.to(dev)
    f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)
    site = [0]

    def drop(kind):
        d = L.adt_dropout()
        d.enabled, d.p, d.seed, d.step, d.site = int(p > 0), p, 77, 5, site[0]
        d.base = b0 * (nh * Lq if kind == "attn" else Lq * H)
        site[0] += 1
        return d

    def lin(n_out, n_in):
        return rnd(n_out, n_in, sc=n_in ** -0.5), rnd(n_out, sc=0.1)

    def ln():
        return 1.0 + rnd(H, sc=0.1), rnd(H, sc=0.1)

    keep = []                     # the C structs hold raw pointers: the tensors behind them must outlive the calls

    def mha():
        w, o = lin(3 * H, H), lin(H, H)
        keep.extend(w + o)
        return L.fill(L.adt_mha_w(), in_w=w[0], in_b=w[1], out_w=o[0], out_b=o[1])

    out, grads = {}, []

    def gmha():
        t = [f(3 * H, H), f(3 * H), f(H, H), f(H)]
        grads.extend(t)
        return L.fill(L.adt_mha_g(), in_w=t[0], in_b=t[1], out_w=t[2], out_b=t[3]), t

    def gffn():
        t = [f(H, H), f(H), f(H, H), f(H)]
        grads.extend(t)
        return L.fill(L.adt_ffn_g(), w1=t[0], b1=t[1], w2=t[2], b2=t[3]), t

    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    # ---- encoder block
    x = rnd(M, H)
    ln1, ln2, attn, c1, c2 = ln(), ln(), mha(), lin(H, H), lin(H, H)
    ffn = L.fill(L.adt_ffn_w(), w1=c1[0], b1=c1[1], w2=c2[0], b2=c2[1])
    spw, spb = rnd(nh, H // nh, sc=0.3), rnd(nh, sc=0.1)
    sv = {k: f(M, H) for k in ("q", "k", "v", "ctx", "y", "h1", "out")}
    sv["lse"], sv["rec"] = f(B, nh, Lq), f(M, nh, nh)
    da, d1, d2 = drop("attn"), drop("row"), drop("row")
    a = L.fill(L.adt_enc_block_fwd_args(), x=x, ids=ids, ln1_w=ln1[0], ln1_b=ln1[1], attn=attn, ln2_w=ln2[0], ln2_b=ln2[1], ffn=ffn,
               sparse_w=spw, sparse_b=spb, nll_acc=None, B=B, L=Lq, H=H, nh=nh, training=1, mask_mode=mask_mode, drop_attn=da,
               drop_ffn1=d1, drop_ffn2=d2, precision=1, tc_scratch=None, **sv)
    L.check(L.lib().adt_enc_block_fwd(ctypes.byref(a), stream), "adt_enc_block_fwd")
    sc = {k: f(M, H) for k in ("dq", "dk", "dv", "dctx", "dy", "dx")}
    gl1, gl2, gsp = [f(H), f(H)], [f(H), f(H)], [f(nh, H // nh), f(nh)]
    grads.extend(gl1 + gl2 + gsp)
    ga, _ = gmha()
    gf, _ = gffn()
    dout, dx_extra, drec = rnd(M, H), rnd(M, H), rnd(M, nh, nh, sc=0.1)
    a = L.fill(L.adt_enc_block_bwd_args(), x=x, ids=ids, ln1_w=ln1[0], ln1_b=ln1[1], attn=attn, ln2_w=ln2[0], ln2_b=ln2[1], ffn=ffn,
               sparse_w=spw, sparse_b=spb, q=sv["q"], k=sv["k"], v=sv["v"], ctx=sv["ctx"], lse=sv["lse"], y=sv["y"], h1=sv["h1"],
               dout=dout, dx_extra=dx_extra, drec=drec, nll_coef=0.3, wgrad_scratch=None,
               g_ln1_w=gl1[0], g_ln1_b=gl1[1], g_attn=ga, g_ln2_w=gl2[0], g_ln2_b=gl2[1], g_ffn=gf, g_sparse_w=gsp[0], g_sparse_b=gsp[1],
               B=B, L=Lq, H=H, nh=nh, mask_mode=mask_mode, drop_attn=da, drop_ffn1=d1, drop_ffn2=d2, precision=1, **sc)
    L.check(L.lib().adt_enc_block_bwd(ctypes.byref(a), stream), "adt_enc_block_bwd")
    out.update({"enc/" + k: v for k, v in sv.items()})
    out.update({"enc/" + k: sc[k] for k in ("dx", "dctx", "dy")})
    # ---- decoder block
    x, feats = rnd(M, H), rnd(M, H)
    lnd, slf, enc, c1, c2 = ln(), mha(), mha(), lin(H, H), lin(H, H)
    ffn = L.fill(L.adt_ffn_w(), w1=c1[0], b1=c1[1], w2=c2[0], b2=c2[1])
    keys = ("d", "q1", "k1", "v1", "ctx1", "a", "q2", "k2", "v2", "ctx2", "c", "h1", "out")
    sv = {k: f(M, H) for k in keys}
    sv["lse1"], sv["lse2"] = f(B, nh, Lq), f(B, nh, Lq)
    ds, de, d1, d2 = drop("attn"), drop("attn"), drop("row"), drop("row")
    a = L.fill(L.adt_dec_block_fwd_args(), x=x, feats=feats, ids=ids, ln_w=lnd[0], ln_b=lnd[1], slf=slf, enc=enc, ffn=ffn, enc_in=None,
               mse_acc=None, B=B, L=Lq, H=H, nh=nh, training=1, mask_mode=mask_mode, drop_slf=ds, drop_enc=de, drop_ffn1=d1,
               drop_ffn2=d2, precision=1, tc_scratch=None, **sv)
    L.check(L.lib().adt_dec_block_fwd(ctypes.byref(a), stream), "adt_dec_block_fwd")
    sc = {k: f(M, H) for k in ("dq", "dk", "dv", "dctx", "dd", "dq2", "dk2", "dv2", "dctx2", "dx", "dfeats")}
    gln = [f(H), f(H)]
    grads.extend(gln)
    gs, _ = gmha()
    ge, _ = gmha()
    gf, _ = gffn()
    dout = rnd(M, H)
    a = L.fill(L.adt_dec_block_bwd_args(), x=x, feats=feats, ids=ids, ln_w=lnd[0], ln_b=lnd[1], slf=slf, enc=enc, ffn=ffn, enc_in=None,
               mse_coef=0.0, dout=dout, denc=None, wgrad_scratch=None, g_ln_w=gln[0], g_ln_b=gln[1], g_slf=gs, g_enc=ge, g_ffn=gf,
               B=B, L=Lq, H=H, nh=nh, mask_mode=mask_mode, drop_slf=ds, drop_enc=de, drop_ffn1=d1, drop_ffn2=d2, precision=1,
               **{k: v for k, v in sv.items() if k != "out"}, out=sv["out"], **sc)
    L.check(L.lib().adt_dec_block_bwd(ctypes.byref(a), stream), "adt_dec_block_bwd")
    out.update({"dec/" + k: v for k, v in sv.items()})
    out.update({"dec/" + k: sc[k] for k in ("dx", "dfeats", "dctx", "dd", "dctx2")})
    out.update({f"grad/{i}": t for i, t in enumerate(grads)})
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def _kernel_names(case):
    from adt_b200 import _lib as L
    lib = L.lib()
    lib.adt_timing_enable(1)
    _run_blocks(case)
    buf, tot, cnt = ctypes.create_string_buffer(4096), (ctypes.c_float * 64)(), (ctypes.c_int * 64)()
    n = lib.adt_timing_collect(buf, 4096, tot, cnt, 64)
    lib.adt_timing_enable(0)
    return buf.value.decode().split("\n")[:n]


def _trainer_step():
    """one C2-shaped training step (B 64) captured in and replayed from a CUDA graph -> (loss, gradient norm)"""
    import types
    import torch
    from adt_b200 import synth
    from adt_b200.model import SASRecADT
    from adt_b200.trainer import FusedTrainer
    cfg = dict(synth.CONFIGS["C2"], B=64)
    torch.manual_seed(0)
    args = types.SimpleNamespace(device="cuda", num_heads=cfg["nh"], maxlen=cfg["L"], num_layers=cfg["nl"], hidden_units=cfg["H"], dropout=0.5)
    m = SASRecADT(1, cfg["items"], args)
    for _, prm in m.named_parameters():
        if prm.dim() >= 2:
            torch.nn.init.xavier_normal_(prm.data)
    m = m.cuda().train()
    tr = FusedTrainer(m, [0.0124, 0.122], [0.0001, 0.05], weight_decay=1e-4, seed=5, precision="bf16", use_graph=True)
    tr.step(*synth.make_batch(np.random.default_rng(3), cfg))
    return tr.loss(), tr.grad_norm()


if __name__ == "__main__":      # helper process: python <this file> <case | step> <out.npz>
    if sys.argv[1] == "step":
        loss, gnorm = _trainer_step()
        np.savez(sys.argv[2], loss=loss, gnorm=gnorm)
    else:
        c = _CASES[int(sys.argv[1])]
        res = _run_blocks(c)
        np.savez(sys.argv[2], names=np.array(_kernel_names(c)), **res)
    sys.exit(0)


def _both(arg, tmp_path):
    here = os.path.abspath(__file__)
    res = []
    for fused in ("1", "0"):
        f = str(tmp_path / f"fused{fused}.npz")
        e = dict(os.environ, ADT_ATTN_FUSED=fused)
        e["PYTHONPATH"] = os.path.dirname(os.path.dirname(here)) + os.pathsep + e.get("PYTHONPATH", "")
        subprocess.run([sys.executable, here, arg, f], check=True, env=e, timeout=600)
        res.append(np.load(f))
    return res


@pytest.mark.parametrize("case", range(len(_CASES)))
def test_fused_attention_matches_separate_launches(case, tmp_path):
    a, b = _both(str(case), tmp_path)
    L_, nh = _CASES[case][1], _CASES[case][2]
    names_a, names_b = set(a["names"].tolist()), set(b["names"].tolist())
    fused = L_ > 32
    assert ("pre_attn_fwd" in names_a) == fused and "pre_attn_fwd" not in names_b
    assert ("mid_attn_fwd" in names_a) == fused and "mid_attn_fwd" not in names_b
    assert ("attn_pre_bwd" in names_a) == (fused and nh in (2, 4)) and "attn_pre_bwd" not in names_b
    for k in _ROW_OUT:
        assert np.array_equal(a[k], b[k]), (k, float(np.abs(a[k] - b[k]).max()))
    for k in a.files:
        if k.startswith("grad/"):
            x, y = a[k], b[k]
            assert np.abs(x - y).max() <= 1e-5 * np.abs(y).max() + 1e-12, (k, float(np.abs(x - y).max()), float(np.abs(y).max()))


def test_fused_attention_graphed_trainer_step(tmp_path):
    a, b = _both("step", tmp_path)
    assert abs(float(a["loss"]) - float(b["loss"])) <= 1e-6 * abs(float(b["loss"]))
    assert abs(float(a["gnorm"]) - float(b["gnorm"])) <= 1e-6 * float(b["gnorm"])
