"""Sequences longer than 256 positions: the fused tcgen05 flash attention (flash_tc.cu) through the C ABI and the models.

The attention core is compared with an fp64 restatement on the same bf16-rounded q / k / v and the same Philox keep masks
(oracle.philox.keep_mask_attn), in both mask modes, with padding at the left, inside and everywhere, with and without dropout.  The
backward restatement takes P = exp(s - lse) with the fp32 lse, as both tensor-core paths define it (a fully padded row of mask
mode 1 has lse = -1e9 + log L, which fp32 rounds to -1e9)."""
import ctypes
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _st(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _scratch(B, L, H, nh, backward, flash):
    """scratch of adt_attention_fwd / _bwd, or of the flash entry at any L (sized as for 257 positions when L is shorter)"""
    from adt_b200 import _lib as L_
    f = L_.lib().adt_attention_scratch_bytes
    f.restype = ctypes.c_int64
    n = int(f(B, max(L, 257) if flash else L, H, nh, backward))
    return torch.empty(n, dtype=torch.uint8, device="cuda")


def _inputs(B, L, H, nh, mask_mode, pad, seed):
    g = torch.Generator().manual_seed(seed)
    q = (torch.randn(B * L, H, generator=g) / (H // nh) ** 0.25).float()
    k = (torch.randn(B * L, H, generator=g) / (H // nh) ** 0.25).float()
    v = torch.randn(B * L, H, generator=g).float()
    dctx = torch.randn(B * L, H, generator=g).float()
    ids = torch.ones(B, L, dtype=torch.int32)
    rng = np.random.default_rng(seed)
    for b in range(B):
        kind = pad[b % len(pad)]
        if kind == "left":
            ids[b, : int(rng.integers(1, L))] = 0
        elif kind == "inside":
            ids[b, torch.from_numpy(rng.random(L) < 0.3)] = 0
        elif kind == "all":
            ids[b] = 0
    return q, k, v, dctx, ids


def _drop(p, seed, step, base, step_dev=None):
    from adt_b200 import _lib as L_
    d = L_.adt_dropout()
    d.enabled, d.p, d.seed, d.step, d.site, d.base = int(p > 0), float(p), seed, step, 5, base
    d.step_dev = step_dev.data_ptr() if step_dev is not None else None
    return d


def _run(fwd, bwd, q, k, v, dctx, ids, B, L, H, nh, mask_mode, drop, precision=1):
    """one fwd + bwd through the C ABI; returns ctx, lse, dq, dk, dv on the host"""
    from adt_b200 import _lib as L_
    lib = L_.lib()
    dev = torch.device("cuda")
    q, k, v, dctx, ids = (t.to(dev).contiguous() for t in (q, k, v, dctx, ids))
    ctx = torch.empty_like(q)
    lse = torch.empty(B, nh, L, device=dev)
    dq, dk, dv = torch.empty_like(q), torch.empty_like(q), torch.empty_like(q)
    a = L_.fill(L_.adt_attention_args(), q=q, k=k, v=v, ctx=ctx, lse=lse, key_ids=ids if mask_mode == 1 else None, B=B, L=L, H=H, nh=nh,
                mask_mode=mask_mode, training=1, drop=drop, precision=precision, tc_scratch=_scratch(B, L, H, nh, 0, 'flash' in fwd))
    L_.check(getattr(lib, fwd)(ctypes.byref(a), _st(dev)), fwd)
    a = L_.fill(L_.adt_attention_args(), q=q, k=k, v=v, ctx=ctx, lse=lse, key_ids=ids if mask_mode == 1 else None, dctx=dctx, dq=dq, dk=dk,
                dv=dv, B=B, L=L, H=H, nh=nh, mask_mode=mask_mode, training=1, drop=drop, precision=precision,
                tc_scratch=_scratch(B, L, H, nh, 1, 'flash' in bwd))
    L_.check(getattr(lib, bwd)(ctypes.byref(a), _st(dev)), bwd)
    torch.cuda.synchronize()
    return tuple(t.cpu() for t in (ctx, lse, dq, dk, dv))


def _reference(q, k, v, dctx, ids, B, L, H, nh, mask_mode, p, seed, step, base):
    """fp64 attention core on bf16-rounded operands; the backward uses the fp32-rounded lse (see module docstring)"""
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


def _err(a, b):
    a, b = a.double().ravel(), b.double().ravel()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30)), float(a @ b / (a.norm() * b.norm()).clamp_min(1e-30))


CORE = [
    # L, hd, nh, mask_mode, padding kinds, dropout p
    (257, 64, 2, 0, ("none",), 0.0),
    (300, 16, 4, 1, ("left", "inside", "all", "none"), 0.5),
    (513, 32, 2, 1, ("inside", "left"), 0.0),
    (513, 128, 1, 0, ("none",), 0.5),
    (1000, 96, 2, 1, ("left", "all"), 0.5),
    (1000, 48, 1, 0, ("none",), 0.0),
    (2048, 64, 2, 0, ("none",), 0.5),
    (2048, 128, 1, 1, ("inside",), 0.0),
    (777, 80, 1, 1, ("none", "inside"), 0.5),
]


@pytest.mark.parametrize("L,hd,nh,mask_mode,pad,p", CORE)
def test_flash_core_against_fp64(L, hd, nh, mask_mode, pad, p):
    """adt_attention_fwd / _bwd at L > 256 (the flash kernels) against fp64: lse, ctx, dq, dk, dv; dropout with a non-zero data-parallel
    row offset and a device-side step counter"""
    B, H = 2, hd * nh
    q, k, v, dctx, ids = _inputs(B, L, H, nh, mask_mode, pad, seed=L + hd)
    base, step, sdev = 3 * nh * L, 11, 4
    step_dev = torch.tensor([sdev], dtype=torch.int32, device="cuda")
    got = _run("adt_attention_fwd", "adt_attention_bwd", q, k, v, dctx, ids, B, L, H, nh, mask_mode, _drop(p, 99, step, base, step_dev))
    ref = _reference(q, k, v, dctx, ids, B, L, H, nh, mask_mode, p, 99, step + sdev, base)
    assert float((got[1].double() - ref[1].float().double()).abs().max()) <= 1e-4     # fp32 lse: -1e9 + log L of a padded row is -1e9
    e, c = _err(got[0], ref[0])
    assert e <= 1e-2 and c >= 0.9999, (e, c)
    for name, a, b in zip(("dq", "dk", "dv"), got[2:], ref[2:]):
        e, c = _err(a, b)
        assert e <= 3e-2 and c >= 0.999, (name, e, c)


@pytest.mark.parametrize("L,mask_mode,p", [(65, 0, 0.0), (200, 1, 0.5), (256, 0, 0.5)])
def test_flash_no_worse_than_batched_path(L, mask_mode, p):
    """at L <= 256 the flash entry and the batched tcgen05 path run on identical inputs: against fp64, the flash error is at most
    twice the batched path's (plus a floor at fp32 rounding)"""
    B, H, nh = 3, 128, 2
    q, k, v, dctx, ids = _inputs(B, L, H, nh, mask_mode, ("left", "inside", "none"), seed=L)
    d = _drop(p, 5, 2, nh * L)
    ref = _reference(q, k, v, dctx, ids, B, L, H, nh, mask_mode, p, 5, 2, nh * L)
    fl = _run("adt_attention_flash_fwd", "adt_attention_flash_bwd", q, k, v, dctx, ids, B, L, H, nh, mask_mode, d)
    bt = _run("adt_attention_fwd", "adt_attention_bwd", q, k, v, dctx, ids, B, L, H, nh, mask_mode, d)
    for i, name in enumerate(("ctx", "lse", "dq", "dk", "dv")):
        ef = float((fl[i].double() - ref[i]).abs().max())
        eb = float((bt[i].double() - ref[i]).abs().max())
        assert ef <= 2 * eb + 1e-5, (name, ef, eb)


def test_flash_bitwise_reproducible():
    """two identical fwd + bwd calls give identical bits (plain stores, no atomics)"""
    B, L, H, nh = 2, 700, 128, 2
    q, k, v, dctx, ids = _inputs(B, L, H, nh, 1, ("inside",), seed=3)
    d = _drop(0.3, 8, 1, 0)
    r1 = _run("adt_attention_fwd", "adt_attention_bwd", q, k, v, dctx, ids, B, L, H, nh, 1, d)
    r2 = _run("adt_attention_fwd", "adt_attention_bwd", q, k, v, dctx, ids, B, L, H, nh, 1, d)
    for a, b in zip(r1, r2):
        assert torch.equal(a, b)


@pytest.mark.parametrize("H,nh,use_graph", [(64, 2, True), (256, 2, False)])
def test_sasrec_step_at_512_against_live_oracle(H, nh, use_graph):
    """a whole SASRec-ADT training step at maxlen 512 -- the H = 64 row-tile block kernels and the H = 256 tcgen05 block path, the
    attention of both in the flash kernels -- against the oracle evaluated live on the host (test_round2_gpu's check)"""
    from adt_b200 import synth
    from test_round2_gpu import _against_live_oracle
    cfg = dict(synth.CONFIGS["C2"], H=H, nh=nh, L=512, B=8, items=3000, geo=1.0 / 300, lo=100, add=6)
    _against_live_oracle(cfg, "bf16", use_graph)


def test_sasrec_eval_at_512_against_oracle():
    """final_feats and the full-catalog top-K at maxlen 512 against oracle.sasrec_oracle.encode / predict + full_sort_topk"""
    from adt_b200 import synth
    from adt_b200.evaluate import CatalogScorer
    from oracle import sasrec_oracle as O
    from test_round2_gpu import _c2_model
    cfg = dict(synth.CONFIGS["C2"], H=64, nh=2, L=512, B=8, items=3000, geo=1.0 / 300, lo=100, add=6)
    m = _c2_model(cfg).eval()
    m.engine.precision = 1          # beyond 256 positions only the bf16 mode runs (the fp32 cores are refused)
    seq = synth.make_batch(np.random.default_rng(5), cfg)[0]
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    ocfg = O.Cfg(cfg["items"], cfg["L"], cfg["H"], cfg["nh"], cfg["nl"], cfg["p"])
    with torch.no_grad():
        ref = O.encode(sd, ocfg, torch.from_numpy(seq).long(), O.Drop(train=False))[0][:, -1].double()
        got = m.final_feats(torch.from_numpy(seq).to('cuda', torch.int32)).detach().cpu().double().view(ref.shape)
    assert float((got - ref).abs().max() / ref.abs().max()) < 2e-2
    seen = [np.unique(r[r > 0]) for r in seq]
    ip = np.concatenate([[0], np.cumsum([len(x) for x in seen])]).astype(np.int32)
    ix = np.concatenate(seen).astype(np.int32)
    _, ids = CatalogScorer(m, K=10, use_tensor_cores=False).topk(seq, ip, ix)
    want = O.full_sort_topk(O.predict(sd, ocfg, torch.from_numpy(seq).long(), None, True).numpy(), seen, k=10)
    overlap = np.mean([len(set(a) & set(b)) / 10 for a, b in zip(ids.cpu().numpy(), want)])
    assert overlap > 0.9, overlap       # the same top-10 sets up to bf16-level near-ties


def test_bert_at_512_against_oracle():
    """Bert4Rec fused_loss + backward at maxlen 512 (H 256, nh 4: hd 64), one short and one full sequence, against the oracle"""
    from adt_b200.bert4rec import BertModel
    from oracle import bert_oracle as BO
    from oracle.sasrec_oracle import Drop
    B, L, H, nh, nl, I, inner, p, pa = 2, 512, 256, 4, 1, 1500, 1024, 0.5, 0.5
    torch.manual_seed(0)
    args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=L, num_layers=nl, hidden_units=H, dropout=p, attention_dropout=pa,
                                 inner_units=inner, type_vocab_size=2)
    m = BertModel(10, I, args)
    for prm in m.parameters():
        prm.data.normal_(0.01, 0.05) if prm.dim() >= 2 else prm.data.add_(0.1 * torch.randn(prm.shape))
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    rng = np.random.default_rng(4)
    seq = np.zeros((B, L), np.int64); dec = seq.copy(); lab = seq.copy()
    for b, n in enumerate([512, 61]):
        items = rng.integers(1, I + 1, size=n)
        msk = rng.random(n) < 0.2
        msk[-1] = True
        dec[b, L - n:] = items
        seq[b, L - n:] = np.where(msk, I + 1, items)
        lab[b, L - n:] = np.where(msk, items, 0)
    cfg = BO.BCfg(I, L, H, nh, nl, inner, p, pa)
    out = BO.forward(sd, cfg, torch.from_numpy(seq), torch.from_numpy(dec), Drop(0.5, 77, 5, train=True))
    l1, l2 = [0.005], [0.0019]
    ref = BO.loss(cfg, out, torch.from_numpy(lab), l1, l2)
    ref.backward()
    m = m.cuda().train()
    m.drop_seed, m.drop_step = 77, 5
    m.precision = 1
    loss = m.fused_loss(seq, dec, lab, l1, l2)
    assert abs(float(loss.detach()) - float(ref.detach())) / abs(float(ref.detach())) < 2e-2
    loss.backward()
    for k, prm in m.named_parameters():
        a, b = prm.grad.detach().cpu().numpy().ravel().astype(np.float64), sd[k].grad.numpy().ravel().astype(np.float64)
        if np.linalg.norm(b) > 1e-7:
            assert a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30) > 0.98, k


def test_stosa_beyond_256_still_refused():
    """STOSA-ADT's Wasserstein attention keeps its own shared-memory limit: L = 300 is refused as before"""
    from adt_b200 import _lib as L_
    from adt_b200.stosa import WAttnFn
    B, L, H, nh = 1, 300, 64, 1
    t = [torch.randn(B * L, H, device="cuda") for _ in range(6)]
    ids = torch.ones(B, L, dtype=torch.int32, device="cuda")
    with pytest.raises(L_.AdtError, match="does not fit shared memory"):
        WAttnFn.apply(*t, ids, (B, L, nh), _drop(0.0, 0, 0, 0))
