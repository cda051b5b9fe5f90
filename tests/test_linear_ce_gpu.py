"""The fused vocabulary head + cross entropy (adt_linear_ce_fwd / _bwd, ops.linear_cross_entropy) on the B200:
(1) the op against fp64 on the same bf16-rounded operands, (2) BertModel.fused_loss on the fused head against the [R, V] logits path,
(3) against the oracle through the public entry, (4) the memory of a 1M-item head, (5) forward + backward replayed from a CUDA graph."""
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _bf16_round(t):
    return t.to(torch.bfloat16).float()


def _inputs(R, V, H, bias, seed):
    """x like a LayerNorm output, W scaled so that the scores spread to about +-80 (exercises the running max), labels at column 0 of a
    tile, at V - 1 (inside the ragged last tile) and at random columns."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(R, H, device="cuda", generator=g)
    W = torch.randn(V, H, device="cuda", generator=g) * (18.0 / H ** 0.5)
    b = torch.randn(V, device="cuda", generator=g) * 2.0 if bias else None
    lab = torch.randint(0, V, (R,), device="cuda", generator=g, dtype=torch.int32)
    special = [V - 1, 0, 128 * ((V // 3) // 128), V - 1 - (V - 1) % 128]
    for i, v in enumerate(special[:R]):
        lab[i] = v
    return x, W, b, lab


def _ref(x, W, b, lab):
    """fp64 on the bf16-rounded operands: (lse, loss, dx, dW, db) of the mean cross entropy"""
    X, Wd = _bf16_round(x).double(), _bf16_round(W).double()
    z = X @ Wd.T
    if b is not None:
        z += b.double()
    R = z.shape[0]
    lse = torch.logsumexp(z, 1)
    r = torch.arange(R, device=z.device)
    loss = (lse - z[r, lab.long()]).mean()
    P = torch.exp(z - lse[:, None])
    P[r, lab.long()] -= 1.0
    P /= R
    return lse, loss, P @ Wd, P.T @ X, P.sum(0)


def _run(x, W, b, lab, scratch_bytes=None):
    from adt_b200.ops import linear_cross_entropy
    h = x.clone().requires_grad_(True)
    Wp = W.clone().requires_grad_(True)
    bp = b.clone().requires_grad_(True) if b is not None else None
    loss = linear_cross_entropy(h, Wp, bp, lab, scratch_bytes)
    lse = loss.grad_fn.saved_tensors[4].clone()
    loss.backward()
    return lse, loss.detach(), h.grad, Wp.grad, bp.grad if bp is not None else None


def _close(a, ref, tol, cos=0.9999):
    a, ref = a.double().flatten(), ref.double().flatten()
    m = ref.abs().max().item()
    assert (a - ref).abs().max().item() <= tol * m, ((a - ref).abs().max().item(), m)
    c = (a @ ref / (a.norm() * ref.norm() + 1e-300)).item()
    assert c >= cos, c


@pytest.mark.parametrize("variant", ["nobias", "bias", "bias_3chunks"])
@pytest.mark.parametrize("H", [64, 128, 256])
@pytest.mark.parametrize("V", [1600, 26844, 70001])
@pytest.mark.parametrize("R", [1, 129, 4099])
def test_linear_ce_against_fp64(R, V, H, variant):
    """Tolerances:
    - lse within 1e-4 abs: the scores are exact bf16 products summed in fp32 over H <= 256 (16 MMA K-steps), an error of a few 2^-24
      |z| ~ 1e-5 at |z| ~ 80; the log-sum-exp adds the fp32 rounding of the running (max, sum exp) merges and of __expf.
    - loss within 1e-5 rel: the mean of lse - z[label] (both within ~1e-5 of fp64 at values of tens) summed in fp64.
    - g_bias within 1e-4 max|ref|: exp(z - lse) inherits the ~1e-5..1e-4 absolute error of z - lse as a relative error, and the fp32
      column sums add R rounding steps; the sums are taken before dS is rounded to bf16, so bf16 does not enter.
    - dx, dW within 1e-2 max|ref| and cosine >= 0.9999: both products read dS rounded to bf16 (relative error 2^-9 per element,
      accumulated in fp32), as the materialising path's dgrad / wgrad do."""
    from adt_b200 import ops
    bias = variant != "nobias"
    x, W, b, lab = _inputs(R, V, H, bias, seed=R * 7 + V + H)
    nbytes = None
    if variant == "bias_3chunks":          # a vocabulary chunk of about V / 3.3 columns: >= 3 chunks, the last one ragged
        from test_linear_ce_cpu import _layout_bytes
        target = 128 * max(1, int(V / 3.3) // 128)
        nbytes = _layout_bytes(R, target)       # exactly what one chunk of `target` columns needs
        vc, _ = ops.linear_ce_plan(R, V, H, nbytes)
        assert vc == target and -(-V // vc) >= 3 and V % vc != 0
        lab[min(4, R - 1)] = vc             # first column of the second chunk
    lse, loss, dx, dW, db = _run(x, W, b, lab, nbytes)
    rlse, rloss, rdx, rdW, rdb = _ref(x, W, b, lab)
    assert (lse.double() - rlse).abs().max().item() < 1e-4
    assert abs(loss.item() - rloss.item()) <= 1e-5 * abs(rloss.item())
    _close(dx, rdx, 1e-2)
    _close(dW, rdW, 1e-2)
    if bias:
        _close(db, rdb, 1e-4, cos=0.99999)


def _bert(itemnum, H=64, nh=2, L=64, dropout=0.1):
    from adt_b200.bert4rec import BertModel
    torch.manual_seed(0)
    args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=L, num_layers=1, hidden_units=H, dropout=dropout,
                                 attention_dropout=dropout, inner_units=4 * H, type_vocab_size=2)
    m = BertModel(10, itemnum, args)
    for prm in m.parameters():
        prm.data.normal_(0.0, 0.05) if prm.dim() >= 2 else prm.data.add_(0.1 * torch.randn(prm.shape))
    return m.cuda().train()


def _cloze(B, L, I, seed, mask_prob=0.3):
    rng = np.random.default_rng(seed)
    seq = np.zeros((B, L), np.int64); dec = seq.copy(); lab = seq.copy()
    for b in range(B):
        n = int(rng.integers(L // 2, L + 1))
        items = rng.integers(1, I + 1, size=n)
        msk = rng.random(n) < mask_prob
        msk[-1] = True
        dec[b, L - n:] = items
        seq[b, L - n:] = np.where(msk, I + 1, items)
        lab[b, L - n:] = np.where(msk, items, 0)
    return seq, dec, lab


def _loss_and_grads(m, batch):
    m.zero_grad(set_to_none=True)
    m.drop_seed, m.drop_step = 11, 3
    seq, dec, lab = batch
    loss = m.fused_loss(seq, dec, lab, [0.005], [0.0019])
    loss.backward()
    return float(loss), {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}


def test_fused_head_matches_the_materialising_path(monkeypatch):
    """same BertModel and batch (R >= 128, so the materialising head runs on adt_gemm_tc too) with fused_loss's vocabulary threshold
    moved below and above V: both compute the same bf16 products, so the loss agrees to 1e-5 and every gradient to 2e-3 max / cosine
    0.9999 (the two differ in the order of the exp sums and where dS rounds to bf16)."""
    from adt_b200 import bert4rec
    I = 3000
    m = _bert(I)
    m.precision = 1
    batch = _cloze(16, 64, I, seed=5)
    assert (batch[2] != 0).sum() >= 128
    calls = []
    real = bert4rec.linear_cross_entropy
    monkeypatch.setattr(bert4rec, "linear_cross_entropy", lambda *a, **k: calls.append(1) or real(*a, **k))
    monkeypatch.setattr(bert4rec, "FUSED_HEAD_MIN_VOCAB", 1 << 30)
    loss0, g0 = _loss_and_grads(m, batch)
    assert not calls
    monkeypatch.setattr(bert4rec, "FUSED_HEAD_MIN_VOCAB", 0)
    loss1, g1 = _loss_and_grads(m, batch)
    assert calls
    assert abs(loss1 - loss0) <= 1e-5 * abs(loss0)
    assert g0.keys() == g1.keys()
    for k in g0:
        a, r = g1[k].double().flatten(), g0[k].double().flatten()
        if r.norm() == 0:
            assert a.norm() == 0, k
            continue
        assert (a - r).abs().max() <= 2e-3 * r.abs().max(), k
        assert (a @ r / (a.norm() * r.norm())).item() >= 0.9999, k


def test_fused_head_vs_oracle_through_fused_loss():
    """test_bert_ml20m_like_shape_vs_oracle's setup with 65,536 items in the bf16 mode: fused_loss picks the fused head by itself
    (V = 65,636 >= FUSED_HEAD_MIN_VOCAB); loss within 2e-2 and every gradient's cosine > 0.98 against the fp32 oracle."""
    from adt_b200 import bert4rec
    from adt_b200.bert4rec import BertModel
    from oracle import bert_oracle as BO
    from oracle.sasrec_oracle import Drop
    B, L, H, nh, nl, I, inner, p, pa = 2, 200, 256, 4, 1, 65536, 1024, 0.5, 0.5
    assert I + 100 >= bert4rec.FUSED_HEAD_MIN_VOCAB
    torch.manual_seed(0)
    args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=L, num_layers=nl, hidden_units=H, dropout=p, attention_dropout=pa,
                                 inner_units=inner, type_vocab_size=2)
    m = BertModel(10, I, args)
    for prm in m.parameters():
        prm.data.normal_(0.01, 0.05) if prm.dim() >= 2 else prm.data.add_(0.1 * torch.randn(prm.shape))
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    rng = np.random.default_rng(4)
    seq = np.zeros((B, L), np.int64); dec = seq.copy(); lab = seq.copy()
    for b, n in enumerate([200, 61]):
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
    assert m._fused_head(int((lab != 0).sum()))
    loss = m.fused_loss(seq, dec, lab, l1, l2)
    assert abs(float(loss) - float(ref)) / abs(float(ref)) < 2e-2
    loss.backward()
    for k, prm in m.named_parameters():
        a, b = prm.grad.detach().cpu().numpy().ravel().astype(np.float64), sd[k].grad.numpy().ravel().astype(np.float64)
        if np.linalg.norm(b) > 1e-7:
            assert a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30) > 0.98, k


def test_one_million_item_head_memory_and_rows():
    """R 10,240, V 1,000,100, H 256: the peak memory of forward + backward rises by less than the bf16 copies + dW + dx + the declared
    scratch + 64 MB (< 5 % of one fp32 [R, V] tensor); 256 rows checked against fp64 (dx and lse depend on their own row only)."""
    from adt_b200 import ops
    R, V, H = 10240, 1000100, 256
    x, W, b, lab = _inputs(R, V, H, True, seed=1)
    h = x.clone().requires_grad_(True)
    Wp = W.clone().requires_grad_(True)
    bp = b.clone().requires_grad_(True)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    loss = ops.linear_cross_entropy(h, Wp, bp, lab)
    lse = loss.grad_fn.saved_tensors[4]
    loss.backward()
    torch.cuda.synchronize()
    rise = torch.cuda.max_memory_allocated() - base
    scratch = ops.linear_ce_scratch_bytes(R, V, H)
    bound = (R * H + V * H) * 2 + V * H * 4 + R * H * 4 + scratch + (64 << 20)
    assert bound < 0.05 * R * V * 4
    assert rise < bound, (rise, bound)
    sub = torch.randperm(R, generator=torch.Generator().manual_seed(0))[:256].cuda()
    X, Wd = _bf16_round(x[sub]).double(), _bf16_round(W).double()
    z = X @ Wd.T + b.double()
    rlse = torch.logsumexp(z, 1)
    assert (lse[sub].double() - rlse).abs().max().item() < 1e-4
    P = torch.exp(z - rlse[:, None])
    P[torch.arange(256, device="cuda"), lab[sub].long()] -= 1.0
    _close(h.grad[sub], (P / R) @ Wd, 1e-2)


def test_graph_replay_matches_eager():
    """forward + backward make no host synchronisation (the upstream gradient reaches the backward as a device scalar): captured in a
    CUDA graph, a replay gives the eager results (up to the order of the fp32 / fp64 atomics)."""
    from adt_b200.ops import linear_cross_entropy
    R, V, H = 777, 70001, 128
    x, W, b, lab = _inputs(R, V, H, True, seed=3)
    h, Wp, bp = (t.clone().requires_grad_(True) for t in (x, W, b))
    loss = linear_cross_entropy(h, Wp, bp, lab)
    eager = (loss.detach(),) + torch.autograd.grad(loss, (h, Wp, bp))
    del loss
    # the captured leaves are only ever used on the capture's side stream (a leaf first used on the legacy default stream would make
    # autograd synchronise with that stream inside the capture)
    h, Wp, bp = (t.clone().requires_grad_(True) for t in (x, W, b))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            loss = linear_cross_entropy(h, Wp, bp, lab)
            torch.autograd.grad(loss, (h, Wp, bp))
        del loss
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        gl = linear_cross_entropy(h, Wp, bp, lab)
        gout = (gl.detach(),) + torch.autograd.grad(gl, (h, Wp, bp))
    for t in gout:
        t.zero_()
    graph.replay()
    torch.cuda.synchronize()
    for a, e in zip(gout, eager):
        assert (a.double() - e.double()).abs().max().item() <= 1e-5 * e.double().abs().max().item() + 1e-12
