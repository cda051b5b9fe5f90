"""GPU: STOSA-ADT's Wasserstein attention on the tcgen05 flash kernels (adt_wattention_flash_fwd/bwd) against the fp64 oracle.

(a) the core, called through the C exports directly, at lengths around the resident kernels' limits (72, 133, 209), tile edges (257) and
    up to 2048; head sizes 16 / 32 / 64, nh 1 / 2 / 4; every key-id pattern (an all-padding sequence, no padding, a padding id inside,
    random left padding); dropout with a later rank's base and a device step counter; init-like (sigma 0.02) and wider inputs;
(b) agreement with the resident fp32 kernels where both serve, and bitwise reproducibility;
(c) WAttnFn's choice of path, a training step at L 512 against fp64 autograd, a CUDA-graphed step against the eager one, and evaluation.
Every oracle run is fp64 on the CPU on the same fp32 inputs the kernels see."""
import ctypes
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import stosa_catalog_ref as R
from oracle import stosa_oracle as SO
from oracle.bert_oracle import _Sites
from oracle.sasrec_oracle import Drop

pytestmark = pytest.mark.gpu

SEED, STEP, STEP_DEV = 1234, 7, 3      # dropout seed / host step / device step counter of the dropout cases


def _err(a, b):
    """max |a - b| / max |b|"""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _cos(a, b):
    a, b = a.detach().double().cpu().flatten(), b.detach().double().cpu().flatten()
    return float(F.cosine_similarity(a, b, dim=0))


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _key_ids(rng, B, L):
    """random left padding; sequence 0 is all padding, 1 has none, 2 has a padding id inside the sequence"""
    ids = np.zeros((B, L), np.int32)
    for b in range(B):
        n = (0, L, L)[b] if b < 3 else int(rng.integers(1, L + 1))
        ids[b, L - n:] = rng.integers(1, 1000, size=n)
    if L > 2:
        ids[2, L // 2] = 0
    return ids


def _inputs(rng, B, L, H, sigma, zero_cov=False):
    """six projected streams [B*L, H] as float32: means 0.01 + sigma N(0, 1), covariances elu(.) + 1 (1 % exactly 0 if zero_cov)"""
    M = B * L
    mean = lambda: 0.01 + sigma * rng.standard_normal((M, H))
    cov = lambda: F.elu(torch.from_numpy(mean())).numpy() + 1.0
    mq, cq, mk, ck, mv, cv = mean(), cov(), mean(), cov(), mean(), cov()
    for c in (cq, ck) if zero_cov else ():
        c[rng.random(c.shape) < 0.01] = 0.0
    return [x.astype(np.float32) for x in (mq, cq, mk, ck, mv, cv)]


def _drop(p, b0, nh, L, H, step_dev):
    from adt_b200.blocks import DropCfg
    return DropCfg(p, SEED, STEP, True, b0=b0, step_dev=step_dev).next("attn", nh, L, H)


def _flash(B, L, H, nh, p, b0, xs, ids, up):
    """the flash kernels through the C exports -> (mctx, cctx, row statistics, the six input gradients)"""
    from adt_b200 import _lib as Lb
    from adt_b200.ops import _st
    lib = Lb.lib()
    lib.adt_wattention_scratch_bytes.restype = ctypes.c_int64
    t = [_dev(x) for x in xs]
    kid = _dev(ids)
    step_dev = torch.full((1,), STEP_DEV, dtype=torch.int32, device="cuda")
    drop = _drop(p, b0, nh, L, H, step_dev)
    mctx, cctx = torch.empty_like(t[0]), torch.empty_like(t[0])
    stat = torch.empty(B, nh, L, 2, device="cuda")
    ws = torch.empty(lib.adt_wattention_scratch_bytes(B, L, H, nh, 1), dtype=torch.uint8, device="cuda")
    a = Lb.fill(Lb.adt_wattention_args(), mq=t[0], cq=t[1], mk=t[2], ck=t[3], mv=t[4], cv=t[5], mctx=mctx, cctx=cctx, lse=stat,
                key_ids=kid, B=B, L=L, H=H, nh=nh, drop=drop, tc_scratch=ws)
    Lb.check(lib.adt_wattention_flash_fwd(ctypes.byref(a), _st(mctx.device)), "adt_wattention_flash_fwd")
    g = [torch.empty_like(t[0]) for _ in range(6)]
    a = Lb.fill(Lb.adt_wattention_args(), mq=t[0], cq=t[1], mk=t[2], ck=t[3], mv=t[4], cv=t[5], lse=stat, key_ids=kid,
                dmctx=up[0], dcctx=up[1], dmq=g[0], dcq=g[1], dmk=g[2], dck=g[3], dmv=g[4], dcv=g[5], B=B, L=L, H=H, nh=nh, drop=drop,
                tc_scratch=ws, mctx_in=mctx, cctx_in=cctx)
    Lb.check(lib.adt_wattention_flash_bwd(ctypes.byref(a), _st(mctx.device)), "adt_wattention_flash_bwd")
    torch.cuda.synchronize()
    return mctx, cctx, stat, g


def _resident(B, L, H, nh, p, b0, xs, ids, up):
    from adt_b200.stosa import WAttnFn
    t = [_dev(x).requires_grad_(True) for x in xs]
    step_dev = torch.full((1,), STEP_DEV, dtype=torch.int32, device="cuda")
    mctx, cctx = WAttnFn.apply(*t, _dev(ids), (B, L, nh), _drop(p, b0, nh, L, H, step_dev))
    stat = mctx.grad_fn.saved_tensors[6]
    torch.autograd.backward([mctx, cctx], list(up))
    torch.cuda.synchronize()
    return mctx, cctx, stat, [x.grad for x in t]


def _upstream(B, L, H):
    g = torch.Generator(device="cuda").manual_seed(B * L + H)
    return [torch.randn(B * L, H, device="cuda", generator=g) for _ in range(2)]


def _oracle(B, L, H, nh, p, b0, xs, ids, up):
    """fp64 attention_core -> (mctx, cctx, scores [B, nh, L, L], the six gradients)"""
    hd = H // nh
    leaves = [torch.from_numpy(x).double().requires_grad_(True) for x in xs]
    heads = [x.view(B, L, nh, hd).permute(0, 2, 1, 3) for x in leaves]
    mask = SO.masks(torch.from_numpy(ids).long())
    mctx, cctx = SO.attention_core(*heads, mask, p, Drop(p, SEED, STEP + STEP_DEV, b0, train=True), _Sites())
    mctx, cctx = mctx.reshape(B * L, H), cctx.reshape(B * L, H)
    torch.autograd.backward([mctx, cctx], [u.double().cpu() for u in up])
    with torch.no_grad():
        s = SO.attention_scores(*heads[:4], mask)
    return mctx.detach(), cctx.detach(), s, [x.grad for x in leaves]


GRADS = ("dmq", "dcq", "dmk", "dck", "dmv", "dcv")


# Bounds: 2x the largest error measured on a B200 over every case below (contexts 2.4e-3, gradients 1.2e-2 of max, 1/sum 2.0e-3).
def _check(got, ref, ids, L, record, ctx_tol=5e-3, grad_tol=2.5e-2):
    mctx, cctx, stat, g = got
    rm, rc, s, rg = ref
    for name, a, b in (("mctx", mctx, rm), ("cctx", cctx, rc)):
        e, c = _err(a, b), _cos(a, b)
        record(name, e)
        assert e <= ctx_tol and c >= 0.9999, (name, e, c)
    for name, a, b in zip(GRADS, g, rg):
        e, c = _err(a, b), _cos(a, b)
        record(name, e)
        assert e <= grad_tol and c >= 0.999, (name, e, c)
    # row statistics: 1/sum to 3e-3 (it carries the absolute error of the stored max score, ~bf16 rounding of the score terms);
    # rows with no valid key (before the sequence's first valid key) bit for bit
    stat = stat.cpu()
    inv = 1.0 / torch.exp(s - s.max(-1, keepdim=True).values).sum(-1)
    e_inv = float(((stat[..., 1].double() - inv).abs() / inv).max())
    record("row_inv_sum", e_inv)
    assert e_inv <= 3e-3, e_inv
    first = np.array([np.flatnonzero(r > 0)[0] if (r > 0).any() else L for r in ids])
    none = torch.from_numpy(np.arange(L)[None, :] < first[:, None])[:, None, :].expand_as(stat[..., 0])
    assert none.any()
    assert (stat[..., 0][none] == -4294967296.0).all()
    assert (stat[..., 1][none] == np.float32(1.0) / np.float32(L)).all()


# (B, L, H, nh, attention dropout, data-parallel rank offset b0, some covariances exactly 0: the clamp branches)
CORE_CASES = [
    (4, 72, 64, 1, 0.0, 0, False),        # hd 64 at the resident backward's limit
    (4, 133, 64, 2, 0.5, 2, False),       # hd 32, one past its resident backward limit, L % 8 != 0
    (5, 209, 64, 4, 0.5, 0, False),       # hd 16, one past its resident backward limit
    (4, 257, 128, 2, 0.5, 2, True),       # hd 64, one row into a third tile
    (4, 512, 32, 2, 0.0, 0, False),       # hd 16, nh 2
    (4, 1024, 64, 1, 0.5, 0, False),      # hd 64, nh 1
    (4, 2048, 32, 1, 0.5, 2, False),      # hd 32, the longest sequence
]


@pytest.mark.parametrize("sigma", [0.02, 0.3])
@pytest.mark.parametrize("case", CORE_CASES, ids=lambda c: "B%d_L%d_H%d_nh%d_p%g_b0%d" % c[:6] + ("_zc" if c[6] else ""))
def test_wflash_vs_fp64(case, sigma, record_property):
    B, L, H, nh, p, b0, zero_cov = case
    rng = np.random.default_rng([B, L, H, nh, int(sigma * 100)])
    xs = _inputs(rng, B, L, H, sigma, zero_cov)
    ids = _key_ids(rng, B, L)
    up = _upstream(B, L, H)
    _check(_flash(B, L, H, nh, p, b0, xs, ids, up), _oracle(B, L, H, nh, p, b0, xs, ids, up), ids, L, record_property)


@pytest.mark.parametrize("case", [(4, 200, 64, 4), (4, 130, 64, 2)], ids=["L200_hd16", "L130_hd32"])
def test_wflash_agrees_with_resident(case, record_property):
    """where both paths serve, the flash kernels meet the fp64 bounds; the resident kernels' own error is recorded beside theirs"""
    B, L, H, nh = case
    rng = np.random.default_rng(list(case))
    xs = _inputs(rng, B, L, H, 0.02)
    ids = _key_ids(rng, B, L)
    up = _upstream(B, L, H)
    ref = _oracle(B, L, H, nh, 0.5, 2, xs, ids, up)
    _check(_flash(B, L, H, nh, 0.5, 2, xs, ids, up), ref, ids, L, record_property)
    res = _resident(B, L, H, nh, 0.5, 2, xs, ids, up)
    for name, a, b in zip(("mctx", "cctx") + GRADS, res[:2] + tuple(res[3]), ref[:2] + tuple(ref[3])):
        record_property("resident_" + name, _err(a, b))


def test_wflash_is_deterministic():
    B, L, H, nh = 4, 700, 64, 2
    rng = np.random.default_rng(5)
    xs = _inputs(rng, B, L, H, 0.3)
    ids = _key_ids(rng, B, L)
    up = _upstream(B, L, H)
    r1, r2 = _flash(B, L, H, nh, 0.5, 0, xs, ids, up), _flash(B, L, H, nh, 0.5, 0, xs, ids, up)
    for a, b in zip(r1[:3] + tuple(r1[3]), r2[:3] + tuple(r2[3])):
        assert torch.equal(a, b)


def test_wattnfn_selects_flash_beyond_the_resident_limit():
    """precision 1 runs the flash kernels only where the resident tile does not fit; precision 0 keeps the resident refusal"""
    from adt_b200._lib import AdtError
    from adt_b200.stosa import WAttnFn
    B, H, nh = 4, 128, 4
    for L, flash in ((100, False), (200, True)):        # hd 32: the backward tile fits up to L 132
        rng = np.random.default_rng(L)
        t = [_dev(x).requires_grad_(True) for x in _inputs(rng, B, L, H, 0.3)]
        ids = _dev(_key_ids(rng, B, L))
        mctx, cctx = WAttnFn.apply(*t, ids, (B, L, nh), _drop(0.0, 0, nh, L, H, None), 1)
        assert len(mctx.grad_fn.saved_tensors) == (9 if flash else 7)
        (mctx.sum() + cctx.sum()).backward()
        assert all(torch.isfinite(x.grad).all() for x in t)
    mctx, cctx = WAttnFn.apply(*t, ids, (B, 200, nh), _drop(0.0, 0, nh, 200, H, None))
    with pytest.raises(AdtError, match=r"\(L, H/nh\) tile does not fit shared memory"):
        (mctx.sum() + cctx.sum()).backward()


# ---- (c) the model at L 512 -----------------------------------------------------------------------------------------------------
def _batch(rng, B, L, I):
    """left-padded batch with random lengths; sequence 0 is full length, 1 has one item, 2 is all padding"""
    seq, pos, neg = (np.zeros((B, L), np.int64) for _ in range(3))
    for b in range(B):
        n = (L, 1, 0)[b] if b < 3 else int(rng.integers(1, L + 1))
        it = rng.integers(1, I + 1, size=n + 1)
        seq[b, L - n:], pos[b, L - n:], neg[b, L - n:] = it[:-1], it[1:], rng.integers(1, I + 1, size=n)
    dec = np.zeros_like(seq)
    dec[:, 1:] = seq[:, :-1]
    return seq, dec, pos, neg


def _model(I, B, L, H, nh, p, sd=None):
    from adt_b200.stosa import DisenDistSAModel
    args = types.SimpleNamespace(item_size=I + 2, num_users=B, maxlen=L, hidden_units=H, num_heads=nh, num_layers=1, dropout=p,
                                 attention_dropout=p, initializer_range=0.02, pvn_weight=0.005)
    m = DisenDistSAModel(args)
    if sd is not None:
        m.load_state_dict(sd)
    m = m.cuda()
    m.precision = 1
    return m, args


@pytest.mark.parametrize("H,nh", [(64, 2), (128, 2)])
def test_stosa_step_l512_vs_fp64(H, nh, record_property):
    B, L, I, p = 16, 512, 3000, 0.3
    rng = np.random.default_rng([H, nh])
    seq, dec, pos, neg = _batch(rng, B, L, I)
    l1, l2 = [0.0021], [0.0009]
    cfg = SO.SCfg(I + 2, B, L, H, nh, 1, p, p)
    sd = SO.init_state(cfg, seed=H + nh)
    m, _ = _model(I, B, L, H, nh, p, sd)
    m.train()
    m.drop_seed, m.drop_step = SEED, STEP
    loss = m.fused_loss(seq, dec, pos, neg, l1, l2)[0]
    loss.backward()
    torch.cuda.synchronize()
    r = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    ids = [torch.from_numpy(x) for x in (seq, dec, pos, neg)]
    out = SO.forward(r, cfg, ids[0], ids[1], Drop(p, SEED, STEP, train=True))
    rtotal = SO.loss(r, cfg, out, ids[2], ids[3], l1, l2)[0]
    rtotal.backward()
    e = abs(float(loss) - float(rtotal)) / abs(float(rtotal))
    record_property("loss", e)
    assert e <= 2e-2, e
    # parameters whose gradient carries signal: norm at least 1e-3 of the largest (a covariance-query bias sums dcq over all B L rows,
    # where sum_j dS_ij = 0 cancels it far below the other gradients, so its direction is set by rounding, in fp32 as in bf16)
    grads = {k: r[k].grad for k, _ in m.named_parameters() if r[k].grad is not None and float(r[k].grad.abs().max()) > 0.0}
    top = max(float(g.norm()) for g in grads.values())
    worst = (1.0, "")
    for k, prm in m.named_parameters():
        if k in grads and float(grads[k].norm()) >= 1e-3 * top:
            worst = min(worst, (_cos(prm.grad, grads[k]), k))
    record_property("worst_param_grad_cos", worst[0])
    record_property("worst_param", worst[1])
    assert worst[0] >= 0.98, worst


def test_stosa_graphed_step_l512_matches_eager():
    from adt_b200.dp import FlatOptimizer, GraphedStep
    B, L, H, nh, I = 8, 512, 64, 2, 2000
    rng = np.random.default_rng(11)
    batch = _batch(rng, B, L, I)
    l1, l2 = [0.01], [0.001]
    torch.manual_seed(0)
    m0, _ = _model(I, B, L, H, nh, 0.3)
    sd = {k: v.clone() for k, v in m0.state_dict().items()}
    m0.train()
    o0 = FlatOptimizer(m0, lr=1e-3)
    losses0 = []
    for _ in range(3):
        o0.zero_grad()
        loss = m0.fused_loss(*batch, l1, l2)[0]
        loss.backward()
        o0.step()
        losses0.append(float(loss))
    m1, _ = _model(I, B, L, H, nh, 0.3)
    m1.load_state_dict(sd)
    m1.train()
    o1 = FlatOptimizer(m1, lr=1e-3)
    gs = GraphedStep(m1, o1, lambda s, d, p, n: m1.fused_loss(s, d, p, n, l1, l2)[0])
    losses1 = [float(gs.step(*batch)) for _ in range(3)]
    assert np.allclose(losses0, losses1, rtol=2e-5), (losses0, losses1)
    # Adam moves a parameter by up to lr per step whatever the gradient's size, so gradients near zero that differ in their last bits
    # (the tcgen05 linear layers' reduction order) may move a few parameters apart by up to 2 lr per step
    d = (o0.pflat - o1.pflat).abs()
    assert float(d.max()) <= 3 * 2e-3 and float((d > 2e-5 + 1e-3 * o0.pflat.abs()).float().mean()) <= 1e-3


def test_stosa_eval_l512():
    """full_sort_topk and a GraphedScorer batch at L 512 give the same ids; the encoder's last-position (mean, cov) is within bf16
    tolerance of the fp64 oracle"""
    from adt_b200.evaluate import CatalogScorer, GraphedScorer
    U, L, H, nh, I, K = 32, 512, 64, 2, 2000, 10
    cfg = SO.SCfg(I + 2, U, L, H, nh, 1)
    sd = SO.init_state(cfg, seed=3)
    m, _ = _model(I, U, L, H, nh, 0.0, sd)
    m.eval()
    rng = np.random.default_rng(3)
    seq = np.zeros((U, L), np.int32)
    for u in range(U):
        n = int(rng.integers(3, L + 1))
        seq[u, L - n:] = rng.integers(1, I + 1, size=n)
    _, ip, ix = R.seen_sets(seq)
    ids = m.full_sort_topk(seq, ip, ix, K=K)
    gs = GraphedScorer(CatalogScorer(m, K=K), U, L, max_seen=len(ix))
    ids_g = gs.topk(seq, ip, ix)[1]
    assert torch.equal(ids, ids_g)
    mean, cov = m._last_states(seq)
    r = {k: v.double() for k, v in sd.items()}
    out = SO.forward(r, cfg, torch.from_numpy(seq).long(), torch.zeros(U, L, dtype=torch.long), Drop(0.0, 0, 0, train=False))
    em, ec = _err(mean, out["mean"][:, -1]), _err(cov, out["cov"][:, -1])
    assert em <= 2e-2 and ec <= 2e-2 and _cos(mean, out["mean"][:, -1]) >= 0.9999, (em, ec)
