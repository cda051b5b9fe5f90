"""Full-catalog top-K for Bert4Rec-ADT on the GPU: BertModel.full_sort_topk against the oracle's head (fixtures of the unmodified
reference), the per-item bias in both K7 kernels (exact fp32 and tcgen05 with the exact re-score), GraphedScorer on a BertModel
across a FlatOptimizer step, and item-sharded evaluation on two GPUs."""
import glob
import os
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMES = sorted(os.path.basename(p)[5:-4] for p in glob.glob(os.path.join(GOLDEN, "bert_*.npz")))


def _load(name):
    z = np.load(os.path.join(GOLDEN, f"bert_{name}.npz"))
    return {k: z[k] for k in z.files}


def _fixture_model(g, prefix="sd1/"):
    from adt_b200.bert4rec import BertModel
    B, L, H, nh, nl, I, inner = [int(v) for v in g["cfg"]]
    args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=L, num_layers=nl, hidden_units=H, dropout=float(g["p"]),
                                 attention_dropout=float(g["pa"]), inner_units=inner, type_vocab_size=2)
    m = BertModel(100, I, args)
    m.load_state_dict({k[len(prefix):]: torch.from_numpy(np.array(v)) for k, v in g.items() if k.startswith(prefix)})
    return m.cuda().eval()


def _seen_csr(seq, I):
    seen = [np.unique(r[(r >= 1) & (r <= I)]) for r in np.asarray(seq)]
    ip = np.concatenate([[0], np.cumsum([len(s) for s in seen])]).astype(np.int32)
    ix = np.concatenate(seen + [np.zeros(0)]).astype(np.int32)
    return seen, ip, ix


def _ref_topk(scores, K):
    """[U, I] scores of ids 1..I (-inf = excluded) -> ids [U, K] under (score desc, id asc), and the scores in that order."""
    U, I = scores.shape
    ids = np.stack([np.lexsort((np.arange(1, I + 1), -scores[u]))[:K] + 1 for u in range(U)])
    return ids, np.take_along_axis(scores, ids - 1, 1)


def _check_against(ids, sc, ref_scores, K, rel=1e-5):
    """ids identical to the reference top-K except where the reference's own scores tie within fp32 rounding; scores within `rel`."""
    ref_ids, ref_sorted = _ref_topk(ref_scores, K)
    tol = rel * np.abs(ref_sorted[np.isfinite(ref_sorted)]).max()
    mine = np.take_along_axis(ref_scores, ids - 1, 1)
    assert np.isfinite(mine).all()                                    # nothing seen, nothing outside 1..I
    assert np.all((ids == ref_ids) | (np.abs(mine - ref_sorted) <= tol))
    assert np.abs(sc - mine).max() <= tol
    assert all(len(set(r)) == K for r in ids)


@pytest.mark.parametrize("name", NAMES)
def test_full_sort_topk_exact_vs_oracle(name):
    from adt_b200.evaluate import CatalogScorer, hit_ndcg_mrr, metrics_from_acc
    from oracle import bert_oracle as BO
    from oracle.sasrec_oracle import Drop
    g = _load(name)
    B, L, H, nh, nl, I, inner = [int(v) for v in g["cfg"]]
    m = _fixture_model(g)
    seq = g["seq"]
    seen, ip, ix = _seen_csr(seq, I)
    K = min(10, I - max(len(s) for s in seen))
    ans = np.random.default_rng(1).integers(1, I + 1, size=B).astype(np.int32)
    acc = torch.zeros(6, dtype=torch.float64, device="cuda")
    sc, ids = m.full_sort_topk(seq, ip, ix, K=K, answers=ans, metric_acc=acc)
    scorer = m._scorers[(K, m.mask_bias.device)]
    assert not scorer._uses_tc(H, *scorer.bounds())                   # a fixture-sized catalog runs on the exact fp32 kernel
    sc, ids = sc.cpu().numpy(), ids.cpu().numpy()
    assert ids.min() >= 1 and ids.max() <= I
    # the oracle in eval mode: forward -> downstream at the last position -> ids 1..I -> mask seen
    sd = {k[4:]: torch.from_numpy(np.array(v)) for k, v in g.items() if k.startswith("sd1/")}
    cfg = BO.BCfg(I, L, H, nh, nl, inner)
    src = torch.from_numpy(seq).long()
    with torch.no_grad():
        out = BO.forward(sd, cfg, src, src, Drop(train=False), with_logits=False)
        logits = BO.downstream(sd, cfg, out["feats"][:, -1, :]).numpy()[:, 1:I + 1].astype(np.float64)
    for u, s in enumerate(seen):
        logits[u, s - 1] = -np.inf
    _check_against(ids, sc, logits, K)
    # fused metric sums == the host metrics of the returned lists
    got, exp = metrics_from_acc(acc), hit_ndcg_mrr(ans, ids)
    assert got["users"] == B
    for k_, v in exp.items():
        assert abs(got[k_] - v) < 1e-12, k_
    # what a user does today: predict over every item 1..I, mask, sort
    pos, sent = torch.arange(L).repeat(B, 1), torch.zeros(B, L, dtype=torch.long)
    pred = m.predict(None, torch.from_numpy(seq), pos, sent, torch.arange(1, I + 1).repeat(B, 1)).cpu().numpy().astype(np.float64)
    for u, s in enumerate(seen):
        pred[u, s - 1] = -np.inf
    _check_against(ids, sc, pred, K)
    # the same through a CatalogScorer built by the caller
    s2, i2 = CatalogScorer(m, K=K).topk(seq, ip, ix)
    assert np.array_equal(i2.cpu().numpy(), ids) and np.array_equal(s2.cpu().numpy(), sc)


# ---------------------------------------------------------------------------------------------------- tensor-core path with a bias
U_TC = 512


@pytest.fixture(scope="module", params=[(50_000, 64), (100_000, 64), (100_000, 256), (1_000_000, 64), (1_000_000, 256)],
                ids=lambda p: f"I{p[0]}_H{p[1]}")
def synth_catalog(request):
    I, H = request.param
    gen = torch.Generator(device="cuda").manual_seed(I + H)
    E = torch.randn(I, H, device="cuda", generator=gen) * (2.0 / (I + H)) ** 0.5 * 30
    feats = torch.randn(U_TC, H, device="cuda", generator=gen)
    rng = np.random.default_rng(H)
    seen = [np.unique(rng.integers(1, I + 1, size=30)) for _ in range(U_TC)]
    ip = torch.from_numpy(np.concatenate([[0], np.cumsum([len(s) for s in seen])]).astype(np.int32)).cuda()
    ix = torch.from_numpy(np.concatenate(seen).astype(np.int32)).cuda()
    ans = torch.from_numpy(rng.integers(1, I + 1, size=U_TC).astype(np.int32)).cuda()
    yield I, H, E, feats, ip, ix, ans
    del E
    torch.cuda.empty_cache()


def _holder(E, b, first_id=1):
    from adt_b200.evaluate import Catalog
    return types.SimpleNamespace(scoring_catalog=lambda: Catalog(E, b, first_id, E.shape[1]))


@pytest.mark.parametrize("case", ["zero", "realistic", "adversarial", "ties"])
def test_tc_bias_equals_exact(synth_catalog, case):
    from adt_b200.evaluate import CatalogScorer
    I, H, E, feats, ip, ix, ans = synth_catalog
    gen = torch.Generator(device="cuda").manual_seed(7)
    dot_std = float((feats[:64] @ E[:4096].t()).std())
    if case == "zero":
        b = torch.zeros(I, device="cuda")
    elif case == "realistic":
        b = torch.randn(I, device="cuda", generator=gen) * dot_std           # |b| ~ |<f, e>|
    elif case == "adversarial":
        b = torch.randn(I, device="cuda", generator=gen) * dot_std * 1e6     # fp32 rounding of the bias outweighs most dot products
    else:
        E = E.clone()
        E[1::2] = E[0::2][:I // 2]                                           # rows 2j, 2j+1 identical ...
        b = torch.randn(I, device="cuda", generator=gen) * dot_std
        b[1::2] = b[0::2][:I // 2]                                           # ... and so are their biases: exact ties
    K = 10
    acc_tc = torch.zeros(6, dtype=torch.float64, device="cuda")
    acc_ex = torch.zeros(6, dtype=torch.float64, device="cuda")
    tc = CatalogScorer(_holder(E, b), K=K)
    assert tc._uses_tc(H, *tc.bounds())
    s_tc, i_tc = [t.clone() for t in tc.topk_from_feats(feats, ip, ix, ans, acc_tc)]
    ex = CatalogScorer(_holder(E, b), K=K, use_tensor_cores=False)
    s_ex, i_ex = [t.clone() for t in ex.topk_from_feats(feats, ip, ix, ans, acc_ex)]
    flagged = tc.fallback_users
    print(f"I={I} H={H} case={case}: {flagged} of {U_TC} users re-run on the exact kernel")
    assert torch.equal(i_tc, i_ex) and torch.equal(s_tc, s_ex)
    assert torch.allclose(acc_tc, acc_ex, rtol=1e-12, atol=0)        # same terms, summed by atomics in another order
    assert int(i_tc.min()) >= 1 and int(i_tc.max()) <= I
    if case == "zero":     # a zero bias changes nothing: same lists as the unbiased tensor-core call
        s0, i0 = CatalogScorer(_holder(E, None), K=K).topk_from_feats(feats, ip, ix)
        assert torch.equal(i0, i_tc) and torch.equal(s0, s_tc)
    if case == "ties":     # equal pairs stay adjacent, lower id first
        ids = i_tc.cpu().numpy()
        sc = s_tc.cpu().numpy()
        same = sc[:, 1:] == sc[:, :-1]
        assert np.all(ids[:, 1:][same] > ids[:, :-1][same])


# ---------------------------------------------------------------------------------------------------- graph + optimizer step
def _small_bert(I, H=64, L=20, seed=0):
    from adt_b200.bert4rec import BertModel
    torch.manual_seed(seed)
    args = types.SimpleNamespace(device="cuda", num_heads=2, maxlen=L, num_layers=1, hidden_units=H, dropout=0.1, attention_dropout=0.1,
                                 inner_units=2 * H, type_vocab_size=2)
    m = BertModel(10, I, args)
    with torch.no_grad():
        m.mask_bias.normal_(0.0, 0.5)
    return m.cuda()


def _eval_batch(rng, I, U, L):
    seq = np.zeros((U, L), np.int32)
    for u in range(U):
        n = int(rng.integers(3, L))
        seq[u, L - n:] = rng.integers(1, I + 1, size=n)
    seq[:, -1] = I + 1                                                       # the mask token in the last position, as predict takes it
    seen, ip, ix = _seen_csr(seq, I)
    return seq, ip, ix, rng.integers(1, I + 1, size=U).astype(np.int32)


def test_graphed_scorer_bert_matches_eager_across_an_optimizer_step():
    from adt_b200.dp import FlatOptimizer
    from adt_b200.evaluate import CatalogScorer, GraphedScorer, metrics_from_acc
    I, L, U = 40_000, 20, 128
    m = _small_bert(I, L=L)
    opt = FlatOptimizer(m, lr=1e-2, clip=5.0)      # before the graph: the optimiser moves the parameters into its flat buffer
    m.eval()
    rng = np.random.default_rng(3)
    batches = [_eval_batch(rng, I, U, L) for _ in range(3)]
    max_seen = max(len(b[2]) for b in batches)
    gs = GraphedScorer(CatalogScorer(m, K=10), U, L, max_seen=max_seen)
    assert gs.tc                                    # 40k rows, H 64: the tensor-core path with the bias
    eager = CatalogScorer(m, K=10)

    def compare():
        acc = torch.zeros(6, dtype=torch.float64, device="cuda")
        out = []
        for seq, ip, ix, ans in batches:
            s_g, i_g = [t.clone() for t in gs.topk(seq, ip, ix, ans)]
            s_e, i_e = eager.topk(seq, ip, ix, ans, acc)
            assert torch.equal(i_g, i_e) and torch.equal(s_g, s_e)
            assert int(i_g.min()) >= 1 and int(i_g.max()) <= I
            out.append(i_g)
        got, exp = gs.metrics(), metrics_from_acc(acc)
        assert got["users"] == exp["users"] == U * len(batches)
        assert all(abs(got[k] - exp[k]) <= 1e-12 for k in exp)
        return out

    before = compare()
    # one cloze training step: the item table and mask_bias change through the optimiser's raw pointers
    m.train()
    B = 16
    dec = np.asarray([rng.integers(1, I + 1, size=L) for _ in range(B)], dtype=np.int64)
    msk = rng.random((B, L)) < 0.3
    msk[:, -1] = True
    src, lab = np.where(msk, I + 1, dec), np.where(msk, dec, 0)
    opt.zero_grad()
    m.fused_loss(src, dec, lab, [0.01], [0.001]).backward()
    b0 = m.mask_bias.detach().clone()
    opt.step()
    assert not torch.equal(b0, m.mask_bias.detach())
    m.eval()
    after = compare()
    assert any(not torch.equal(a, b) for a, b in zip(before, after))
    # an in-place edit of the bias alone is picked up too (the tc bound uses max|bias|)
    with torch.no_grad():
        m.mask_bias[1:I + 1] += 100.0 * torch.randn(I, device="cuda")
    compare()


# ---------------------------------------------------------------------------------------------------- two GPUs, item-sharded
def _shard_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from adt_b200.evaluate import CatalogScorer
        I, L, U = 70_000, 20, 256
        m = _small_bert(I, L=L).eval()
        seq, ip, ix, ans = _eval_batch(np.random.default_rng(5), I, U, L)
        res = []
        for tc in (True, False):
            acc_s = torch.zeros(6, dtype=torch.float64, device="cuda")
            acc_1 = torch.zeros(6, dtype=torch.float64, device="cuda")
            sh = CatalogScorer(m, K=10, shard=True, use_tensor_cores=tc)
            assert sh.sharded and (sh.bounds()[1] - sh.bounds()[0]) < I
            s_s, i_s = [t.clone() for t in sh.topk(seq, ip, ix, ans, acc_s)]
            one = CatalogScorer(m, K=10, shard=False, use_tensor_cores=False)
            s_1, i_1 = one.topk(seq, ip, ix, ans, acc_1)
            res += [torch.equal(i_s, i_1), torch.equal(s_s, s_1), torch.equal(acc_s, acc_1)]
        ret[rank] = tuple(res)
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_item_sharded_bert_matches_single_gpu():
    import torch.multiprocessing as mp
    world = 2
    ret = mp.Manager().dict()
    mp.spawn(_shard_worker, args=(world, 29700 + os.getpid() % 150, ret), nprocs=world, join=True)
    assert dict(ret) == {r: (True,) * 6 for r in range(world)}, dict(ret)
