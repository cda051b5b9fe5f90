"""STOSA full-catalog ranking on the GPU through the shared catalog path: the centred rows, bias and mu of adt_wcatalog_build and the
user rows of adt_wcatalog_user against the fp64 restatement (tests/stosa_catalog_ref.py), full_sort_topk against the reference's
distance matrix with the fused metrics, the tcgen05 path equal to the exact kernel on synthetic tables up to 1M items at H 64 and 128,
GraphedScorer refreshing the derived catalog before every replay, the hidden-size limit, and item-sharded evaluation on two GPUs."""
import os
import types

import numpy as np
import pytest
import torch

import stosa_catalog_ref as R

pytestmark = pytest.mark.gpu


def _fixture_model(g, prefix="sd1/"):
    from adt_b200.stosa import DisenDistSAModel
    m = DisenDistSAModel(R.args_of(g))
    m.load_state_dict(R.state_dict(g, prefix))
    return m.cuda().eval()


@pytest.mark.parametrize("name", R.NAMES)
def test_built_catalog_and_user_rows_match_fp64(name):
    from adt_b200.evaluate import catalog_of
    from adt_b200.testing import rel_err
    g = R.load(name)
    m = _fixture_model(g)
    c = catalog_of(m)
    sd = R.state_dict(g)
    mu, e, b = R.catalog(sd["item_mean_embeddings.weight"], sd["item_cov_embeddings.weight"])
    mu_d, e_d, b_d = (t.cpu().numpy().astype(np.float64) for t in (m._wcat[0], c.table, c.bias))
    assert c.first_id == 0 and c.table.shape == e.shape and c.hidden == e.shape[1]
    for got, exp in ((mu_d, mu), (e_d, e), (b_d, b)):
        assert np.abs(got - exp).max() <= 1e-6 * np.abs(exp).max()
    # fixed-order reduction: rebuilding an unchanged table gives the same bits
    before = [t.clone() for t in m._wcat[:3]]
    m._build_catalog()
    assert all(torch.equal(x, y) for x, y in zip(before, m._wcat[:3]))
    # final_feats = the oracle's evaluation-mode last position mapped through the same mu
    um, uc = R.last_states(g, sd)
    f = m.final_feats(g["seq"])
    assert rel_err(f, R.feats(um, uc, mu_d)) < 5e-5


@pytest.mark.parametrize("name", R.NAMES)
def test_full_sort_topk_vs_reference_with_metrics(name):
    from adt_b200.evaluate import hit_ndcg_mrr, metrics_from_acc
    from oracle import stosa_oracle as O
    g = R.load(name)
    m = _fixture_model(g)
    B = g["seq"].shape[0]
    seen, ip, ix = R.seen_sets(g["seq"])
    dist = np.asarray(g["dist"], np.float64)
    K = 10
    ans = np.random.default_rng(2).integers(0, dist.shape[1], size=B).astype(np.int32)
    ans[: B // 2] = O.full_sort_topk(dist, seen, K)[: B // 2, 3]               # half the answers inside the lists
    acc = torch.zeros(6, dtype=torch.float64, device="cuda")
    ids = m.full_sort_topk(g["seq"], ip, ix, K=K, answers=ans, metric_acc=acc).cpu().numpy()
    R.assert_same_up_to_near_ties(ids, O.full_sort_topk(dist, seen, K), dist, 1e-4)
    for u, s in enumerate(seen):
        assert not set(ids[u]) & set(s)
    got, exp = metrics_from_acc(acc), hit_ndcg_mrr(ans, ids)
    assert got["users"] == B
    for k, v in exp.items():
        assert abs(got[k] - v) <= 1e-12, k


# ---------------------------------------------------------------------------------------------------- tensor-core path
U_TC, K_TC = 512, 40
SPREAD = {"init": 0.02, "spread": 0.3}      # std of both item tables (mean 0.01): the model's initialisation and a trained-like spread


def synthetic_model(I, H, std, seed=0, maxlen=8):
    from adt_b200.stosa import DisenDistSAModel
    args = types.SimpleNamespace(item_size=I, num_users=4, maxlen=maxlen, hidden_units=H, num_heads=2, num_layers=1, dropout=0.0,
                                 attention_dropout=0.0, initializer_range=0.02)
    torch.manual_seed(seed)
    m = DisenDistSAModel(args).cuda().eval()
    gen = torch.Generator(device="cuda").manual_seed(seed + I + H)
    with torch.no_grad():
        for t in (m.item_mean_embeddings.weight, m.item_cov_embeddings.weight):
            t.normal_(0.01, std, generator=gen)
    return m


def synthetic_users(H, U, seed=1):
    """last-position states shaped like the encoder's: mean = ELU(LayerNorm(.)) ~ O(1), cov = ELU + 1"""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    mean = torch.nn.functional.elu(torch.randn(U, H, device="cuda", generator=gen))
    cov = torch.nn.functional.elu(torch.randn(U, H, device="cuda", generator=gen)) + 1.0
    return mean, cov


@pytest.fixture(scope="module", params=[(I, H, d) for I in (50_000, 100_000, 1_000_000) for H in (64, 128) for d in SPREAD],
                ids=lambda p: f"I{p[0]}_H{p[1]}_{p[2]}")
def synth(request):
    I, H, d = request.param
    m = synthetic_model(I, H, SPREAD[d])
    mean, cov = synthetic_users(H, U_TC)
    rng = np.random.default_rng(H)
    seen = [np.unique(rng.integers(0, I, size=30)) for _ in range(U_TC)]
    ip = torch.from_numpy(np.concatenate([[0], np.cumsum([len(s) for s in seen])]).astype(np.int32)).cuda()
    ix = torch.from_numpy(np.concatenate(seen).astype(np.int32)).cuda()
    yield I, H, d, m, mean, cov, seen, ip, ix
    del m
    torch.cuda.empty_cache()


def test_tc_equals_exact_and_fp64(synth):
    from adt_b200.evaluate import CatalogScorer
    I, H, d, m, mean, cov, seen, ip, ix = synth
    feats = m.user_feats(mean, cov)
    tc = CatalogScorer(m, K=K_TC)
    assert tc._uses_tc(2 * H, *tc.bounds())
    s_tc, i_tc = [t.clone() for t in tc.topk_from_feats(feats, ip, ix)]
    ex = CatalogScorer(m, K=K_TC, use_tensor_cores=False)
    s_ex, i_ex = ex.topk_from_feats(feats, ip, ix)
    print(f"I={I} H={H} {d}: fallback_users {tc.fallback_users} of {U_TC}")
    assert torch.equal(i_tc, i_ex) and torch.equal(s_tc, s_ex)
    # fp64 distances of the same parameters: the lists are the nearest unseen items up to fp32 near-ties
    Em, Ec = (t.detach().double() for t in (m.item_mean_embeddings.weight, m.item_cov_embeddings.weight))
    y = torch.cat([Em, torch.sqrt(torch.clamp(torch.where(Ec > 0, Ec + 1, torch.exp(Ec)), min=R.CLAMP))], 1)
    x = torch.cat([mean.double(), torch.sqrt(torch.clamp(cov.double(), min=R.CLAMP))], 1)
    dist = (x * x).sum(1, keepdim=True) + (y * y).sum(1)[None, :] - 2.0 * x @ y.t()
    for u, s in enumerate(seen):
        dist[u, torch.from_numpy(s).cuda().long()] = float("inf")
    ref = torch.topk(dist, K_TC, dim=1, largest=False).values
    mine = torch.gather(dist, 1, i_tc.long())
    assert torch.isfinite(mine).all()
    # near-ties: the rounding bound of an fp32 dot product of length 2H plus the bias, (2H + 2) 2^-24 (|f| max|e| + max|b|)
    c = m.scoring_catalog()
    scale = feats.double().norm(dim=1) * float(c.table.double().norm(dim=1).max()) + float(c.bias.abs().max())
    assert bool(((torch.sort(mine, dim=1).values - ref).abs() <= (2 * H + 2) * 2.0 ** -24 * scale[:, None]).all())
    assert all(len(set(r)) == K_TC for r in i_tc.cpu().numpy())


# ---------------------------------------------------------------------------------------------------- graph replay
def _eval_batch(rng, I, U, L):
    seq = np.zeros((U, L), np.int32)
    for u in range(U):
        n = int(rng.integers(3, L))
        seq[u, L - n:] = rng.integers(1, I, size=n)
    seen, ip, ix = R.seen_sets(seq)
    return seq, ip, ix, rng.integers(0, I, size=U).astype(np.int32)


@pytest.mark.parametrize("I", [5_000, 40_000], ids=["exact", "tc"])
def test_graphed_scorer_matches_eager_across_step_and_table_edit(I):
    from adt_b200.dp import FlatOptimizer
    from adt_b200.evaluate import CatalogScorer, GraphedScorer, metrics_from_acc
    L, U, H = 20, 128, 64
    from adt_b200.stosa import DisenDistSAModel
    args = types.SimpleNamespace(item_size=I, num_users=16, maxlen=L, hidden_units=H, num_heads=2, num_layers=1, dropout=0.1,
                                 attention_dropout=0.1, initializer_range=0.02, pvn_weight=0.005)
    torch.manual_seed(0)
    m = DisenDistSAModel(args).cuda()
    opt = FlatOptimizer(m, lr=1e-2)                   # before the graph: the optimiser moves the parameters into its flat buffer
    m.eval()
    rng = np.random.default_rng(3)
    batches = [_eval_batch(rng, I, U, L) for _ in range(3)]
    gs = GraphedScorer(CatalogScorer(m, K=10), U, L, max_seen=max(len(b[2]) for b in batches))
    assert gs.tc == (I >= 32768)

    def compare():
        acc = torch.zeros(6, dtype=torch.float64, device="cuda")
        out = []
        for seq, ip, ix, ans in batches:
            i_g = gs.topk(seq, ip, ix, ans)[1].clone()
            i_e = m.full_sort_topk(seq, ip, ix, K=10, answers=ans, metric_acc=acc)
            assert torch.equal(i_g, i_e)
            out.append(i_g)
        got, exp = gs.metrics(), metrics_from_acc(acc)
        assert got["users"] == exp["users"] == U * len(batches)
        assert all(abs(got[k] - exp[k]) <= 1e-12 for k in exp)
        return out

    before = compare()
    m.train()
    B = 16
    seq = np.asarray([rng.integers(1, I, size=L) for _ in range(B)], dtype=np.int64)
    dec = np.zeros_like(seq)
    dec[:, 1:] = seq[:, :-1]
    pos = np.roll(seq, -1, axis=1)
    neg = rng.integers(1, I, size=(B, L))
    opt.zero_grad()
    m.fused_loss(seq, dec, pos, neg, [0.01], [0.001])[0].backward()
    c0 = m.item_cov_embeddings.weight.detach().clone()
    opt.step()                                         # raw-pointer write: only _adt_param_version announces it
    assert not torch.equal(c0, m.item_cov_embeddings.weight.detach())
    m.eval()
    after = compare()
    assert any(not torch.equal(a, b) for a, b in zip(before, after))
    with torch.no_grad():
        m.item_cov_embeddings.weight.add_(torch.randn_like(m.item_cov_embeddings.weight))     # in place: the tensor version moves
    edited = compare()
    assert any(not torch.equal(a, b) for a, b in zip(after, edited))


# ---------------------------------------------------------------------------------------------------- hidden-size limits
def test_h128_on_both_paths_and_h256_refused():
    from adt_b200._lib import AdtError
    from adt_b200.evaluate import CatalogScorer
    rng = np.random.default_rng(4)
    for I in (3_000, 40_000):                          # exact kernel, tensor cores
        m = synthetic_model(I, 128, 0.3, maxlen=12)
        seq, ip, ix, _ = _eval_batch(rng, I, 64, 12)
        tc = CatalogScorer(m, K=20)
        assert tc._uses_tc(256, *tc.bounds()) == (I >= 32768)
        i_tc = tc.topk(seq, ip, ix)[1].clone()
        i_ex = CatalogScorer(m, K=20, use_tensor_cores=False).topk(seq, ip, ix)[1]
        assert torch.equal(i_tc, i_ex)
        assert torch.equal(m.full_sort_topk(seq, ip, ix, K=20), i_tc)
    m = synthetic_model(1000, 256, 0.3, maxlen=12)
    with pytest.raises(AdtError, match="128"):
        m.full_sort_topk(_eval_batch(rng, 1000, 4, 12)[0], K=10)


# ---------------------------------------------------------------------------------------------------- two GPUs, item-sharded
def _shard_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from adt_b200.evaluate import CatalogScorer
        I, H = 70_000, 64
        m = synthetic_model(I, H, 0.3)
        feats = m.user_feats(*synthetic_users(H, 256))
        rng = np.random.default_rng(5)
        seen = [np.unique(rng.integers(0, I, size=20)) for _ in range(256)]
        ip = torch.from_numpy(np.concatenate([[0], np.cumsum([len(s) for s in seen])]).astype(np.int32)).cuda()
        ix = torch.from_numpy(np.concatenate(seen).astype(np.int32)).cuda()
        ans = torch.from_numpy(rng.integers(0, I, size=256).astype(np.int32)).cuda()
        res = []
        for tc in (True, False):
            acc_s = torch.zeros(6, dtype=torch.float64, device="cuda")
            acc_1 = torch.zeros(6, dtype=torch.float64, device="cuda")
            sh = CatalogScorer(m, K=10, shard=True, use_tensor_cores=tc)
            assert sh.sharded and (sh.bounds()[1] - sh.bounds()[0]) < I
            s_s, i_s = [t.clone() for t in sh.topk_from_feats(feats, ip, ix, ans, acc_s)]
            one = CatalogScorer(m, K=10, shard=False, use_tensor_cores=False)
            s_1, i_1 = one.topk_from_feats(feats, ip, ix, ans, acc_1)
            res += [torch.equal(i_s, i_1), torch.equal(s_s, s_1), torch.equal(acc_s, acc_1)]
        ret[rank] = tuple(res)
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_item_sharded_stosa_matches_single_gpu():
    import torch.multiprocessing as mp
    world = 2
    ret = mp.Manager().dict()
    mp.spawn(_shard_worker, args=(world, 29850 + os.getpid() % 100, ret), nprocs=world, join=True)
    assert dict(ret) == {r: (True,) * 6 for r in range(world)}, dict(ret)
