"""Hidden sizes 256 < H <= 512 on the GPU: whole SASRec-ADT training steps (fused trainer, eager and CUDA-graph replay) and the compat
forward / backward against the oracle evaluated live on the host, evaluation (final_feats, predict, sampled metrics), the tensor-core
catalog scorer on its K-blocked ring (H 320 .. 512, with and without a per-item bias, eager and graphed) against the exact kernel,
Bert4Rec-ADT's fused loss (materialising and fused head) and full_sort_topk against its oracle, and the supernet on the wide path."""
import types

import numpy as np
import pytest
import torch

from test_round2_gpu import _against_live_oracle, _c2_model

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ SASRec-ADT training step
@pytest.mark.parametrize("H,nh,Lq,B,use_graph", [
    (384, 3, 40, 8, False),      # M = 320 < 512: the tcgen05 block path at a row count the row-tile kernels used to take
    (384, 6, 200, 4, True),
    (384, 4, 200, 4, False),     # head size 96
    (384, 3, 512, 2, False),     # flash attention, hd 128
    (512, 4, 40, 8, True),       # M = 320, graph replay
    (512, 8, 200, 4, False),
    (512, 4, 512, 2, False),
    (512, 8, 512, 2, True),
])
def test_wide_training_step_against_live_oracle(H, nh, Lq, B, use_graph):
    """loss, gradient norm, bit-exact embedding gather and every parameter's gradient direction against the fp32 oracle"""
    from adt_b200 import synth
    cfg = dict(synth.CONFIGS["C2"], H=H, nh=nh, L=Lq, B=B, items=3000)
    if Lq > 64:
        cfg.update(geo=1.0 / 160, lo=16, add=15)
    _against_live_oracle(cfg, "bf16", use_graph)


def test_wide_compat_forward_backward_against_oracle_autograd():
    """the reference-style model(...) call at H 512: outputs and autograd gradients of the reference loss built on them"""
    from adt_b200 import synth
    from adt_b200.lambdas import get_lambdas
    from oracle import sasrec_oracle as O
    cfg = dict(synth.CONFIGS["C2"], H=512, nh=8, L=60, B=8, items=2000)
    m = _c2_model(cfg).train()
    m.engine.precision = 1
    m.engine.drop_seed, m.engine.drop_step = 99, 3
    sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    l1, l2 = get_lambdas(cfg["dataset"])
    seq, dec, pos, neg = synth.make_batch(np.random.default_rng(11), cfg)
    pl, nl_, enc_in, dec_out, rec = m(None, seq, dec, pos, neg)
    # the reference loss on host copies of the outputs (the copies are differentiable: autograd brings the gradients back to the model)
    host = lambda t: [x.cpu() for x in t] if isinstance(t, list) else t.cpu()
    out = {"pos_logits": pl, "neg_logits": nl_, "enc_inputs": enc_in, "dec_outputs": dec_out, "rec_ind": rec}
    out = {k: host(v) for k, v in out.items()}
    ocfg = O.Cfg(cfg["items"], cfg["L"], cfg["H"], cfg["nh"], cfg["nl"], cfg["p"])
    loss, _ = O.loss({"item_emb.weight": m.item_emb.weight.cpu()}, ocfg, out, torch.from_numpy(pos).long(), l1, l2, cfg["wd"])
    loss.backward()
    ref_out = O.forward(sd, ocfg, *(torch.from_numpy(a).long() for a in (seq, dec, pos, neg)), drop=O.Drop(cfg["p"], 99, 3))
    ref, _ = O.loss(sd, ocfg, ref_out, torch.from_numpy(pos).long(), l1, l2, cfg["wd"])
    ref.backward()
    assert abs(float(loss) - float(ref)) / abs(float(ref)) < 2e-2, (float(loss), float(ref))
    assert np.array_equal(enc_in[0].detach().cpu().numpy(), ref_out["enc_inputs"][0].detach().numpy())
    a, b = out["pos_logits"].detach().numpy().ravel(), ref_out["pos_logits"].detach().numpy().ravel()
    assert np.abs(a - b).max() <= 5e-2 * np.abs(b).max() + 1e-3
    for k, prm in m.named_parameters():
        if sd[k].grad is None:
            continue
        a, b = prm.grad.detach().cpu().numpy().ravel().astype(np.float64), sd[k].grad.numpy().ravel().astype(np.float64)
        if np.linalg.norm(b) > 1e-7:
            assert a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30) > 0.99, k


# ------------------------------------------------------------------------------------------------ SASRec-ADT evaluation
@pytest.mark.parametrize("H,nh,Lq,B", [(384, 6, 50, 64), (512, 8, 200, 16), (512, 4, 512, 4)])
def test_wide_evaluation_against_oracle(H, nh, Lq, B):
    """final_feats (the phase 1 / phase 2 last-position tail on the tcgen05 path), predict over candidates and the whole table, and
    the fused sampled metrics against the oracle's predict"""
    from adt_b200 import synth
    from adt_b200.evaluate import sampled_rank, sampled_metrics_from_acc
    from oracle import sasrec_oracle as O
    cfg = dict(synth.CONFIGS["C2"], H=H, nh=nh, L=Lq, B=B, items=4000, geo=1.0 / 40, lo=8, add=6)
    m = _c2_model(cfg).eval()
    m.engine.precision = 1
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    ocfg = O.Cfg(cfg["items"], cfg["L"], cfg["H"], cfg["nh"], cfg["nl"], cfg["p"])
    seq = synth.make_batch(np.random.default_rng(5), cfg)[0]
    with torch.no_grad():
        feats_ref, _, _, _ = O.encode(sd, ocfg, torch.from_numpy(seq).long(), O.Drop(train=False))
    f = m.final_feats(torch.from_numpy(seq).cuda()).cpu()
    r = feats_ref[:, -1, :]
    cos = torch.nn.functional.cosine_similarity(f.double(), r.double(), dim=1)
    assert float(cos.min()) > 0.999, float(cos.min())
    full = m.predict(None, seq, None, True).cpu()
    ref_full = O.predict(sd, ocfg, torch.from_numpy(seq).long(), full=True)
    assert (full - ref_full).abs().max() <= 2e-2 * ref_full.abs().max()
    # exact fp32 scoring on top of the features: full=True equals feats @ E^T in fp32
    assert torch.allclose(full, f @ sd["item_emb.weight"].t(), rtol=1e-4, atol=1e-4 * float(full.abs().max()))
    rng = np.random.default_rng(9)
    cand = np.stack([rng.permutation(cfg["items"])[:101] + 1 for _ in range(B)])
    pc = m.predict(None, seq, cand).cpu()
    assert torch.allclose(pc, torch.gather(full, 1, torch.from_numpy(cand)), rtol=1e-5, atol=1e-5 * float(full.abs().max()))
    acc = torch.zeros(7, dtype=torch.float64, device="cuda")
    rank, scores = sampled_rank(m, seq, cand, metric_acc=acc)
    ref_rank = (-scores.cpu()).argsort(dim=1).argsort(dim=1)[:, 0].numpy()
    assert np.array_equal(rank.cpu().numpy(), ref_rank)
    (ndcg, hr), auc, mrr = sampled_metrics_from_acc(acc)
    (o_ndcg, o_hr), o_auc, _ = O.rank_metrics(-scores.cpu())
    for k in (5, 10):
        assert abs(hr[k] - o_hr[k]) < 1e-12 and abs(ndcg[k] - o_ndcg[k]) < 1e-6
    assert abs(auc - o_auc) < 1e-12


# ------------------------------------------------------------------------------------------------ tensor-core catalog scorer
U_TC = 512


@pytest.fixture(scope="module", params=[(I, H) for H in (320, 384, 448, 512) for I in (100_000, 1_000_000)],
                ids=lambda p: f"I{p[0]}_H{p[1]}")
def wide_catalog(request):
    I, H = request.param
    gen = torch.Generator(device="cuda").manual_seed(I + H)
    E = torch.randn(I + 1, H, device="cuda", generator=gen) * (2.0 / (I + H)) ** 0.5 * 30
    feats = torch.randn(U_TC, H, device="cuda", generator=gen)
    rng = np.random.default_rng(H)
    seen = [np.unique(rng.integers(1, I + 1, size=int(rng.integers(0, 40)))) for _ in range(U_TC)]
    ip = np.concatenate([[0], np.cumsum([len(s) for s in seen])]).astype(np.int32)
    ix = np.concatenate(seen).astype(np.int32)
    ans = rng.integers(1, I + 1, size=U_TC).astype(np.int32)
    yield I, H, E, feats, seen, ip, ix, ans
    del E
    torch.cuda.empty_cache()


def _holder(E, b):
    from adt_b200.evaluate import Catalog
    return types.SimpleNamespace(scoring_catalog=lambda: Catalog(E[1:], b, 1, E.shape[1]))


@pytest.mark.parametrize("bias", [False, True])
def test_wide_tensor_core_scorer_equals_exact(wide_catalog, bias):
    """adt_score_topk_tc on the K-blocked ring (KB 5 .. 8): ids and scores equal to the exact fp32 kernel's (the re-score keeps the
    exact kernel's sequential fmaf order, flagged users are re-run on it), seen items excluded, fused HIT/NDCG/MRR equal to the
    oracle's metrics of the returned lists; with and without Bert4Rec's per-item bias"""
    from adt_b200.evaluate import CatalogScorer, metrics_from_acc
    from oracle import sasrec_oracle as O
    I, H, E, feats, seen, ip, ix, ans = wide_catalog
    b = None
    if bias:
        gen = torch.Generator(device="cuda").manual_seed(3)
        b = torch.randn(I, device="cuda", generator=gen) * float((feats[:64] @ E[1:4097].t()).std())
    for K in (10, 40):
        acc_tc = torch.zeros(6, dtype=torch.float64, device="cuda")
        acc_ex = torch.zeros(6, dtype=torch.float64, device="cuda")
        tc = CatalogScorer(_holder(E, b), K=K)
        assert tc._uses_tc(H, *tc.bounds())
        s_tc, i_tc = [t.clone() for t in tc.topk_from_feats(feats, ip, ix, ans, acc_tc)]
        ex = CatalogScorer(_holder(E, b), K=K, use_tensor_cores=False)
        s_ex, i_ex = [t.clone() for t in ex.topk_from_feats(feats, ip, ix, ans, acc_ex)]
        print(f"I={I} H={H} K={K} bias={bias}: {tc.fallback_users} of {U_TC} users re-run on the exact kernel")
        assert torch.equal(i_tc, i_ex) and torch.equal(s_tc, s_ex)
        ids = i_tc.cpu().numpy()
        for u in range(U_TC):
            assert not set(ids[u].tolist()) & set(seen[u].tolist())
        got, exp = metrics_from_acc(acc_tc), O.full_sort_metrics(ans.reshape(-1, 1), ids)
        assert got["users"] == U_TC
        for key in ("HIT@5", "NDCG@5", "HIT@10", "NDCG@10", "MRR"):
            assert abs(got[key] - exp[key]) < 1e-9, (key, got[key], exp[key])


def test_wide_graphed_scorer_equals_eager():
    """GraphedScorer of a SASRec-ADT model at H 512 (tensor-core scorer on 40k items) equals eager scoring, list for list"""
    from adt_b200 import synth
    from adt_b200.evaluate import CatalogScorer, GraphedScorer, metrics_from_acc
    I, Lq, U = 40_000, 50, 128
    cfg = dict(synth.CONFIGS["C2"], H=512, nh=8, L=Lq, B=U, items=I)
    m = _c2_model(cfg).eval()
    m.engine.precision = 1
    rng = np.random.default_rng(3)
    batches = []
    for _ in range(2):
        seq = synth.make_batch(rng, cfg)[0]
        seen = [np.unique(r[r > 0]) for r in seq]
        ip = np.concatenate([[0], np.cumsum([len(s) for s in seen])]).astype(np.int32)
        batches.append((seq, ip, np.concatenate(seen).astype(np.int32), rng.integers(1, I + 1, size=U).astype(np.int32)))
    gs = GraphedScorer(CatalogScorer(m, K=10), U, Lq, max_seen=max(len(b[2]) for b in batches))
    assert gs.tc
    eager = CatalogScorer(m, K=10)
    acc = torch.zeros(6, dtype=torch.float64, device="cuda")
    for seq, ip, ix, ans in batches:
        s_g, i_g = [t.clone() for t in gs.topk(seq, ip, ix, ans)]
        s_e, i_e = eager.topk(seq, ip, ix, ans, acc)
        assert torch.equal(i_g, i_e) and torch.equal(s_g, s_e)
    got, exp = gs.metrics(), metrics_from_acc(acc)
    assert got["users"] == exp["users"] == 2 * U
    assert all(abs(got[k] - exp[k]) <= 1e-12 for k in exp)


# ------------------------------------------------------------------------------------------------ Bert4Rec-ADT
def _bert_case(I):
    from adt_b200.bert4rec import BertModel
    from oracle import bert_oracle as BO
    B, L, H, nh, nl, inner, p, pa = 2, 200, 512, 8, 1, 2048, 0.5, 0.5
    torch.manual_seed(0)
    args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=L, num_layers=nl, hidden_units=H, dropout=p, attention_dropout=pa,
                                 inner_units=inner, type_vocab_size=2)
    m = BertModel(10, I, args)
    for prm in m.parameters():
        prm.data.normal_(0.01, 0.03) if prm.dim() >= 2 else prm.data.add_(0.1 * torch.randn(prm.shape))
    rng = np.random.default_rng(4)
    seq = np.zeros((B, L), np.int64); dec = seq.copy(); lab = seq.copy()
    for b, n in enumerate([200, 61]):
        items = rng.integers(1, I + 1, size=n)
        msk = rng.random(n) < 0.2
        msk[-1] = True
        dec[b, L - n:] = items
        seq[b, L - n:] = np.where(msk, I + 1, items)
        lab[b, L - n:] = np.where(msk, items, 0)
    return m, BO.BCfg(I, L, H, nh, nl, inner, p, pa), seq, dec, lab


@pytest.mark.parametrize("I,fused", [(1500, False), (65536, True)])
def test_wide_bert_fused_loss_against_oracle(I, fused):
    """fused_loss at H 512 (nh 8, inner 2048, L 200) in the bf16 mode with the materialising head and with the fused head (vocabulary
    >= 65,536): loss within 2e-2 and every gradient's cosine > 0.98 against the fp32 oracle"""
    from oracle import bert_oracle as BO
    from oracle.sasrec_oracle import Drop
    m, cfg, seq, dec, lab = _bert_case(I)
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    out = BO.forward(sd, cfg, torch.from_numpy(seq), torch.from_numpy(dec), Drop(0.5, 77, 5, train=True))
    l1, l2 = [0.005], [0.0019]
    ref = BO.loss(cfg, out, torch.from_numpy(lab), l1, l2)
    ref.backward()
    m = m.cuda().train()
    m.drop_seed, m.drop_step = 77, 5
    m.precision = 1
    assert m._fused_head(int((lab != 0).sum())) == fused
    loss = m.fused_loss(seq, dec, lab, l1, l2)
    assert abs(float(loss) - float(ref)) / abs(float(ref)) < 2e-2, (float(loss), float(ref))
    loss.backward()
    for k, prm in m.named_parameters():
        a, b = prm.grad.detach().cpu().numpy().ravel().astype(np.float64), sd[k].grad.numpy().ravel().astype(np.float64)
        if np.linalg.norm(b) > 1e-7:
            assert a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30) > 0.98, k


def test_wide_bert_full_sort_topk_against_oracle_head():
    """full_sort_topk at H 512 (50k items: the tensor-core scorer with the per-item bias) against the oracle's head on the same
    weights: ids equal up to rounding-level ties of the oracle's fp32 logits, seen items excluded, and equal to the exact kernel's"""
    from adt_b200.evaluate import CatalogScorer
    from oracle import bert_oracle as BO
    from oracle.sasrec_oracle import Drop
    I = 50_000
    m, cfg, seq, dec, lab = _bert_case(I)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.cuda().eval()
    m.precision = 1
    src = np.where(seq == I + 1, dec, seq)
    seen = [np.unique(r[r > 0]) for r in src]
    ip = np.concatenate([[0], np.cumsum([len(s) for s in seen])]).astype(np.int32)
    ix = np.concatenate(seen).astype(np.int32)
    K = 10
    sc, ids = m.full_sort_topk(src, ip, ix, K=K)
    assert m._scorers[(K, m.mask_bias.device)]._uses_tc(512, *m._scorers[(K, m.mask_bias.device)].bounds())
    s_ex, i_ex = CatalogScorer(m, K=K, use_tensor_cores=False).topk(src, ip, ix)
    assert torch.equal(ids, i_ex) and torch.equal(sc, s_ex)
    with torch.no_grad():
        t = torch.from_numpy(src).long()
        out = BO.forward(sd, cfg, t, t, Drop(train=False), with_logits=False)
        logits = BO.downstream(sd, cfg, out["feats"][:, -1, :]).numpy()[:, 1:I + 1].astype(np.float64)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    for u, s in enumerate(seen):
        logits[u, s - 1] = -np.inf
        assert not set(ids[u].tolist()) & set(s.tolist())
        ref = np.argsort(-logits[u], kind="stable")[:K] + 1
        scale = np.abs(logits[u][np.isfinite(logits[u])]).max()
        for r in range(K):     # the bf16 encoder moves scores by ~1e-2 relative: a swap is only allowed between near-equal logits
            if ids[u, r] != ref[r]:
                assert abs(logits[u, ids[u, r] - 1] - logits[u, ref[r] - 1]) <= 3e-2 * scale, (u, r)


# ------------------------------------------------------------------------------------------------ supernet
REC = [0, 0.0001, 0.0005, 0.001, 0.005, 0.01]
IND = [0, 0.0001, 0.0005, 0.001, 0.0015, 0.002]


def test_wide_supernet_forward_backward():
    """SuperSASRecModel at H 512 runs forward and backward through the tcgen05 block path (every block of every candidate)"""
    from adt_b200.supernet import SuperSASRecModel
    from adt_b200 import synth
    cfg = dict(synth.CONFIGS["C2"], H=512, nh=8, L=40, B=16, items=1000)
    torch.manual_seed(0)
    args = types.SimpleNamespace(device="cuda", num_heads=8, maxlen=40, num_layers=2, hidden_units=512, dropout=0.2)
    m = SuperSASRecModel(100, 1000, REC, IND, args).cuda().train()
    m.precision = 1
    seq, dec, pos, neg = synth.make_batch(np.random.default_rng(1), cfg)
    pl, nl_, enc_in, dec_out, rec = m(None, seq, dec, pos, neg)
    valid = torch.from_numpy(pos).cuda() != 0
    bce = torch.nn.functional.binary_cross_entropy_with_logits
    loss = bce(pl[valid], torch.ones_like(pl[valid])) + bce(nl_[valid], torch.zeros_like(nl_[valid]))
    for i in range(2):
        loss = loss + 0.01 * torch.nn.functional.mse_loss(enc_in[i], dec_out[i]) + 0.001 * rec[i].mean()
    assert torch.isfinite(loss)
    loss.backward()
    used = [(k, p) for k, p in m.named_parameters() if p.grad is not None]
    assert len(used) > 10
    for k, p in used:
        assert torch.isfinite(p.grad).all(), k
    assert sum(float(p.grad.abs().sum()) for _, p in used) > 0


def test_wide_population_evaluator_matches_serial_candidate_fitness():
    """test_supernet.py's protocol at H 512 in the bf16 mode: the population evaluator and the serial reference loop agree"""
    from adt_b200.supernet import SuperSASRecModel
    from adt_b200.evolution import PopulationEvaluator, candidate_fitness, set_choice_from_candidate
    from adt_b200.sampler import DeviceSampler
    rng = np.random.default_rng(2)
    usernum, itemnum, L, H, nh, nl = 300, 500, 20, 512, 8, 2
    train, valid, test = {}, {}, {}
    for u in range(1, usernum + 1):
        h = [int(x) for x in rng.integers(1, itemnum + 1, size=int(rng.integers(4, 30)))]
        train[u], valid[u], test[u] = h[:-2], [h[-2]], [h[-1]]
    torch.manual_seed(0)
    args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=L, num_layers=nl, hidden_units=H, dropout=0.2)
    m = SuperSASRecModel(usernum, itemnum, REC, IND, args).cuda().eval()
    m.precision = 1
    ds = DeviceSampler(train, valid, test, usernum, itemnum, L, seed=4)
    users = np.arange(1, usernum + 1, dtype=np.int32)
    batches = [ds.eval_batch(users[i:i + 128], mode="val", n_candidates=100) for i in range(0, usernum, 128)]
    cands = [list(rng.random(2 * nl) * 0.98) for _ in range(4)]
    pe = PopulationEvaluator(m, batches, REC, IND, in_flight=3)
    got = pe.evaluate(cands)
    for c, cand in enumerate(cands):
        set_choice_from_candidate(m, cand, REC, IND)
        auc, ndcg, hr = candidate_fitness(m, [(None, s, i) for s, i in batches], k=10)
        assert abs(got[c][0] - auc) < 1e-9 and abs(got[c][1] - ndcg) < 1e-6 and abs(got[c][2] - hr) < 1e-9, (c, got[c], (auc, ndcg, hr))
    assert len({tuple(np.round(r, 6)) for r in got}) > 1
