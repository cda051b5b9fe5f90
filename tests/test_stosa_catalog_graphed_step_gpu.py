"""STOSA full-catalog ranking after training steps replayed by GraphedStep.  The replayed Adam kernel writes the item tables through
raw pointers and moves no tensor version, so the ranked catalog (and the scorer's bf16 copy) must be refreshed from GraphedStep's own
announcement: eager full_sort_topk and a GraphedScorer evaluated between GraphedStep epochs must equal a model whose catalog is built
from scratch out of the same parameters, and the tables must have moved between evaluations."""
import types

import numpy as np
import pytest
import torch

import stosa_catalog_ref as R

pytestmark = pytest.mark.gpu


def _args(I, L, H=64):
    return types.SimpleNamespace(item_size=I, num_users=16, maxlen=L, hidden_units=H, num_heads=2, num_layers=1, dropout=0.1,
                                 attention_dropout=0.1, initializer_range=0.02, pvn_weight=0.005)


def _train_batch(rng, I, B, L):
    seq = np.asarray([rng.integers(1, I, size=L) for _ in range(B)], dtype=np.int64)
    dec = np.zeros_like(seq)
    dec[:, 1:] = seq[:, :-1]
    return seq, dec, np.roll(seq, -1, axis=1), rng.integers(1, I, size=(B, L))


def _eval_batch(rng, I, U, L):
    seq = np.zeros((U, L), np.int32)
    for u in range(U):
        n = int(rng.integers(3, L))
        seq[u, L - n:] = rng.integers(1, I, size=n)
    seen, ip, ix = R.seen_sets(seq)
    return seq, ip, ix, rng.integers(0, I, size=U).astype(np.int32)


@pytest.mark.parametrize("I", [5_000, 40_000], ids=["exact", "tc"])
def test_ranking_follows_graphed_step_training(I):
    from adt_b200.dp import FlatOptimizer, GraphedStep
    from adt_b200.evaluate import CatalogScorer, GraphedScorer, metrics_from_acc
    from adt_b200.stosa import DisenDistSAModel
    L, U, B, K = 20, 128, 16, 10
    torch.manual_seed(0)
    m = DisenDistSAModel(_args(I, L)).cuda().train()
    opt = FlatOptimizer(m, lr=1e-2)
    step = GraphedStep(m, opt, lambda s, d, p, n: m.fused_loss(s, d, p, n, [0.01], [0.001])[0])
    rng = np.random.default_rng(7)
    train = [_train_batch(rng, I, B, L) for _ in range(3)]
    seq, ip, ix, ans = _eval_batch(rng, I, U, L)

    def epoch():
        for b in train:
            step.step(*b)
        torch.cuda.synchronize()

    def from_scratch():
        """a second model holding the same parameters: its catalog is built once, from the current tables"""
        fresh = DisenDistSAModel(_args(I, L)).cuda().eval()
        fresh.load_state_dict(m.state_dict())
        acc = torch.zeros(6, dtype=torch.float64, device="cuda")
        ids = fresh.full_sort_topk(seq, ip, ix, K=K, answers=ans, metric_acc=acc)
        return fresh, ids, metrics_from_acc(acc)

    epoch()
    gs = GraphedScorer(CatalogScorer(m, K=K), U, L, max_seen=len(ix))
    assert gs.tc == (I >= 32768)
    rows = []
    for _ in range(3):                                  # evaluate, train one GraphedStep epoch, evaluate again, ...
        fresh, ids_ref, met_ref = from_scratch()
        rows.append(fresh.scoring_catalog().table.clone())
        for got, want in zip(m.scoring_catalog()[:2], fresh.scoring_catalog()[:2]):
            assert torch.equal(got, want)                # the ranked rows and bias are those of the current tables
        acc = torch.zeros(6, dtype=torch.float64, device="cuda")
        ids = m.full_sort_topk(seq, ip, ix, K=K, answers=ans, metric_acc=acc)
        assert torch.equal(ids, ids_ref)
        ids_g = gs.topk(seq, ip, ix, ans)[1].clone()
        assert torch.equal(ids_g, ids_ref)
        met, met_g = metrics_from_acc(acc), gs.metrics()
        assert all(abs(met[k] - met_ref[k]) <= 1e-12 and abs(met_g[k] - met_ref[k]) <= 1e-12 for k in met_ref)
        epoch()
    # training moved the tables between evaluations, so rows kept from an earlier evaluation would have failed the comparison above
    assert not torch.equal(rows[0], rows[1]) and not torch.equal(rows[1], rows[2])
