"""STOSA full-catalog ranking, host side: the centred-dot-product identity in fp64 on the reference fixtures, when the model's derived
catalog is stale, how it is keyed and sharded.  No GPU needed: nothing here launches a kernel."""
import types

import numpy as np
import pytest
import torch

import stosa_catalog_ref as R
from adt_b200.evaluate import Catalog, CatalogScorer, catalog_of, shard_bounds
from adt_b200.stosa import DisenDistSAModel
from oracle import stosa_oracle as O


@pytest.mark.parametrize("name", R.NAMES)
def test_identity_reproduces_reference_distances(name):
    g = R.load(name)
    sd = R.state_dict(g)
    mu, e, b = R.catalog(sd["item_mean_embeddings.weight"], sd["item_cov_embeddings.weight"])
    assert np.allclose(mu, R.item_rows(sd["item_mean_embeddings.weight"], sd["item_cov_embeddings.weight"]).mean(0))
    um, uc = R.last_states(g, sd)
    f = R.feats(um, uc, mu)
    x = R.user_rows(um, uc) - mu
    neg_dist = f @ e.T + b[None, :] - (x * x).sum(1, keepdims=True)
    dist = np.asarray(g["dist"], np.float64)
    assert np.abs(neg_dist + dist).max() <= 1e-5 * np.abs(dist).max()
    # ranking by <f, e> + b (the constant per user dropped) is the reference's full-sort protocol, up to fp32 near-ties
    seen, _, _ = R.seen_sets(g["seq"])
    K = 10
    score = f @ e.T + b[None, :]
    for u, s in enumerate(seen):
        score[u, s] = -np.inf
    order = np.lexsort((np.broadcast_to(np.arange(score.shape[1]), score.shape), -score), axis=1)[:, :K]
    ref = O.full_sort_topk(dist, seen, K)
    R.assert_same_up_to_near_ties(order, ref, dist, 1e-4)
    for u, s in enumerate(seen):
        assert not set(order[u]) & set(s)


def _stosa(item_size=1000, H=16):
    args = types.SimpleNamespace(item_size=item_size, num_users=4, maxlen=8, hidden_units=H, num_heads=2, num_layers=1, dropout=0.1,
                                 attention_dropout=0.1, initializer_range=0.02)
    torch.manual_seed(0)
    m = DisenDistSAModel(args)
    builds = []

    def build():     # the buffers _build_catalog allocates, without the kernel launch
        builds.append(m._catalog_key())
        n, H_ = m.item_mean_embeddings.weight.shape
        m._wcat = (torch.zeros(2 * H_), torch.zeros(n, 2 * H_), torch.zeros(n), None)
        m._wcat_key = m._catalog_key()

    m._build_catalog = build
    return m, builds


def test_catalog_is_every_row_from_id_0_with_bias():
    m, builds = _stosa(1000, 16)
    c = catalog_of(m)
    assert len(builds) == 1
    assert tuple(c.table.shape) == (1000, 32) and tuple(c.bias.shape) == (1000,)
    assert c.first_id == 0 and c.hidden == 32 and c.version == m._catalog_key()


def test_staleness_key_tracks_tables_optimizer_steps_and_replacement_only():
    m, builds = _stosa()
    catalog_of(m)
    k0 = m._catalog_key()
    assert m._catalog_key() == k0
    # nothing else marks it stale: other parameters, a forward's bookkeeping, repeated reads
    with torch.no_grad():
        m.LayerNorm.weight.mul_(1.5)
        m.position_mean_embeddings.weight.add_(1.0)
        m.item_encoder.layer[0].attention.mean_query.weight.add_(1.0)
    m.drop_step += 3
    for _ in range(3):
        catalog_of(m)
    assert m._catalog_key() == k0 and len(builds) == 1
    seen = {k0}
    for edit in (lambda: m.item_mean_embeddings.weight[3, 0].add_(1.0),       # in-place edit of either table
                 lambda: m.item_cov_embeddings.weight[0, 1].sub_(1.0),
                 lambda: setattr(m, "_adt_param_version", getattr(m, "_adt_param_version", 0) + 1),   # FlatOptimizer.step
                 lambda: setattr(m.item_cov_embeddings, "weight", torch.nn.Parameter(m.item_cov_embeddings.weight.detach().clone()))):
        with torch.no_grad():
            edit()
        k = m._catalog_key()
        assert k not in seen
        seen.add(k)
        c = catalog_of(m)
        assert builds[-1] == k and c.version == k
        catalog_of(m)
        assert builds[-1] == k
    assert len(builds) == 5


def test_table_key_follows_catalog_version():
    E = torch.randn(64, 8)
    cat = {"v": ("a", 1)}
    model = types.SimpleNamespace(scoring_catalog=lambda: Catalog(E, None, 0, 8, cat["v"]))
    sc = CatalogScorer(model, K=5)
    k0 = sc._table_key()
    assert sc._table_key() == k0
    cat["v"] = ("a", 2)                             # rebuilt in place: same storage, same tensor version, new catalog version
    assert sc._table_key() != k0


def test_unversioned_catalogs_keep_their_keys():
    """SASRec (whole item table) and Bert4Rec (tied head rows + bias) catalogs carry no version: their keys change exactly when the
    tensors or the optimiser step change, as before."""
    from adt_b200.bert4rec import BertModel
    args = types.SimpleNamespace(device="cpu", num_heads=2, maxlen=8, num_layers=1, hidden_units=16, dropout=0.1, attention_dropout=0.1,
                                 inner_units=32, type_vocab_size=2)
    bert = BertModel(10, 500, args)
    sas = types.SimpleNamespace(item_emb=types.SimpleNamespace(weight=torch.randn(77, 8)), hidden=8)
    for model, table in ((bert, bert.item_emb.word_emb.weight), (sas, sas.item_emb.weight)):
        assert catalog_of(model).version is None
        sc = CatalogScorer(model, K=5)
        k0 = sc._table_key()
        assert sc._table_key() == k0 and k0[-1] is None
        with torch.no_grad():
            table[2, 0] += 1.0
        assert sc._table_key() != k0


@pytest.mark.parametrize("world", [2, 3, 8])
def test_shards_cover_every_row(world):
    n = 12_103
    m, _ = _stosa(n, 16)
    sc = CatalogScorer(m, K=10)
    assert sc.bounds() == (0, n)
    got = []
    for rank in range(world):
        sc.world, sc.rank, sc.sharded = world, rank, True
        lo, hi = sc.bounds()
        assert (lo, hi) == shard_bounds(n, world, rank) and lo % 4 == 0
        got.extend(range(sc.catalog().first_id + lo, sc.catalog().first_id + hi))
    assert got == list(range(n))


def test_hidden_limit_is_named():
    args = types.SimpleNamespace(item_size=100, num_users=4, maxlen=8, hidden_units=256, num_heads=2, num_layers=1, dropout=0.1,
                                 attention_dropout=0.1, initializer_range=0.02)
    m = DisenDistSAModel(args)
    from adt_b200._lib import AdtError
    with pytest.raises(AdtError, match="128"):
        m._build_catalog()
