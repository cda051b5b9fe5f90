"""Bert4Rec full-catalog evaluation, host side: which rows of the tied table are ranked, how they are sharded, and when the
scorer's bf16 copy (and the bias bound) must be rebuilt.  No GPU needed: nothing here launches a kernel."""
import types

import torch

from adt_b200.bert4rec import BertModel
from adt_b200.evaluate import CatalogScorer, catalog_of, shard_bounds


def _bert(I=1000, H=16):
    args = types.SimpleNamespace(device="cpu", num_heads=2, maxlen=8, num_layers=1, hidden_units=H, dropout=0.1, attention_dropout=0.1,
                                 inner_units=32, type_vocab_size=2)
    torch.manual_seed(0)
    return BertModel(10, I, args)


def test_bert_catalog_is_items_1_to_itemnum_with_mask_bias():
    I, H = 1000, 16
    m = _bert(I, H)
    c = catalog_of(m)
    W, b = m.item_emb.word_emb.weight, m.mask_bias
    assert W.shape[0] == I + 100                       # padding row, items, mask token and the unused vocabulary
    assert tuple(c.table.shape) == (I, H) and c.table.data_ptr() == W[1].data_ptr()
    assert tuple(c.bias.shape) == (I,) and c.bias.data_ptr() == b[1:].data_ptr()
    assert c.first_id == 1 and c.hidden == H
    ids = c.first_id + torch.arange(c.table.shape[0])
    assert int(ids.min()) == 1 and int(ids.max()) == I   # never 0 (padding) nor I+1 (the mask token)


def test_plain_models_keep_the_whole_table_without_bias():
    E = torch.randn(77, 8)
    c = catalog_of(types.SimpleNamespace(item_emb=types.SimpleNamespace(weight=E), hidden=8))
    assert c.table is E and c.bias is None and c.first_id == 0 and c.hidden == 8


def test_shards_partition_the_bert_catalog():
    I = 70_001
    m = _bert(I)
    sc = CatalogScorer(m, K=10)
    assert sc.bounds() == (0, I)
    for world in (2, 3, 8):
        got = []
        for rank in range(world):
            sc.world, sc.rank, sc.sharded = world, rank, True
            lo, hi = sc.bounds()
            assert (lo, hi) == shard_bounds(I, world, rank) and lo % 4 == 0
            got.extend(range(sc.catalog().first_id + lo, sc.catalog().first_id + hi))
        assert got == list(range(1, I + 1))


def test_table_key_tracks_table_bias_and_optimizer_steps():
    m = _bert()
    sc = CatalogScorer(m, K=10)
    k0 = sc._table_key()
    assert sc._table_key() == k0
    with torch.no_grad():
        m.mask_bias[5] += 1.0                      # in-place edit of the bias alone
    k1 = sc._table_key()
    assert k1 != k0
    with torch.no_grad():
        m.item_emb.word_emb.weight[3, 0] += 1.0    # ... of the table
    k2 = sc._table_key()
    assert k2 != k1
    m._adt_param_version = getattr(m, "_adt_param_version", 0) + 1     # what FlatOptimizer.step does after writing through pointers
    assert sc._table_key() != k2
