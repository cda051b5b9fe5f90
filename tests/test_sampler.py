"""SURVEY 8f-1: device-side batch assembly / negative sampling.  CPU: the oracle restatement against what the UNMODIFIED reference
datasets produce (stored in tests/golden, and live where the reference checkout exists) for everything that is not random, and the
validity of what is.  GPU: the kernels against the oracle, bit for bit."""
import os

import numpy as np
import pytest
import torch

from oracle import make_golden_sampler as G
from oracle.make_golden_sampler import toy_histories as _toy


def _reference_layouts(part):
    """what the reference's dataset classes produce on the toy histories: the copy stored in tests/golden/sampler_ref.npz
    (oracle/make_golden_sampler.py) and, where the reference checkout exists, the live result as well."""
    got = []
    if os.path.exists(G.OUT):
        z = np.load(G.OUT)
        got.append({k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(part + "/")})
    if os.path.isdir(os.path.join(G.REF, part)):
        got.append(getattr(G, part + "_layout")())
    if not got:
        pytest.skip(f"neither {G.OUT} nor a reference checkout at {G.REF}: run `python -m oracle.make_golden_sampler` where it exists")
    return got


def test_oracle_batch_layout_matches_reference_datasets():
    """seq / dec / pos of WarpDataset.sample_data and seq / answer of EvalDataset.sample_data are deterministic: the oracle must equal
    the unmodified reference exactly; the random parts must satisfy the reference's constraints."""
    from oracle import sampler_oracle as S
    from adt_b200.sampler import alias_table
    train, valid, test, usernum, itemnum = _toy(np.random.default_rng(0))
    L = G.SASREC_L
    for ref in _reference_layouts("sasrec"):
        assert list(ref["train_users"]) == [u for u in range(1, usernum + 1) if len(train[u]) >= 1]
        for b, u in enumerate(int(x) for x in ref["train_users"]):
            o_seq, o_dec, o_pos, o_neg = S.train_sample(train[u], u, L, itemnum, seed=5, epoch=1)
            assert np.array_equal(ref["train_seq"][b], o_seq) and np.array_equal(ref["train_dec"][b], o_dec), u
            assert np.array_equal(ref["train_pos"][b], o_pos), u
            assert np.array_equal(ref["train_neg_mask"][b], o_neg != 0)
            assert not set(o_neg[o_neg != 0].tolist()) & set(train[u])
            assert o_neg.max(initial=0) <= itemnum
        popular_p = ref["popular_p"]
        ap, ai = alias_table(np.asarray(popular_p, dtype=np.float64))
        for mode in ("val", "test"):
            for b, u in enumerate(int(x) for x in ref[f"{mode}_users"]):
                seen = set(train[u]) | set(valid[u]) | (set(test[u]) if mode == "test" else set())
                ans = valid[u][0] if mode == "val" else test[u][0]
                o_seq, o_idx = S.eval_sample(train[u], seen, ans, valid[u][0] if mode == "test" else 0, u, L, itemnum, 10, ap, ai, seed=5,
                                             epoch=0)
                assert np.array_equal(ref[f"{mode}_seq"][b], o_seq), (mode, u)
                assert ref[f"{mode}_answer"][b] == o_idx[0] == ans
                neg = o_idx[1:]
                assert len(neg) == 10 and len(set(neg.tolist())) == 10
                assert not set(neg.tolist()) & seen and neg.max() < itemnum and neg.min() >= 0
                assert all(popular_p[i] > 0 for i in neg)        # only items that can be drawn by popularity (quirk B8: never id 0)


def test_alias_table_reproduces_the_distribution():
    from adt_b200.sampler import alias_table
    rng = np.random.default_rng(1)
    p = rng.random(37) ** 3
    p[5] = 0.0
    p /= p.sum()
    prob, alias = alias_table(p)
    q = np.zeros_like(p)
    for c in range(len(p)):
        q[c] += prob[c] / len(p)
        q[alias[c]] += (1.0 - prob[c]) / len(p)
    assert np.allclose(q, p, atol=1e-6)


@pytest.mark.gpu
def test_device_sampler_matches_oracle_bit_for_bit():
    from adt_b200.sampler import DeviceSampler
    from oracle import sampler_oracle as S
    rng = np.random.default_rng(3)
    train, valid, test, usernum, itemnum = _toy(rng, usernum=120, itemnum=300, maxhist=70)
    L = 50
    ds = DeviceSampler(train, valid, test, usernum, itemnum, L, seed=(7 << 32) | 99)
    users = np.array([u for u in range(1, usernum + 1) if len(train[u]) >= 1], np.int32)
    for epoch in (0, 3):
        seq, dec, pos, neg = [t.cpu().numpy() for t in ds.train_batch(users, epoch=epoch)]
        for b, u in enumerate(users):
            o = S.train_sample(train[int(u)], int(u), L, itemnum, seed=(7 << 32) | 99, epoch=epoch)
            for got, ref, name in zip((seq[b], dec[b], pos[b], neg[b]), o, ("seq", "dec", "pos", "neg")):
                assert np.array_equal(got, ref), (name, int(u), epoch)
    # a sample does not depend on its batch
    sub = users[::7]
    again = [t.cpu().numpy() for t in ds.train_batch(sub, epoch=3)]
    assert np.array_equal(again[3], neg[::7])
    ap, ai = ds.alias_prob.cpu().numpy(), ds.alias_idx.cpu().numpy()
    ev_users = np.array([u for u in range(1, usernum + 1) if len(valid[u]) and len(train[u])], np.int32)
    for mode in ("val", "test"):
        seq, idx = [t.cpu().numpy() for t in ds.eval_batch(ev_users, mode=mode, n_candidates=100, epoch=2)]
        for b, u in enumerate(ev_users):
            u = int(u)
            seen = set(train[u]) | set(valid[u]) | (set(test[u]) if mode == "test" else set())
            ans = valid[u][0] if mode == "val" else test[u][0]
            o_seq, o_idx = S.eval_sample(train[u], seen, ans, valid[u][0] if mode == "test" else 0, u, L, itemnum, 100, ap, ai,
                                         seed=(7 << 32) | 99, epoch=2)
            assert np.array_equal(seq[b], o_seq), (mode, u)
            assert np.array_equal(idx[b], o_idx), (mode, u)


@pytest.mark.gpu
def test_device_candidates_follow_popularity():
    """frequency of the FIRST drawn negative over many epochs ~ popular_p restricted to the unseen items (successive sampling)"""
    from adt_b200.sampler import DeviceSampler
    rng = np.random.default_rng(5)
    train, valid, test, usernum, itemnum = _toy(rng, usernum=30, itemnum=40, maxhist=12)
    ds = DeviceSampler(train, valid, test, usernum, itemnum, 10, seed=11)
    u = next(u for u in range(1, usernum + 1) if len(valid[u]))
    users = np.full(4096, u, np.int32)
    counts = np.zeros(itemnum)
    for epoch in range(8):
        _, idx = ds.eval_batch(users[:1], mode="val", n_candidates=5, epoch=epoch)       # same user, different epochs -> different draws
    firsts = []
    for epoch in range(600):
        _, idx = ds.eval_batch(users[:1], mode="val", n_candidates=5, epoch=epoch)
        firsts.append(int(idx[0, 1]))
    for f in firsts:
        counts[f] += 1
    seen = set(train[u]) | set(valid[u])
    p = ds.popular_p.copy()
    p[list(i for i in seen if i < itemnum)] = 0.0
    p /= p.sum()
    assert counts[[i for i in range(itemnum) if p[i] == 0]].sum() == 0
    assert np.abs(counts / counts.sum() - p).max() < 0.08


def test_cloze_instance_table_and_layout_match_reference_dataset():
    """SURVEY 8f-3: the window enumeration of BertTrainDataset._generate_data and the deterministic layout of sample_data / _mask_last
    (right alignment, decoder copy ending in the mask token, labels) against the UNMODIFIED reference dataset class."""
    from adt_b200.sampler import ClozeSampler
    from oracle import sampler_oracle as S
    train, L, itemnum = G.bert_histories(), G.BERT_L, G.BERT_ITEMS
    tab = ClozeSampler.instance_table(train, G.BERT_USERS, L, 2, 0.5)
    for ref in _reference_layouts("bert4rec"):
        assert len(tab) == len(ref["tok"])
        # with mask_prob = 0 nothing is masked: tokens = window, decoder copy = window with the last position masked, labels = 0
        for b, row in enumerate(tab):
            u, st, ln, dup = [int(x) for x in row]
            tok, dec, lab = S.cloze_sample(train[u], u, st, ln, dup, L, itemnum, 0.0, seed=1, epoch=0)
            assert np.array_equal(tok, ref["tok"][b]) and np.array_equal(dec, ref["dec"][b]) and np.array_equal(lab, ref["labels"][b]), row


@pytest.mark.gpu
def test_device_cloze_batches_match_oracle_and_mask_rates():
    from adt_b200.sampler import ClozeSampler
    from oracle import sampler_oracle as S
    rng = np.random.default_rng(4)
    usernum, itemnum, L = 60, 500, 40
    train = {u: [int(x) for x in rng.integers(1, itemnum + 1, size=int(rng.integers(0, 120)))] for u in range(1, usernum + 1)}
    cs = ClozeSampler(train, usernum, itemnum, L, mask_prob=0.2, dupe_factor=3, prop_sliding_window=0.5, seed=(3 << 32) | 5)
    idx = np.arange(len(cs))
    tok, dec, lab = [t.cpu().numpy() for t in cs.batch(idx, epoch=2)]
    for b in range(0, len(cs), 7):
        u, st, ln, dup = [int(x) for x in cs.table[b]]
        o = S.cloze_sample(train[u], u, st, ln, dup, L, itemnum, 0.2, seed=(3 << 32) | 5, epoch=2)
        assert np.array_equal(tok[b], o[0]) and np.array_equal(dec[b], o[1]) and np.array_equal(lab[b], o[2]), b
    reg = cs.table[:, 3] >= 0
    valid = tok[reg] != 0
    masked = lab[reg] != 0
    rate = masked.sum() / valid.sum()
    assert abs(rate - 0.2) < 0.02
    m = masked
    frac_mask = (tok[reg][m] == itemnum + 1).mean()
    assert abs(frac_mask - 0.8) < 0.05
    # different epochs -> different masks; same epoch -> identical (counter based)
    tok2 = cs.batch(idx, epoch=3)[0].cpu().numpy()
    assert not np.array_equal(tok, tok2)
    assert np.array_equal(tok, cs.batch(idx, epoch=2)[0].cpu().numpy())
