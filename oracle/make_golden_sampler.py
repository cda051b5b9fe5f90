"""TEST INFRASTRUCTURE ONLY.  Writes tests/golden/sampler_ref.npz: what the UNMODIFIED reference's dataset classes produce on
the toy histories of tests/test_sampler.py, for the parts that are not random.

    python -m oracle.make_golden_sampler      # needs the reference checkout (oracle/build_ref.REF)

  sasrec/   WarpDataset.sample_data (sasrec/utils.py:288-307): seq / dec / pos and which positions get a negative, per user;
            PopularSampler.popular_p; EvalDataset.sample_data per mode: seq and the answer in column 0 of item_idx
  bert4rec/ BertTrainDataset(generate=True, mask_prob 0): the instance list datas / labels (tokens, decoder copy, labels)
"""
import importlib
import os
import sys
import types

import numpy as np

from oracle.build_ref import REF

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "sampler_ref.npz")
SASREC_L, BERT_USERS, BERT_ITEMS, BERT_L = 12, 25, 80, 10


def toy_histories(rng, usernum=40, itemnum=60, maxhist=30):
    train, valid, test = {}, {}, {}
    for u in range(1, usernum + 1):
        n = int(rng.integers(0, maxhist))
        h = [int(x) for x in rng.integers(1, itemnum + 1, size=n)]
        if len(h) >= 3:
            train[u], valid[u], test[u] = h[:-2], [h[-2]], [h[-1]]
        else:
            train[u], valid[u], test[u] = h, [], []
    return train, valid, test, usernum, itemnum


def bert_histories():
    rng = np.random.default_rng(2)
    return {u: [int(x) for x in rng.integers(1, BERT_ITEMS + 1, size=int(rng.integers(0, 35)))] for u in range(1, BERT_USERS + 1)}


def sasrec_layout():
    for name in ("matplotlib", "matplotlib.pyplot"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.path.insert(0, os.path.join(REF, "sasrec"))
    R = importlib.import_module("utils")
    train, valid, test, usernum, itemnum = toy_histories(np.random.default_rng(0))
    wd = R.WarpDataset(train, usernum, itemnum, SASREC_L)
    users = [u for u in range(1, usernum + 1) if len(train[u]) >= 1]
    rows = [[np.asarray(a) for a in wd.sample_data(u)[1:]] for u in users]
    out = {"train_users": np.array(users), "train_seq": np.stack([r[0] for r in rows]), "train_dec": np.stack([r[1] for r in rows]),
           "train_pos": np.stack([r[2] for r in rows]), "train_neg_mask": np.stack([r[3] != 0 for r in rows])}
    sampler = R.PopularSampler(train, valid, test, usernum, itemnum, 10)
    out["popular_p"] = np.asarray(sampler.popular_p, dtype=np.float64)
    for mode in ("val", "test"):
        ds = R.EvalDataset(train, valid, test, usernum, itemnum, SASREC_L, sampler, mode=mode, eval_set=-1)
        rows = [ds.sample_data(u) for u in ds.users]
        out[f"{mode}_users"] = np.array([int(u) for u in ds.users])
        out[f"{mode}_seq"] = np.stack([np.asarray(r[1]) for r in rows])
        out[f"{mode}_answer"] = np.array([int(np.asarray(r[2])[0]) for r in rows])
    return out


def bert4rec_layout():
    pkg = types.ModuleType("refbert_datasets")          # the reference's `datasets/` has no __init__.py: mount it as a package
    pkg.__path__ = [os.path.join(REF, "bert4rec", "datasets")]
    sys.modules["refbert_datasets"] = pkg
    mod = importlib.import_module("refbert_datasets.dataset")
    d = mod.BertTrainDataset(bert_histories(), {}, {}, BERT_USERS, BERT_ITEMS, BERT_L, None, 0.0, 1, generate=True, dupe_factor=2,
                             prop_sliding_window=0.5)
    return {"tok": np.stack([np.asarray(x[0]) for x in d.datas]), "dec": np.stack([np.asarray(x[1]) for x in d.datas]),
            "labels": np.stack([np.asarray(y) for y in d.labels])}


if __name__ == "__main__":
    arrays = {f"sasrec/{k}": v for k, v in sasrec_layout().items()}
    arrays.update({f"bert4rec/{k}": v for k, v in bert4rec_layout().items()})
    np.savez_compressed(OUT, **arrays)
    print(f"wrote {OUT} ({os.path.getsize(OUT)} bytes)")
