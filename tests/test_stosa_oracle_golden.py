"""CPU: the STOSA oracle restatement (oracle/stosa_oracle.py) against fixtures produced by the UNMODIFIED reference
(oracle/make_golden_stosa.py: DisenDistSAModel.finetune + DistSAModelTrainer.{bpr_optimization,iteration,dist_predict_full})."""
import glob
import os
import numpy as np
import pytest
import torch

from oracle import stosa_oracle as SO
from oracle.sasrec_oracle import Drop
from helpers import rel_err, GOLDEN

NAMES = sorted(os.path.basename(p)[6:-4] for p in glob.glob(os.path.join(GOLDEN, "stosa_*.npz")))


def load(name):
    z = np.load(os.path.join(GOLDEN, f"stosa_{name}.npz"))
    return {k: z[k] for k in z.files}


def test_fixtures_present():
    assert len(NAMES) >= 3


@pytest.mark.parametrize("name", NAMES)
def test_stosa_forward_loss_grads(name):
    g = load(name)
    B, L, H, nh, nl, I = [int(v) for v in g["cfg"]]
    cfg = SO.SCfg(I + 2, B, L, H, nh, nl, float(g["p"]), float(g["pa"]), float(g["pvn"]))
    sd = {k[4:]: torch.from_numpy(np.array(v)).requires_grad_(True) for k, v in g.items() if k.startswith("sd0/")}
    seq, dec, pos, neg = (torch.from_numpy(g[k]) for k in ("seq", "dec", "pos", "neg"))
    drop = Drop(0.5, int(g["drop_seed"]), int(g["drop_step"]), train=True)
    out = SO.forward(sd, cfg, seq, dec, drop)
    assert rel_err(out["mean"].detach(), g["mean"]) < 2e-5
    assert rel_err(out["cov"].detach(), g["cov"]) < 2e-5
    dec_rev = list(reversed(out["dec_outputs"]))
    for l in range(nl):
        for j, s in enumerate(("mean", "cov")):
            assert rel_err(out["enc_inputs"][l][j].detach(), g[f"enc_in_{s}{l}"]) < 2e-5
            assert rel_err(dec_rev[l][j].detach(), g[f"dec_out_{s}{l}"]) < 2e-5
            assert rel_err(out["recs"][l][j].detach(), g[f"rec_{s}{l}"]) < 2e-5
    total, bpr, pvn, auc = SO.loss(sd, cfg, out, pos, neg, list(g["lambda1"]), list(g["lambda2"]))
    assert abs(float(total) - float(g["loss"])) / abs(float(g["loss"])) < 1e-5
    assert abs(float(bpr) - float(g["bpr"])) / abs(float(g["bpr"])) < 1e-5
    assert abs(float(pvn) - float(g["pvn_loss"])) / abs(float(g["pvn_loss"])) < 1e-5
    assert abs(float(auc) - float(g["auc"])) < 1e-6
    total.backward()
    n = 0
    for k, p in sd.items():
        if "grad/" + k in g:
            assert rel_err(p.grad, g["grad/" + k]) < 5e-4, k
            n += 1
        else:   # user margins, the discarded decoder self attention, decLayerNorm: never reached by the loss
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
    assert n > 50
    # evaluation scores of the updated model + the reference's top-40 protocol
    sd1 = {k[4:]: torch.from_numpy(np.array(v)) for k, v in g.items() if k.startswith("sd1/")}
    dist = SO.predict_full(sd1, cfg, seq).numpy()
    assert rel_err(dist, g["dist"]) < 2e-5
    seen = [set(int(v) for v in row if v > 0) for row in g["seq"]]
    top = SO.full_sort_topk(dist, seen, K=10)
    ref = SO.full_sort_topk(g["dist"], seen, K=10)
    assert (top == ref).mean() > 0.95


@pytest.mark.parametrize("name", NAMES)
def test_init_state_layout(name):
    """init_state builds the reference's state dict: the fixture's sd0/ names, in order, with its shapes."""
    g = load(name)
    B, L, H, nh, nl, I = [int(v) for v in g["cfg"]]
    sd = SO.init_state(SO.SCfg(I + 2, B, L, H, nh, nl), seed=0)
    ref = [(k[4:], g[k].shape) for k in g if k.startswith("sd0/")]
    assert [(k, tuple(v.shape)) for k, v in sd.items()] == ref


def _c4_batch(rng, B, L, I):
    """left-padded batch with random lengths in 1..L; sequence 0 is full length, 1 has one item, 2 is all padding."""
    seq, pos, neg = (np.zeros((B, L), np.int64) for _ in range(3))
    for b in range(B):
        n = (L, 1, 0)[b] if b < 3 else int(rng.integers(1, L + 1))
        it = rng.integers(1, I + 1, size=n + 1)
        seq[b, L - n:], pos[b, L - n:], neg[b, L - n:] = it[:-1], it[1:], rng.integers(1, I + 1, size=n)
    dec = np.zeros_like(seq)
    dec[:, 1:] = seq[:, :-1]
    return [torch.from_numpy(x) for x in (seq, dec, pos, neg)]


def _oracle_step(sd, cfg, batch, drop, l1, l2):
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
    out = SO.forward(sd, cfg, batch[0], batch[1], drop)
    total = SO.loss(sd, cfg, out, batch[2], batch[3], l1, l2)[0]
    total.backward()
    return float(total.detach()), {k: v.grad for k, v in sd.items()}


def test_fp64_oracle_matches_fp32_at_c4_shape():
    """The fp64 oracle is a valid reference for the fp32 kernels at the benchmarked shape (B 16 of C4: L 100, H 64, nh 4, nl 1,
    dropout 0.3 / 0.3).  Left-padded query rows are all-masked; only the fp32 mask semantics of attention_core keep their softmax
    uniform in fp64, as the reference (and the kernel) compute it.  Without them the worst gradient is off by a few percent of its max."""
    B, L, H, nh, I = 16, 100, 64, 4, 3000
    cfg = SO.SCfg(I + 2, B, L, H, nh, 1, 0.3, 0.3)
    batch = _c4_batch(np.random.default_rng(0), B, L, I)
    sd = SO.init_state(cfg, seed=0)
    drop = Drop(0.3, 11, 3, train=True)
    l1, l2 = [0.0021], [0.0009]
    loss32, g32 = _oracle_step(sd, cfg, batch, drop, l1, l2)
    loss64, g64 = _oracle_step({k: v.double() for k, v in sd.items()}, cfg, batch, drop, l1, l2)
    assert abs(loss32 - loss64) <= 1e-6 * abs(loss64)
    n = 0
    for k, g in g64.items():
        if g is None or float(g.abs().max()) == 0.0:
            assert g32[k] is None or float(g32[k].abs().max()) == 0.0, k
            continue
        assert rel_err(g32[k], g) <= 1e-4, (k, rel_err(g32[k], g))
        n += 1
    assert n > 50
