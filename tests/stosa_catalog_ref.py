"""fp64 restatement of STOSA's full-catalog ranking as a centred, biased dot product (adt_wcatalog_build / adt_wcatalog_user), and the
fixture glue the STOSA catalog tests share.  With item rows y_i = [mean_i | sqrt(elu(cov_i)+1)], user rows x_u = [mean_u | sqrt(cov_u)]
and mu the column mean of the y_i:
    -|x_u - y_i|^2 = <f_u, e_i> + b_i - |x_u - mu|^2,   f_u = 2 (x_u - mu), e_i = y_i - mu, b_i = -|e_i|^2."""
import glob
import os
import types

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMES = sorted(os.path.basename(p)[6:-4] for p in glob.glob(os.path.join(GOLDEN, "stosa_*.npz")))
CLAMP = 1e-24          # torch.clamp(cov, min=1e-24) before the square root (stosa/modules.py:24-25)


def load(name):
    z = np.load(os.path.join(GOLDEN, f"stosa_{name}.npz"))
    return {k: z[k] for k in z.files}


def args_of(g):
    B, L, H, nh, nl, I = [int(v) for v in g["cfg"]]
    return types.SimpleNamespace(item_size=I + 2, num_users=B, maxlen=L, hidden_units=H, num_heads=nh, num_layers=nl,
                                 dropout=float(g["p"]), attention_dropout=float(g["pa"]), initializer_range=0.02,
                                 pvn_weight=float(g["pvn"]))


def state_dict(g, prefix="sd1/"):
    return {k[len(prefix):]: torch.from_numpy(np.array(v)) for k, v in g.items() if k.startswith(prefix)}


def item_rows(Em, Ec):
    Em, Ec = np.asarray(Em, np.float64), np.asarray(Ec, np.float64)
    cov = np.where(Ec > 0, Ec + 1.0, np.exp(Ec))                     # elu + 1
    return np.concatenate([Em, np.sqrt(np.maximum(cov, CLAMP))], axis=1)


def user_rows(m, c):
    m, c = np.asarray(m, np.float64), np.asarray(c, np.float64)
    return np.concatenate([m, np.sqrt(np.maximum(c, CLAMP))], axis=1)


def catalog(Em, Ec):
    """-> (mu [2H], e [n, 2H], b [n])"""
    y = item_rows(Em, Ec)
    mu = y.mean(axis=0)
    e = y - mu
    return mu, e, -(e * e).sum(axis=1)


def feats(m, c, mu):
    return 2.0 * (user_rows(m, c) - mu)


def last_states(g, sd):
    """the oracle's evaluation-mode (mean, cov) of the last position, fp32 as the reference computes them"""
    from oracle import stosa_oracle as O
    B, L, H, nh, nl, I = [int(v) for v in g["cfg"]]
    cfg = O.SCfg(I + 2, B, L, H, nh, nl)
    ids = torch.from_numpy(np.asarray(g["seq"])).long()
    out = O.forward({k: v.float() for k, v in sd.items()}, cfg, ids, ids)
    return out["mean"][:, -1, :].numpy(), out["cov"][:, -1, :].numpy()


def seen_sets(seq):
    seen = [sorted(set(int(v) for v in row if v > 0)) for row in seq]
    indptr = np.concatenate([[0], np.cumsum([len(s) for s in seen])]).astype(np.int32)
    return seen, indptr, np.concatenate(seen).astype(np.int32)


def assert_same_up_to_near_ties(ids, ref, dist, tol):
    """ids / ref [U, K]: equal, or the distances (fp64 [U, n]) of the two lists agree position by position within tol"""
    ids, ref = np.asarray(ids), np.asarray(ref)
    for u in range(ids.shape[0]):
        if (ids[u] == ref[u]).all():
            continue
        du = dist[u]
        assert np.abs(np.sort(du[ids[u]]) - du[ref[u]]).max() <= tol * max(1.0, np.abs(du[ref[u]]).max()), (u, ids[u], ref[u])
