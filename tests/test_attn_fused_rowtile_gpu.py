"""Attention fused into the H = 64 projection kernels (ADT_ATTN_FUSED=1, sequences of 33 .. 64 positions) against the separate
attention launches (ADT_ATTN_FUSED=0, separate process: the switch is read once per process), through the block C ABI.  The per-row
arithmetic is the same on both paths, so the forward outputs and the row-wise backward outputs (dx, dfeats, dctx, ...) must agree
bit for bit; the weight gradients are fp32 atomic sums over differently cut row tiles and agree to re-association.  At L <= 32 both
settings run the separate launches."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# (B, L, nh, mask_mode, dropout, left padding of each sequence, data-parallel batch offset)
_CASES = [
    (7, 50, 2, 0, 0.5, [0, 1, 20, 49, 50, 3, 0], 3),      # C2 shape, an empty sequence, non-zero DP offset
    (5, 64, 4, 1, 0.3, [0, 63, 10, 5, 0], 0),            # L = 64, four heads, key-padding mask
    (3, 33, 1, 0, 0.0, [0, 32, 7], 0),                   # L = 33, one head (forward fused, backward separate), no dropout
    (6, 63, 2, 1, 0.0, [1, 0, 62, 30, 8, 0], 11),         # odd L, key-padding mask, no dropout
    (4, 40, 4, 0, 0.5, [39, 0, 3, 12], 1),               # four heads with dropout
    (5, 32, 2, 0, 0.5, [0, 5, 31, 2, 0], 0),             # L = 32: not fused
    (3, 20, 4, 1, 0.3, [0, 19, 4], 2),                   # L = 20: not fused
]
_ROW_OUT = ("enc/q", "enc/k", "enc/v", "enc/ctx", "enc/lse", "enc/y", "enc/h1", "enc/out", "enc/rec", "enc/dx", "enc/dctx", "enc/dy",
            "dec/d", "dec/q1", "dec/k1", "dec/v1", "dec/ctx1", "dec/a", "dec/q2", "dec/k2", "dec/v2", "dec/ctx2", "dec/c", "dec/h1",
            "dec/out", "dec/lse1", "dec/lse2", "dec/dx", "dec/dfeats", "dec/dctx", "dec/dd", "dec/dctx2")


def _run_blocks(case):
    """encoder and decoder block, forward and backward, on seeded inputs -> {name: array}, {"names/<call>": kernel names}"""
    import block_harness as BH
    B, Lq, nh, mask_mode, p, pad, b0 = case
    c = BH.Case(B, Lq, 64, nh, pad, mask_mode=mask_mode, p=p, b0=b0)
    return BH.run(c, BH.inputs(c))


def _trainer_step():
    """one C2-shaped training step (B 64) captured in and replayed from a CUDA graph -> (loss, gradient norm)"""
    import types
    import torch
    from adt_b200 import synth
    from adt_b200.model import SASRecADT
    from adt_b200.trainer import FusedTrainer
    cfg = dict(synth.CONFIGS["C2"], B=64)
    torch.manual_seed(0)
    args = types.SimpleNamespace(device="cuda", num_heads=cfg["nh"], maxlen=cfg["L"], num_layers=cfg["nl"], hidden_units=cfg["H"], dropout=0.5)
    m = SASRecADT(1, cfg["items"], args)
    for _, prm in m.named_parameters():
        if prm.dim() >= 2:
            torch.nn.init.xavier_normal_(prm.data)
    m = m.cuda().train()
    tr = FusedTrainer(m, [0.0124, 0.122], [0.0001, 0.05], weight_decay=1e-4, seed=5, precision="bf16", use_graph=True)
    tr.step(*synth.make_batch(np.random.default_rng(3), cfg))
    return tr.loss(), tr.grad_norm()


if __name__ == "__main__":      # helper process: python <this file> <case | step> <out.npz>
    if sys.argv[1] == "step":
        loss, gnorm = _trainer_step()
        np.savez(sys.argv[2], loss=loss, gnorm=gnorm)
    else:
        res = _run_blocks(_CASES[int(sys.argv[1])])
        names = sorted({n for k, v in res.items() if k.startswith("names/") for n in v})
        np.savez(sys.argv[2], names=np.array(names), **{k: v for k, v in res.items() if not k.startswith("names/")})
    sys.exit(0)


def _both(arg, tmp_path):
    here = os.path.abspath(__file__)
    res = []
    for fused in ("1", "0"):
        f = str(tmp_path / f"fused{fused}.npz")
        e = dict(os.environ, ADT_ATTN_FUSED=fused)
        e["PYTHONPATH"] = os.pathsep.join([os.path.dirname(os.path.dirname(here)), os.path.dirname(here), e.get("PYTHONPATH", "")])
        subprocess.run([sys.executable, here, arg, f], check=True, env=e, timeout=600)
        res.append(np.load(f))
    return res


@pytest.mark.parametrize("case", range(len(_CASES)))
def test_fused_attention_matches_separate_launches(case, tmp_path):
    a, b = _both(str(case), tmp_path)
    L_, nh = _CASES[case][1], _CASES[case][2]
    names_a, names_b = set(a["names"].tolist()), set(b["names"].tolist())
    fused = L_ > 32
    assert ("pre_attn_fwd" in names_a) == fused and "pre_attn_fwd" not in names_b
    assert ("mid_attn_fwd" in names_a) == fused and "mid_attn_fwd" not in names_b
    assert ("attn_pre_bwd" in names_a) == (fused and nh in (2, 4)) and "attn_pre_bwd" not in names_b
    for k in _ROW_OUT:
        assert np.array_equal(a[k], b[k]), (k, float(np.abs(a[k] - b[k]).max()))
    for k in a.files:
        if "/g_" in k:
            x, y = a[k], b[k]
            assert np.abs(x - y).max() <= 1e-5 * np.abs(y).max() + 1e-12, (k, float(np.abs(x - y).max()), float(np.abs(y).max()))


def test_fused_attention_graphed_trainer_step(tmp_path):
    a, b = _both("step", tmp_path)
    assert abs(float(a["loss"]) - float(b["loss"])) <= 1e-6 * abs(float(b["loss"]))
    assert abs(float(a["gnorm"]) - float(b["gnorm"])) <= 1e-6 * float(b["gnorm"])
