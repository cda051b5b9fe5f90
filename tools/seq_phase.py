"""debug: per-phase clock64() deltas of CTA 0 of the sequence-resident encoder forward kernel during a C2 evaluation pass (after three
training steps)."""
import ctypes, os, sys, types
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import numpy as np, torch
from adt_b200 import synth, _lib as L
from adt_b200.model import SASRecADT
from adt_b200.trainer import FusedTrainer
from adt_b200.evaluate import CatalogScorer
from adt_b200.lambdas import get_lambdas
cfg = synth.CONFIGS["C2"]
args = types.SimpleNamespace(device="cuda", num_heads=cfg["nh"], maxlen=cfg["L"], num_layers=cfg["nl"], hidden_units=cfg["H"], dropout=cfg["p"])
m = SASRecADT(1, cfg["items"], args).cuda().train()
l1, l2 = get_lambdas("beauty")
tr = FusedTrainer(m, l1, l2, weight_decay=1e-4, precision="bf16")
b = synth.make_batch(np.random.default_rng(0), cfg)
for _ in range(3):
    tr.step(*b)
m.eval()
seq, _, ip, ix = synth.make_eval_batch(np.random.default_rng(1), cfg, 512)
CatalogScorer(m, K=10).topk(seq, ip, ix)
torch.cuda.synchronize()
buf = (ctypes.c_longlong * 64)()
L.lib().adt_debug_read(buf, 64)
v = list(buf)
names = ["issue loads + LN1", "weights wait + sync", "q/k/v projections", "sync", "attention (all heads)", "out-proj", "independence head", "LN2 + FFN", "mask + store"]
tot = v[57] - v[48]
for i, n in enumerate(names):
    print("%-26s %7d cycles" % (n, v[49 + i] - v[48 + i]))
print("total %d cycles = %.1f us at 1.965 GHz" % (tot, tot / 1965.0))
