"""A/B of the sequence-resident evaluation encoder against the three-kernel row-tile forward on the C2 shape (run twice, with
ADT_SEQ_FUSED=0 and =1; tests/test_round2_gpu.py compares the two JSON lines), and -- with a hidden size >= 128 -- of the hoisted tcgen05
weight gradients against the in-kernel ones (ADT_WGRAD_HOIST=1 / 0).   python tools/seq_ab.py [nh] [L] [hidden]"""
import json, os, sys, types
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import numpy as np, torch
from adt_b200 import synth
from adt_b200.model import SASRecADT
from adt_b200.trainer import FusedTrainer
from adt_b200.evaluate import CatalogScorer

nh = int(sys.argv[1]) if len(sys.argv) > 1 else 2
Lq = int(sys.argv[2]) if len(sys.argv) > 2 else 50
Hd = int(sys.argv[3]) if len(sys.argv) > 3 else 64
cfg = dict(synth.CONFIGS["C2"], nh=nh, L=Lq, B=64, H=Hd)
torch.manual_seed(0)
args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=Lq, num_layers=2, hidden_units=Hd, dropout=0.5)
m = SASRecADT(1, cfg["items"], args)
for _, prm in m.named_parameters():
    if prm.dim() >= 2:
        torch.nn.init.xavier_normal_(prm.data)
g = torch.Generator().manual_seed(1)
for _, prm in m.named_parameters():
    if prm.dim() == 1:
        prm.data.add_(0.05 * torch.randn(prm.shape, generator=g))
m = m.cuda().train()
tr = FusedTrainer(m, [0.0124, 0.122], [0.0001, 0.05], weight_decay=1e-4, seed=5, precision="bf16", use_graph=False)
rng = np.random.default_rng(3)
out = {"fused": os.environ.get("ADT_SEQ_FUSED", "1"), "loss": [], "gnorm": [], "gsum": []}
for k in range(3):
    tr.step(*synth.make_batch(rng, cfg))
    out["loss"].append(tr.loss()); out["gnorm"].append(tr.grad_norm())
    out["gsum"].append(float(m.engine.gflat.double().abs().sum()))
    if k == 0:
        out["gnorms"] = {n: float(m.engine.grad_view(n).double().norm()) for n, _ in m.engine.order}
m.eval()
seq, ans, ip, ix = synth.make_eval_batch(rng, cfg, 100)
s, ids = CatalogScorer(m, K=10).topk(seq, ip, ix)
out["ids"] = ids.cpu().numpy().tolist(); out["scores"] = s.cpu().numpy().round(5).tolist()
out["psum"] = float(m.engine.pflat.double().abs().sum())
print(json.dumps(out))
