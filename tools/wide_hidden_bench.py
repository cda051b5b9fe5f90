"""Hidden sizes beyond 256 (tcgen05 block path with four float4 per lane in its row kernels, K-blocked catalog scorer).  Prints one
JSON line.

  python tools/wide_hidden_bench.py [--iters 10]

- SASRec-ADT FusedTrainer step (CUDA-graph replay, bf16) at the C1 shape (3,416 items, L 200, B 256, 2 blocks) with H 256 / nh 2 (the
  benched C1 model), H 384 / nh 4 and H 512 / nh 4 (head size 96 and 128: nh 2 would give head sizes above 128): ms/step, sequences/s.
- Bert4Rec-ADT C3 step (26,744 items, L 200, B 256, 2 blocks, fused_loss + FlatOptimizer, bf16) at H 256 / nh 4 / inner 1024 and
  H 512 / nh 8 / inner 2048.
- K7: CatalogScorer top-10 of 512 users over 1M items at H 256, 384 and 512 on the tensor cores: ms per call (bf16 candidate pass +
  exact re-score + re-run of flagged users), TFLOP/s of the 2 U I H scoring work and its share of the 2,250 TFLOP/s dense bf16
  data-sheet rate, and the number of users re-run on the exact kernel.  The 1M x H bf16 table (up to 1 GB) does not fit L2.
The GPU name, power limit and max SM clock are read in the same run.
"""
import argparse
import json
import os
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from long_seq_bench import PEAK_BF16, gpu_info, timed  # noqa: E402


def sasrec_step(H, nh, iters):
    from adt_b200 import synth
    from adt_b200.lambdas import get_lambdas
    from adt_b200.model import SASRecADT
    from adt_b200.trainer import FusedTrainer
    cfg = dict(synth.CONFIGS["C1"], H=H, nh=nh)
    args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=cfg["L"], num_layers=cfg["nl"], hidden_units=H, dropout=cfg["p"])
    torch.manual_seed(0)
    rng = np.random.default_rng(1)
    batches = [synth.make_batch(rng, cfg) for _ in range(4)]
    l1, l2 = get_lambdas(cfg["dataset"])
    m = SASRecADT(1, cfg["items"], args).cuda().train()
    tr = FusedTrainer(m, l1, l2, weight_decay=cfg["wd"], seed=3, use_graph=True, precision="bf16")
    it = {"i": 0}

    def step():
        tr.step(*batches[it["i"] % 4])
        it["i"] += 1
    torch.cuda.reset_peak_memory_stats()
    ms = timed(step, iters)
    out = {"model": "sasrec C1", "B": cfg["B"], "L": cfg["L"], "H": H, "nh": nh, "ms_per_step": ms, "seqs_per_s": cfg["B"] / ms * 1e3,
           "peak_GiB": torch.cuda.max_memory_allocated() / 2 ** 30, "loss": tr.loss()}
    del m, tr
    torch.cuda.empty_cache()
    return out


def bert_step(H, nh, inner, iters):
    from adt_b200.bert4rec import BertModel
    from adt_b200.dp import FlatOptimizer
    from adt_b200.sampler import ClozeSampler
    B, L, nl, I = 256, 200, 2, 26744
    args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=L, num_layers=nl, hidden_units=H, dropout=0.1, attention_dropout=0.1,
                                 inner_units=inner, type_vocab_size=2)
    torch.manual_seed(0)
    m = BertModel(100, I, args).cuda().train()
    m.precision = 1
    rng = np.random.default_rng(23)
    n_users = 4 * B
    hist = {u: [int(x) for x in rng.integers(1, I + 1, size=int(np.clip(rng.geometric(1.0 / 100) + 2, 3, 2 * L)))] for u in range(1, n_users + 1)}
    cs = ClozeSampler(hist, n_users, I, L, mask_prob=0.2, dupe_factor=2, prop_sliding_window=0.5, device="cuda", seed=23)
    opt = FlatOptimizer(m, lr=1e-3, clip=5.0)
    order = torch.from_numpy(rng.permutation(len(cs))).cuda()
    state = {"i": 0}

    def step():
        idx = order[(state["i"] * B) % (len(cs) - B):][:B]
        state["i"] += 1
        src, dec, lab = cs.batch(idx, epoch=state["i"])
        opt.zero_grad()
        loss = m.fused_loss(src, dec, lab, [0.01, 0.01], [0.001, 0.001])
        loss.backward()
        opt.step()
    torch.cuda.reset_peak_memory_stats()
    ms = timed(step, iters)
    out = {"model": "bert4rec C3", "B": B, "L": L, "H": H, "nh": nh, "inner": inner, "ms_per_step": ms, "seqs_per_s": B / ms * 1e3,
           "peak_GiB": torch.cuda.max_memory_allocated() / 2 ** 30}
    del m, opt, cs
    torch.cuda.empty_cache()
    return out


def k7(H, iters, U=512, I=1_000_000, K=10):
    from adt_b200.evaluate import CatalogScorer
    g = torch.Generator(device="cuda").manual_seed(H)
    E = torch.randn(I + 1, H, device="cuda", generator=g) * 0.1
    fake = types.SimpleNamespace(item_emb=types.SimpleNamespace(weight=E), hidden=H)
    feats = torch.randn(U, H, device="cuda", generator=g)
    sc = CatalogScorer(fake, K=K, use_tensor_cores=True)
    assert sc._uses_tc(H, 0, I + 1)
    sc.refresh_table()
    ms = timed(lambda: sc.topk_from_feats(feats), iters)
    tflops = 2.0 * U * (I + 1) * H / ms / 1e9
    out = {"U": U, "items": I, "H": H, "K": K, "ms": ms, "TFLOPs": tflops, "share_of_bf16_peak": tflops * 1e12 / PEAK_BF16,
           "fallback_users": int(sc.fallback_users)}
    del E, sc
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("wide_hidden_bench.py measures on a CUDA device; none found")
    res = {"device": gpu_info(), "sasrec": [], "bert4rec": [], "k7": []}
    for H, nh in ((256, 2), (384, 4), (512, 4)):
        res["sasrec"].append(sasrec_step(H, nh, a.iters))
    for H, nh, inner in ((256, 4, 1024), (512, 8, 2048)):
        res["bert4rec"].append(bert_step(H, nh, inner, a.iters))
    for H in (256, 384, 512):
        res["k7"].append(k7(H, a.iters))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
