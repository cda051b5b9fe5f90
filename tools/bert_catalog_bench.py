#!/usr/bin/env python
"""Full-catalog top-K for Bert4Rec-ADT on one GPU -> ONE JSON line (GPU name and power limit read in the same run).

    python tools/bert_catalog_bench.py [--batches N] [--reps R]

c3       the Bert4Rec C3 shape (26,744 items, L 200, H 256, 4 heads, inner 1024, 512 users per batch, bf16 linear layers):
         GraphedScorer (encoder + head + catalog scoring with mask_bias + top-10 + metric sums, one CUDA graph per batch) against what a
         user does without it -- the same encoder and head, downstream() over the whole vocabulary, masking in torch, torch.topk --
         alternating in the same run.  The catalog is below CatalogScorer.tc_min_items, so the scorer runs the exact fp32 kernel.
k7_1m    512 users x 1,000,000 items, H 64 and 256 (the tcgen05 two-pass path + exact re-score): the whole scoring call with a per-item
         bias and without, alternating, features resident; fallback users and the ids against the exact fp32 kernel with the same bias.
Timing: CUDA events around each call, median over repetitions; catalogs of >= 1M rows do not fit the L2.  Nothing is written.
"""
import argparse
import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q}


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def eval_batch(rng, I, U, L):
    seq = np.zeros((U, L), np.int32)
    for u in range(U):
        n = int(np.clip(rng.geometric(1.0 / 144) + 2, 3, L - 1))
        seq[u, L - n - 1:L - 1] = rng.integers(1, I + 1, size=n)
    seq[:, -1] = I + 1                                  # mask token last: the history as BertModel.predict takes it
    seen = [np.unique(r[(r >= 1) & (r <= I)]) for r in seq]
    ip = np.concatenate([[0], np.cumsum([len(s) for s in seen])]).astype(np.int32)
    ix = np.concatenate(seen).astype(np.int32)
    return seq, ip, ix, rng.integers(1, I + 1, size=U).astype(np.int32)


def c3(args):
    from adt_b200.bert4rec import BertModel
    from adt_b200.evaluate import CatalogScorer, GraphedScorer
    I, L, H, nh, nl, inner, U, K = 26744, 200, 256, 4, 2, 1024, 512, 10
    torch.manual_seed(0)
    a = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=L, num_layers=nl, hidden_units=H, dropout=0.1, attention_dropout=0.1,
                              inner_units=inner, type_vocab_size=2)
    m = BertModel(100, I, a).cuda().eval()
    m.precision = 1
    with torch.no_grad():
        m.mask_bias.normal_(0.0, 0.5)
    rng = np.random.default_rng(99)
    bt = [eval_batch(rng, I, U, L) for _ in range(4)]
    dev_b = [[torch.from_numpy(x).cuda() for x in b] for b in bt]
    sc = CatalogScorer(m, K=K)
    gs = GraphedScorer(sc, U, L, max_seen=max(len(b[2]) for b in bt))
    pos = torch.arange(L, dtype=torch.int32, device="cuda").repeat(U, 1)
    sent = torch.zeros(U, L, dtype=torch.int32, device="cuda")

    @torch.no_grad()
    def today(b):      # downstream(last) -> restrict to items 1..I -> mask seen -> torch.topk
        seq, ip, ix, _ = b
        from adt_b200.blocks import DropCfg
        x, _, _ = m._encode(seq, pos, sent, DropCfg(0.0, 0, 0, False))
        logits = m.downstream(x.view(U, L, -1)[:, -1, :].contiguous())[:, 1:I + 1]
        rows = torch.repeat_interleave(torch.arange(U, device="cuda"), (ip[1:] - ip[:-1]).long(), output_size=ix.numel())
        logits.index_put_((rows, ix.long() - 1), torch.tensor(float("-inf"), device="cuda"))
        s, i = torch.topk(logits, K, dim=1)
        return s, i + 1

    state = {"k": 0}

    def run_graph():
        b = dev_b[state["k"] % 4]
        state["k"] += 1
        gs.topk(b[0], b[1], b[2], b[3])

    def run_today():
        today(dev_b[state["k"] % 4])
        state["k"] += 1
    for _ in range(3):
        run_graph()
        run_today()
    tg, tt = [], []
    for _ in range(args.reps):
        tg.append(timed(run_graph, args.batches))
        tt.append(timed(run_today, args.batches))
    same_rows, same_all, fp32_rows = 0, True, 0
    W, mb = m.item_emb.word_emb.weight[1:I + 1], m.mask_bias[1:I + 1]
    for b in dev_b:
        _, i_g = gs.topk(b[0], b[1], b[2], b[3])
        _, i_t = today(b)
        eq = (i_g.long() == i_t).all(dim=1)
        same_rows += int(eq.sum())
        same_all &= bool(eq.all())
        with torch.no_grad():     # the same features scored by a plain fp32 matmul + bias in torch: checks the scoring alone
            lg = m.final_feats(b[0]) @ W.t() + mb
            rows = torch.repeat_interleave(torch.arange(U, device="cuda"), (b[1][1:] - b[1][:-1]).long(), output_size=b[2].numel())
            lg.index_put_((rows, b[2].long() - 1), torch.tensor(float("-inf"), device="cuda"))
            fp32_rows += int((torch.topk(lg, K, dim=1)[1] + 1 == i_g.long()).all(dim=1).sum())
    gms, tms = float(np.median(tg)), float(np.median(tt))
    return {"items": I, "users_per_batch": U, "K": K, "dtype": "bf16 linear layers",
            "scoring_path": "tcgen05 + exact re-score" if gs.tc else "exact fp32 kernel with bias (score_topk_kernel; catalog below tc_min_items)",
            "graphed_scorer": {"ms_per_batch": gms, "users_per_sec": U / (gms / 1e3)},
            "downstream_mask_topk": {"ms_per_batch": tms, "users_per_sec": U / (tms / 1e3)},
            "speedup": tms / gms, "ids_equal": same_all, "rows_with_equal_ids": f"{same_rows}/{4 * U}",
            "rows_with_ids_equal_to_fp32_torch_scoring": f"{fp32_rows}/{4 * U}",
            "ids_note": "downstream() in bf16 mode scores on bf16 tensor cores, the scorer in exact fp32: rows differ where bf16 rounding "
                        "reorders near ties; the fp32 comparison scores the same features with torch in fp32 (ties may order differently)",
            "fallback_users": sc.fallback_users}


def k7_1m(args):
    from adt_b200.evaluate import Catalog, CatalogScorer
    I, U, K = 1_000_000, 512, 10
    out = {}
    for H in (64, 256):
        g = torch.Generator(device="cuda").manual_seed(5 + H)
        E = torch.randn(I, H, device="cuda", generator=g) * (2.0 / (I + H)) ** 0.5 * 30
        feats = torch.randn(U, H, device="cuda", generator=g)
        std = float((feats[:64] @ E[:4096].t()).std())
        b = torch.randn(I, device="cuda", generator=g) * std

        def holder(bias):
            return types.SimpleNamespace(scoring_catalog=lambda: Catalog(E, bias, 1, H))
        nb, wb = CatalogScorer(holder(None), K=K), CatalogScorer(holder(b), K=K)
        nb.refresh_table()
        wb.refresh_table()
        for _ in range(3):
            nb.topk_from_feats(feats)
            wb.topk_from_feats(feats)
        tn, tb = [], []
        for _ in range(args.reps):
            tn.append(timed(lambda: nb.topk_from_feats(feats), 10))
            tb.append(timed(lambda: wb.topk_from_feats(feats), 10))
        nb._fallback.zero_()
        wb._fallback.zero_()
        s_b, i_b = [t.clone() for t in wb.topk_from_feats(feats)]
        _, i_n = [t.clone() for t in nb.topk_from_feats(feats)]
        ex = CatalogScorer(holder(b), K=K, use_tensor_cores=False)
        _, i_e = ex.topk_from_feats(feats)
        exn = CatalogScorer(holder(None), K=K, use_tensor_cores=False)
        _, i_en = exn.topk_from_feats(feats)
        msn, msb = float(np.median(tn)), float(np.median(tb))
        out[f"U{U}_I1M_H{H}"] = {"ms_no_bias": msn, "ms_bias": msb, "bias_cost": msb / msn - 1.0,
                                 "ms_no_bias_all": [round(x, 4) for x in tn], "ms_bias_all": [round(x, 4) for x in tb],
                                 "fallback_users_bias": wb.fallback_users, "fallback_users_no_bias": nb.fallback_users,
                                 "ids_equal_exact_bias": bool(torch.equal(i_b, i_e)), "ids_equal_exact_no_bias": bool(torch.equal(i_n, i_en)),
                                 "path": "tcgen05 two-pass" if wb._uses_tc(H, *wb.bounds()) else "exact"}
        del E, nb, wb, ex, exn
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=20, help="calls per timed repetition")
    ap.add_argument("--reps", type=int, default=5, help="alternating repetitions per arm (median reported)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bert_catalog_bench needs a CUDA device")
    line = {"what": "Bert4Rec-ADT full-catalog top-K", **gpu_info(), "c3": c3(args), "k7_1m": k7_1m(args),
            "timing": "CUDA events, median of the alternating repetitions"}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
