#!/usr/bin/env python
"""Full-catalog top-K for STOSA-ADT on one GPU: the centred-dot-product catalog against the augmented-row path it replaces -> ONE JSON
line (GPU name, power limit and max SM clock read in the same run).

    python tools/stosa_catalog_bench.py [--batches N] [--reps R] [--train-steps S]

scoring   512 users x {12,101 (C4); 100,000; 1,000,000} items at H 64 and 1,000,000 at H 128, K 40, synthetic item tables (both
          normal(0.01, sigma): sigma 0.02 is the model's initialisation, 0.3 a trained-like spread) and encoder-like user states:
          old  = what DisenDistSAModel.full_sort_topk did before: adt_wcatalog_rows for the users and the whole catalog, and a new
                 exact-kernel CatalogScorer, on every call;
          new  = user_feats (adt_wcatalog_user) + the model's cached CatalogScorer on the centred catalog (tcgen05 from 32,768 rows);
          alternating, median of repetitions.  Also: the new path's fallback users per distribution, the same centred catalog on the
          exact kernel only (where the tcgen05 path starts to pay), and the catalog rebuild time.
trained   a C4-shaped model (12,101 items, L 100, H 64, 4 heads, 1 layer) after --train-steps fused_loss + FlatOptimizer steps on
          synthetic batches: fallback users of the tcgen05 path forced at that size (tc_min_items 0).
c4_graph  the same trained model, 512-user batches of L 100: GraphedScorer (encoder + scoring + metric sums, one CUDA graph) against the
          old full_sort_topk (encoder AND decoder, augmented rows, exact scorer built per call) + host metrics; and the encoder part alone.
Timing: CUDA events around each call, median over repetitions.  Catalogs of 1M rows (512 MB at H 64) do not fit the L2.  Nothing is
written.
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

U, K = 512, 40
SIGMA = {"init": 0.02, "spread": 0.3}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi name,power.limit,clocks.max.sm": q}


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def model(I, H, sigma=None, L=8, nh=2, seed=0):
    from adt_b200.stosa import DisenDistSAModel
    a = types.SimpleNamespace(item_size=I, num_users=16, maxlen=L, hidden_units=H, num_heads=nh, num_layers=1, dropout=0.3,
                              attention_dropout=0.3, initializer_range=0.02, pvn_weight=0.005)
    torch.manual_seed(seed)
    m = DisenDistSAModel(a).cuda().eval()
    if sigma is not None:
        g = torch.Generator(device="cuda").manual_seed(seed + I + H)
        with torch.no_grad():
            for t in (m.item_mean_embeddings.weight, m.item_cov_embeddings.weight):
                t.normal_(0.01, sigma, generator=g)
    return m


def users(H, seed=1):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.nn.functional.elu(torch.randn(U, H, device="cuda", generator=g)),
            torch.nn.functional.elu(torch.randn(U, H, device="cuda", generator=g)) + 1.0)


def seen_csr(rng, I, n=10):
    seen = [np.unique(rng.integers(1, I, size=n)) for _ in range(U)]
    ip = np.concatenate([[0], np.cumsum([len(s) for s in seen])]).astype(np.int32)
    return torch.from_numpy(ip).cuda(), torch.from_numpy(np.concatenate(seen).astype(np.int32)).cuda()


def old_topk_from_states(m, um, uc, ip, ix):
    """DisenDistSAModel.full_sort_topk before the centred catalog, after the encoder: augmented rows rebuilt and a fresh exact scorer"""
    from adt_b200.evaluate import CatalogScorer
    u = m._rows(um, uc, 1)
    cat = m._rows(m.item_mean_embeddings.weight, m.item_cov_embeddings.weight, 0)
    holder = types.SimpleNamespace(item_emb=types.SimpleNamespace(weight=cat))
    return CatalogScorer(holder, K=K, use_tensor_cores=False).topk_from_feats(u, ip, ix)[1]


@torch.no_grad()
def old_last_states(m, seq):
    """the evaluation forward before: _body with the decoder"""
    mm, c, _, _, _, (B, Lq) = m._body(seq, seq)
    H = m.hidden_units
    return mm.view(B, Lq, H)[:, -1, :].contiguous(), c.view(B, Lq, H)[:, -1, :].contiguous()


def scoring(args):
    from adt_b200.evaluate import CatalogScorer
    out = {}
    for I, H in ((12_101, 64), (100_000, 64), (1_000_000, 64), (1_000_000, 128)):
        for dname, sigma in SIGMA.items():
            m = model(I, H, sigma)
            um, uc = users(H)
            ip, ix = seen_csr(np.random.default_rng(I + H), I)
            new = CatalogScorer(m, K=K)
            tc = new._uses_tc(2 * H, *new.bounds())
            r = {"path": "tcgen05 + exact re-score" if tc else "exact fp32 kernel"}
            run_new = lambda: new.topk_from_feats(m.user_feats(um, uc), ip, ix)
            for _ in range(3):
                run_new()
            if new._fallback is not None:
                new._fallback.zero_()
            i_new = run_new()[1].clone()
            r["fallback_users"] = new.fallback_users
            old_ok = 2 * H + 4 <= 256
            if old_ok:
                run_old = lambda: old_topk_from_states(m, um, uc, ip, ix)
                for _ in range(2):
                    run_old()
                i_old = run_old()
                r["rows_ids_equal_old"] = f"{int((i_old == i_new).all(dim=1).sum())}/{U}"
            if dname == "init" or H == 128:     # timing once per shape (the distribution only moves the fallback count)
                ex = CatalogScorer(m, K=K, use_tensor_cores=False)      # the same centred catalog on the exact fp32 kernel only
                run_ex = lambda: ex.topk_from_feats(m.user_feats(um, uc), ip, ix)
                run_ex()
                tn, to, te = [], [], []
                for _ in range(args.reps):
                    tn.append(timed(run_new, args.batches))
                    te.append(timed(run_ex, args.batches))
                    if old_ok:
                        to.append(timed(run_old, max(1, args.batches // 4)))
                r["new_ms"] = float(np.median(tn))
                r["new_ms_all"] = [round(x, 4) for x in tn]
                r["new_exact_kernel_only_ms"] = float(np.median(te))
                if old_ok:
                    r["old_ms"] = float(np.median(to))
                    r["old_ms_all"] = [round(x, 4) for x in to]
                    r["speedup"] = r["old_ms"] / r["new_ms"]
                else:
                    r["old_ms"] = "refused: 2H+4 > 256 (ADT_E_SHAPE)"

                def rebuild():
                    m._wcat_key = None
                    m.scoring_catalog()
                r["catalog_rebuild_ms"] = float(np.median([timed(rebuild, 5) for _ in range(3)]))
            out[f"I{I}_H{H}_{dname}"] = r
            del m, new
            torch.cuda.empty_cache()
    return out


def c4_batch(rng, I, B, L):
    seq = np.zeros((B, L), np.int64)
    for b in range(B):
        n = int(np.clip(rng.geometric(1.0 / 9) + 3, 3, L))
        seq[b, L - n:] = rng.integers(1, I, size=n)
    return seq


def trained_c4(args):
    from adt_b200.dp import FlatOptimizer
    I, L, H = 12_101, 100, 64
    m = model(I, H, None, L=L, nh=4)
    opt = FlatOptimizer(m, lr=1e-3)
    m.train()
    rng = np.random.default_rng(11)
    losses = []
    for s in range(args.train_steps):
        seq = c4_batch(rng, I, 256, L + 1)
        inp, pos = seq[:, :-1], seq[:, 1:]
        dec = np.zeros_like(inp)
        dec[:, 1:] = inp[:, :-1]
        neg = np.where(pos > 0, rng.integers(1, I, size=pos.shape), 0)
        opt.zero_grad()
        loss = m.fused_loss(inp, dec, pos, neg, [0.0021], [0.0009])[0]
        loss.backward()
        opt.step()
        if s % 50 == 0 or s == args.train_steps - 1:
            losses.append(round(float(loss), 5))
    m.eval()
    return m, losses


def fallback_trained(m):
    from adt_b200.evaluate import CatalogScorer
    rng = np.random.default_rng(12)
    seq = torch.from_numpy(c4_batch(rng, 12_101, U, 100)).cuda()
    ip, ix = seen_csr(rng, 12_101)
    sc = CatalogScorer(m, K=K, tc_min_items=0)
    assert sc._uses_tc(128, *sc.bounds())
    _, i_tc = sc.topk(seq, ip, ix)
    _, i_ex = CatalogScorer(m, K=K, use_tensor_cores=False).topk(seq, ip, ix)
    Em, Ec = m.item_mean_embeddings.weight, m.item_cov_embeddings.weight
    return {"fallback_users": sc.fallback_users, "of_users": U, "ids_equal_exact": bool(torch.equal(i_tc, i_ex)),
            "item_mean_std": float(Em.std()), "item_cov_std": float(Ec.std())}


def c4_graph(args, m):
    from adt_b200.evaluate import CatalogScorer, GraphedScorer, hit_ndcg_mrr
    I, L = 12_101, 100
    rng = np.random.default_rng(13)
    bt = []
    for _ in range(4):
        seq = c4_batch(rng, I, U, L).astype(np.int32)
        seen = [np.unique(r[r > 0]) for r in seq]
        ip = np.concatenate([[0], np.cumsum([len(s) for s in seen])]).astype(np.int32)
        bt.append((seq, ip, np.concatenate(seen).astype(np.int32), rng.integers(1, I, size=U).astype(np.int32)))
    dev_b = [[torch.from_numpy(x).cuda() for x in b] for b in bt]
    gs = GraphedScorer(CatalogScorer(m, K=K), U, L, max_seen=max(len(b[2]) for b in bt))
    st = {"k": 0}

    def run_graph():
        b = dev_b[st["k"] % 4]
        st["k"] += 1
        gs.topk(b[0], b[1], b[2], b[3])

    def run_old():      # the old full_sort_topk + the host metrics a caller computes from its ids
        b, hb = dev_b[st["k"] % 4], bt[st["k"] % 4]
        st["k"] += 1
        ids = old_topk_from_states(m, *old_last_states(m, b[0]), b[1], b[2])
        hit_ndcg_mrr(hb[3], ids, ks=(5, 10))

    def enc_new():
        m._last_states(dev_b[st["k"] % 4][0])

    def enc_old():
        old_last_states(m, dev_b[st["k"] % 4][0])
    for _ in range(3):
        run_graph(); run_old(); enc_new(); enc_old()
    tg, to, ten, teo = [], [], [], []
    for _ in range(args.reps):
        tg.append(timed(run_graph, args.batches))
        to.append(timed(run_old, args.batches))
        ten.append(timed(enc_new, args.batches))
        teo.append(timed(enc_old, args.batches))
    gs.metrics()
    rows_eq = 0
    for b, hb in zip(dev_b, bt):
        i_g = gs.topk(b[0], b[1], b[2], b[3])[1].clone()
        i_o = old_topk_from_states(m, *old_last_states(m, b[0]), b[1], b[2])
        rows_eq += int((i_g == i_o).all(dim=1).sum())
    g, o = float(np.median(tg)), float(np.median(to))
    return {"items": I, "L": L, "users_per_batch": U, "K": K, "graph_path": "tcgen05" if gs.tc else "exact fp32 kernel",
            "graphed_scorer_ms_per_batch": g, "old_full_sort_topk_plus_host_metrics_ms_per_batch": o, "speedup": o / g,
            "graphed_all": [round(x, 4) for x in tg], "old_all": [round(x, 4) for x in to],
            "encoder_only_last_states_ms": float(np.median(ten)), "encoder_plus_decoder_old_ms": float(np.median(teo)),
            "rows_ids_equal_old": f"{rows_eq}/{4 * U}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=20, help="calls per timed repetition")
    ap.add_argument("--reps", type=int, default=5, help="alternating repetitions per arm (median reported)")
    ap.add_argument("--train-steps", type=int, default=300, help="fused_loss steps of the C4-shaped model before the trained measurements")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stosa_catalog_bench needs a CUDA device")
    line = {"what": "STOSA-ADT full-catalog top-K", **gpu_info(), "scoring": scoring(args)}
    m, losses = trained_c4(args)
    line["trained_c4"] = {"train_steps": args.train_steps, "loss_every_50": losses, **fallback_trained(m)}
    line["c4_graph"] = c4_graph(args, m)
    line["timing"] = "CUDA events, median of the alternating repetitions"
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
