"""Bert4Rec-ADT vocabulary head + cross entropy, forward + backward: the fused tcgen05 head (ops.linear_cross_entropy, no [R, V] logits)
against the materialising path fused_loss runs below FUSED_HEAD_MIN_VOCAB (ops.linear on adt_gemm_tc + MaskedCE).  Prints one JSON line.

  python tools/bert_head_bench.py [--iters 10] [--skip-step]

- C3 shape (H 256, R from a real ClozeSampler batch: B 256, L 200, mask_prob 0.2) and V 262,244: both paths, alternated in one run,
  median ms and peak memory of each, and the loss / gradient agreement of the two.
- V 1,000,100: the fused head only; the materialising path's memory is reported as computed from the shapes (3 fp32 [R, V] tensors
  + their bf16 copy live in its backward), not run.
- A C3-shaped training step (B 256, 2 blocks, FlatOptimizer) with 1,000,000 items: ms/step and peak memory.
The tied table of the 1M shapes (1 GB fp32, 512 MB bf16) does not fit the 126 MB L2.  The GPU name and power limit are read in the
same run.
"""
import argparse
import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:       # the name from torch still identifies the card
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def cloze_rows(I, B=256, L=200, mask_prob=0.2, seed=23):
    """number of labelled rows of a real ClozeSampler batch at the C3 shape"""
    from adt_b200.sampler import ClozeSampler
    rng = np.random.default_rng(seed)
    n_users = 512
    hist = {u: [int(x) for x in rng.integers(1, I + 1, size=int(np.clip(rng.geometric(1.0 / 144) + 2, 3, 400)))] for u in range(1, n_users + 1)}
    cs = ClozeSampler(hist, n_users, I, L, mask_prob=mask_prob, dupe_factor=2, prop_sliding_window=0.5, device="cuda", seed=seed)
    idx = torch.from_numpy(rng.permutation(len(cs))[:B]).cuda()
    _, _, lab = cs.batch(idx, epoch=1)
    return int((lab != 0).sum())


def head_inputs(R, V, H, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    h = torch.randn(R, H, device="cuda", generator=g).requires_grad_(True)
    W = (torch.randn(V, H, device="cuda", generator=g) * 0.05).requires_grad_(True)
    b = (torch.randn(V, device="cuda", generator=g) * 0.1).requires_grad_(True)
    lab = torch.randint(1, V, (R,), device="cuda", generator=g, dtype=torch.int32)
    return h, W, b, lab


def run_path(path, h, W, b, lab):
    from adt_b200 import ops
    from adt_b200.bert4rec import MaskedCE
    for t in (h, W, b):
        t.grad = None
    if path == "fused":
        loss = ops.linear_cross_entropy(h, W, b, lab)
    else:
        loss = MaskedCE.apply(ops.linear(h, W, b, 0, 1.0, 1), lab)
    loss.backward()
    return loss.detach()


def timed(path, inp):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_path(path, *inp)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def peak(path, inp):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    run_path(path, *inp)
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated() - base) / 2 ** 30


def agreement(inp):
    out = {}
    res = {}
    for p in ("materialising", "fused"):
        loss = run_path(p, *inp)
        res[p] = (float(loss), [t.grad.detach().clone() for t in inp[:3]])
    (l0, g0), (l1, g1) = res["materialising"], res["fused"]
    out["loss_rel_diff"] = abs(l1 - l0) / abs(l0)
    for name, a, r in zip(("dh", "dW", "db"), g1, g0):
        a, r = a.double().flatten(), r.double().flatten()
        out[name + "_max_diff_over_max"] = float((a - r).abs().max() / r.abs().max())
        out[name + "_cosine"] = float(a @ r / (a.norm() * r.norm()))
    return out


def compare(R, V, H, iters):
    inp = head_inputs(R, V, H)
    for p in ("materialising", "fused"):      # warm-up: modules, tensor maps, allocator pools
        run_path(p, *inp)
    t = {"materialising": [], "fused": []}
    for _ in range(iters):
        for p in ("materialising", "fused"):
            t[p].append(timed(p, inp))
    row = {"R": R, "V": V, "H": H}
    for p in t:
        row[p + "_ms"] = float(np.median(t[p]))
        row[p + "_peak_GiB"] = peak(p, inp)
    row["speedup"] = row["materialising_ms"] / row["fused_ms"]
    row["agreement"] = agreement(inp)
    del inp
    torch.cuda.empty_cache()
    return row


def fused_only(R, V, H, iters):
    from adt_b200 import ops
    inp = head_inputs(R, V, H)
    run_path("fused", *inp)
    ts = [timed("fused", inp) for _ in range(iters)]
    row = {"R": R, "V": V, "H": H, "fused_ms": float(np.median(ts)), "fused_peak_GiB": peak("fused", inp),
           "fused_scratch_GiB": ops.linear_ce_scratch_bytes(R, V, H) / 2 ** 30,
           "materialising_backward_live_GiB_computed": R * V * (3 * 4 + 2) / 2 ** 30, "head_tflop": 4 * 2 * R * V * H / 1e12}
    row["fused_tflops"] = row["head_tflop"] / (row["fused_ms"] / 1e3)
    del inp
    torch.cuda.empty_cache()
    return row


def train_step(I, iters):
    """a C3-shaped training step (bench.py c3_section's model and sampler) with I items: the fused head runs (V >= FUSED_HEAD_MIN_VOCAB)"""
    from adt_b200.bert4rec import BertModel
    from adt_b200.dp import FlatOptimizer
    from adt_b200.sampler import ClozeSampler
    B, L_, H, nh, nl, inner = 256, 200, 256, 4, 2, 1024
    args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=L_, num_layers=nl, hidden_units=H, dropout=0.1, attention_dropout=0.1,
                                 inner_units=inner, type_vocab_size=2)
    torch.manual_seed(0)
    m = BertModel(100, I, args).cuda().train()
    m.precision = 1
    rng = np.random.default_rng(23)
    n_users = 512
    hist = {u: [int(x) for x in rng.integers(1, I + 1, size=int(np.clip(rng.geometric(1.0 / 144) + 2, 3, 400)))] for u in range(1, n_users + 1)}
    cs = ClozeSampler(hist, n_users, I, L_, mask_prob=0.2, dupe_factor=2, prop_sliding_window=0.5, device="cuda", seed=23)
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
        return loss.detach()
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        loss = step()
    e1.record()
    e1.synchronize()
    out = {"items": I, "fused_head": m._fused_head(1), "ms_per_step": e0.elapsed_time(e1) / iters, "steps": iters,
           "peak_GiB": torch.cuda.max_memory_allocated() / 2 ** 30, "loss": loss.item()}
    del m, opt, cs
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--skip-step", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bert_head_bench.py measures on the GPU: no CUDA device")
    import adt_b200  # noqa: F401
    H = 256
    R = cloze_rows(26744)
    out = {"bench": "bert_head", **gpu_info(), "iters": a.iters, "c3_R": R}
    out["c3"] = compare(R, 26844, H, a.iters)
    out["v262k"] = compare(R, 262244, H, a.iters)
    out["v1m"] = fused_only(R, 1000100, H, a.iters)
    if not a.skip_step:
        out["train_step_1m"] = train_step(1000000, 5)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
