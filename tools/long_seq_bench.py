"""Sequences longer than 256 positions (fused tcgen05 flash attention, flash_tc.cu).  Prints one JSON line.

  python tools/long_seq_bench.py [--iters 10] [--skip-steps] [--skip-profile]

- Flash kernels alone (adt_attention_fwd / _bwd at L > 256, causal mask, no dropout): ms and TFLOP/s against the algorithmic count
  (forward 4 B nh L^2 hd halved for the causal mask, backward 2.5x the forward; recomputation not counted) and the share of the
  2,250 TFLOP/s dense bf16 data-sheet rate.  Inputs: q / k / v / dctx of B L H fp32 each (up to 134 MB at B L = 131,072, H 256).
- The flash entry against the batched tcgen05 path at L 128 and 256 on the same inputs (informational).
- Training steps: SASRec-ADT FusedTrainer (CUDA-graph replay) at (B, L) = (256, 512), (128, 1024), (64, 2048) for H 64 / nh 2 (row-tile
  block kernels) and H 256 / nh 2 (tcgen05 block path); a C3-shaped Bert4Rec fused_loss + FlatOptimizer step at L 512 and 1024.
  ms/step, sequences/s, peak memory; the share of the step spent in the flash kernels from torch.profiler in a separate eager run.
The GPU name, power limit and max SM clock are read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

PEAK_BF16 = 2250e12


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=30).stdout.strip().splitlines()[0]
    name, power, clk = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def timed(fn, iters):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def core(B, L, H, nh, iters, flash_entry=False):
    """ms of one forward and one backward of the attention core (causal) through the C ABI"""
    from adt_b200 import _lib as L_
    lib = L_.lib()
    lib.adt_attention_scratch_bytes.restype = ctypes.c_int64
    g = torch.Generator(device="cuda").manual_seed(0)
    q, k, v, dctx = (torch.randn(B * L, H, device="cuda", generator=g) * 0.3 for _ in range(4))
    ctx, dq, dk, dv = (torch.empty_like(q) for _ in range(4))
    lse = torch.empty(B, nh, L, device="cuda")
    n = lib.adt_attention_scratch_bytes(B, max(L, 257) if flash_entry else L, H, nh, 1)
    ws = torch.empty(max(n, 1), dtype=torch.uint8, device="cuda")
    a = L_.fill(L_.adt_attention_args(), q=q, k=k, v=v, ctx=ctx, lse=lse, dctx=dctx, dq=dq, dk=dk, dv=dv, B=B, L=L, H=H, nh=nh, mask_mode=0,
                training=1, drop=L_.adt_dropout(), precision=1, tc_scratch=ws if n else None)
    fwd = lib.adt_attention_flash_fwd if flash_entry else lib.adt_attention_fwd
    bwd = lib.adt_attention_flash_bwd if flash_entry else lib.adt_attention_bwd
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    L_.check(fwd(ctypes.byref(a), st), "fwd")
    L_.check(bwd(ctypes.byref(a), st), "bwd")
    tf = timed(lambda: fwd(ctypes.byref(a), st), iters)
    tb = timed(lambda: bwd(ctypes.byref(a), st), iters)
    flops_f = 4.0 * B * nh * L * L * (H // nh) / 2
    out = {"B": B, "L": L, "H": H, "nh": nh, "fwd_ms": tf, "bwd_ms": tb, "fwd_TFLOPs": flops_f / tf / 1e9, "bwd_TFLOPs": 2.5 * flops_f / tb / 1e9}
    out["fwd_share_of_bf16_peak"] = out["fwd_TFLOPs"] * 1e12 / PEAK_BF16
    out["bwd_share_of_bf16_peak"] = out["bwd_TFLOPs"] * 1e12 / PEAK_BF16
    return out


def flash_share(step):
    """share of the CUDA kernel time of one eager step spent in the flash kernels (torch.profiler)"""
    from torch.profiler import ProfilerActivity, profile
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    tot = fl = 0.0
    for e in prof.key_averages():
        t = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        if e.device_type == torch.autograd.DeviceType.CUDA or "kernel" in e.key.lower() or t > 0:
            if e.key.startswith("cuda") or e.key.startswith("Memcpy") or e.key.startswith("Memset"):
                continue
            tot += t
            if "flash_" in e.key:
                fl += t
    return fl / tot if tot else None


def sasrec_step(B, L, H, nh, iters, profile_share):
    from adt_b200 import synth
    from adt_b200.lambdas import get_lambdas
    from adt_b200.model import SASRecADT
    from adt_b200.trainer import FusedTrainer
    cfg = dict(synth.CONFIGS["C2"], H=H, nh=nh, L=L, B=B, items=12101, geo=1.0 / (L / 2), lo=L // 8, add=6)
    args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=L, num_layers=2, hidden_units=H, dropout=0.5)
    torch.manual_seed(0)
    rng = np.random.default_rng(1)
    batches = [synth.make_batch(rng, cfg) for _ in range(4)]
    l1, l2 = get_lambdas("beauty")
    out = {"model": "sasrec", "B": B, "L": L, "H": H, "nh": nh}
    for graph in (True, False):
        m = SASRecADT(1, cfg["items"], args).cuda().train()
        tr = FusedTrainer(m, l1, l2, weight_decay=1e-4, seed=3, use_graph=graph, precision="bf16")
        it = {"i": 0}

        def step():
            tr.step(*batches[it["i"] % 4])
            it["i"] += 1
        if graph:
            torch.cuda.reset_peak_memory_stats()
            ms = timed(step, iters)
            out.update(ms_per_step=ms, seqs_per_s=B / ms * 1e3, peak_GiB=torch.cuda.max_memory_allocated() / 2 ** 30, loss=tr.loss())
        elif profile_share:
            out["flash_share_eager"] = flash_share(step)
        del m, tr
        torch.cuda.empty_cache()
    return out


def bert_step(L, iters, profile_share):
    from adt_b200.bert4rec import BertModel
    from adt_b200.dp import FlatOptimizer
    from adt_b200.sampler import ClozeSampler
    B, H, nh, nl, inner, I = 256 * 200 // L, 256, 4, 2, 1024, 3416
    args = types.SimpleNamespace(device="cuda", num_heads=nh, maxlen=L, num_layers=nl, hidden_units=H, dropout=0.1, attention_dropout=0.1,
                                 inner_units=inner, type_vocab_size=2)
    torch.manual_seed(0)
    m = BertModel(100, I, args).cuda().train()
    m.precision = 1
    rng = np.random.default_rng(23)
    n_users = 4 * B
    hist = {u: [int(x) for x in rng.integers(1, I + 1, size=int(np.clip(rng.geometric(2.0 / L) + 2, 3, 2 * L)))] for u in range(1, n_users + 1)}
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
    out = {"model": "bert4rec", "B": B, "L": L, "H": H, "nh": nh, "ms_per_step": ms, "seqs_per_s": B / ms * 1e3,
           "peak_GiB": torch.cuda.max_memory_allocated() / 2 ** 30}
    if profile_share:
        out["flash_share_eager"] = flash_share(step)
    del m, opt, cs
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--skip-steps", action="store_true")
    ap.add_argument("--skip-profile", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("long_seq_bench.py measures on a CUDA device; none found")
    res = {"device": gpu_info(), "kernels": [], "flash_vs_batched": [], "steps": []}
    for H, nh in ((64, 2), (256, 2)):
        for B, L in ((256, 512), (128, 1024), (64, 2048)):
            res["kernels"].append(core(B, L, H, nh, a.iters))
        for B, L in ((256, 128), (128, 256)):
            fl, bt = core(B, L, H, nh, a.iters, flash_entry=True), core(B, L, H, nh, a.iters)
            res["flash_vs_batched"].append({"B": B, "L": L, "H": H, "nh": nh, "flash_fwd_ms": fl["fwd_ms"], "flash_bwd_ms": fl["bwd_ms"],
                                            "batched_fwd_ms": bt["fwd_ms"], "batched_bwd_ms": bt["bwd_ms"]})
    if not a.skip_steps:
        for H, nh in ((64, 2), (256, 2)):
            for B, L in ((256, 512), (128, 1024), (64, 2048)):
                res["steps"].append(sasrec_step(B, L, H, nh, a.iters, not a.skip_profile))
        for L in (512, 1024):
            res["steps"].append(bert_step(L, a.iters, not a.skip_profile))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
