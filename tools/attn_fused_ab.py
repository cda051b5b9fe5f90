"""A/B of the attention fused into the H = 64 projection kernels (ADT_ATTN_FUSED=1, the default) against the separate
attention launches (ADT_ATTN_FUSED=0) on the C2 training step of bench.py: same model, batches, trainer settings and CUDA graph, L2
flushed before every timed step as bench.py does.  The switch is read once per process, so run the tool in alternating processes:

    for i in 1 2 3 4 5; do ADT_ATTN_FUSED=0 python tools/attn_fused_ab.py; ADT_ATTN_FUSED=1 python tools/attn_fused_ab.py; done

Prints one JSON line: ms/step of the graphed step, graph kernel nodes per step, the eager per-kernel times, loss and gradient norm
of the last step, and the card's name, power limit and maximum SM clock."""
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

import bench  # noqa: E402
from adt_b200 import _lib as L, synth  # noqa: E402
from adt_b200.lambdas import get_lambdas  # noqa: E402
from adt_b200.trainer import FusedTrainer  # noqa: E402


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.splitlines()[torch.cuda.current_device()].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # noqa: BLE001
        return {"name": torch.cuda.get_device_name(), "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--kernel-steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("attn_fused_ab.py measures on a GPU; none is visible")
    cfg = synth.CONFIGS["C2"]
    cx = types.SimpleNamespace(dev=torch.device("cuda", 0), world=1, rank=0, lib=L.lib(), barrier=torch.cuda.synchronize)
    cx.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=cx.dev)   # > 126 MB L2
    model = bench.make_model(cfg, cx.dev)
    l1, l2 = get_lambdas(cfg["dataset"])
    tr = FusedTrainer(model, l1, l2, weight_decay=cfg["wd"], lr=1e-3, betas=(0.9, 0.98), clip=5.0, seed=23, use_graph=True, precision="bf16")
    rng = np.random.default_rng(23)
    batches = [[torch.from_numpy(a).to(cx.dev) for a in synth.make_batch(rng, cfg)] for _ in range(8)]
    for i in range(args.warmup):
        tr.step(*batches[i % len(batches)])
    torch.cuda.synchronize()
    total_ms, _, _ = bench.timed_steps(cx, tr, batches, args.steps)
    out = {"attn_fused": os.environ.get("ADT_ATTN_FUSED", "1"), "ms_per_step": total_ms / args.steps, "steps": args.steps,
           "gpu_launches_per_step": tr.kernel_nodes(), "loss": tr.loss(), "gnorm": tr.grad_norm()}
    kern = bench.kernel_breakdown(cx, tr, batches, args.kernel_steps)
    out["kernels_us"] = {k: {"avg_us": round(v["avg_us"], 2), "per_step": v["launches"] // args.kernel_steps} for k, v in sorted(kern.items())}
    out["card"] = card()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
