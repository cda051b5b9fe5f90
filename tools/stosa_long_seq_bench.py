"""STOSA-ADT at sequences the resident Wasserstein attention kernels cannot hold (tcgen05 flash kernels, wflash_tc.cu).  Prints JSON lines.

  python tools/stosa_long_seq_bench.py [--iters 10] [--skip-steps]

- Flash kernels alone (adt_wattention_flash_fwd / _bwd incl. their prep launches, dropout 0.5, random left padding) at H 64 with nh 1 / 2 / 4
  and H 128 with nh 2, (B, L) = (256, 512), (128, 1024), (64, 2048): ms and TFLOP/s against the algorithmic count below, and the share of
  the 2,250 TFLOP/s dense bf16 data-sheet rate.  Count per (sequence, head): forward 2 L^2 (2 hd) for the score product + 2 x 2 L^2 hd
  for the two context products; backward 2 x 2 L^2 hd (dP_m, dP_c) + 2 x 2 L^2 hd (dmv, dcv) + 2 x 2 L^2 (2 hd) (query and key side);
  both halved for the causal mask; recomputation of S in the backward not counted.
- A training step (fused_loss + backward + FlatOptimizer, 1 block, dropout 0.5, precision 1) at the same shapes: ms/step, seqs/s, peak GiB.
- At (L 200, hd 16), where both paths serve: the resident fp32 kernels against the flash kernels, forward and backward (informational).
- The C4 step of tools/bench_variants.py (L 100, hd 16, precision 0: the resident path).
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
SHAPES = [(256, 512), (128, 1024), (64, 2048)]
HEADS = [(64, 1), (64, 2), (64, 4), (128, 2)]


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=30).stdout.strip().splitlines()[0]
    name, power, clk = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def timed(fn, iters, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def flops(B, L, H, nh):
    hd = H // nh
    per = L * L * B * nh / 2                                    # causal half of the score matrix
    return per * (2 * 2 * hd + 2 * 2 * hd), per * (4 * 2 * hd + 2 * 2 * 2 * hd)


def core(B, L, H, nh, iters, flash=True):
    """ms of one forward and one backward of the attention core through the C ABI"""
    from adt_b200 import _lib as Lb
    from adt_b200.blocks import DropCfg
    from adt_b200.ops import _st
    lib = Lb.lib()
    lib.adt_wattention_scratch_bytes.restype = ctypes.c_int64
    g = torch.Generator(device="cuda").manual_seed(0)
    mq, mk, mv, dm, dc = (0.01 + 0.3 * torch.randn(B * L, H, device="cuda", generator=g) for _ in range(5))
    cq, ck, cv = (torch.nn.functional.elu(0.3 * torch.randn(B * L, H, device="cuda", generator=g)) + 1 for _ in range(3))
    ids = torch.zeros(B, L, dtype=torch.int32)
    rng = np.random.default_rng(0)
    for b in range(B):
        n = int(rng.integers(L // 4, L + 1))
        ids[b, L - n:] = torch.from_numpy(rng.integers(1, 1000, size=n).astype(np.int32))
    ids = ids.cuda()
    mctx, cctx = torch.empty_like(mq), torch.empty_like(mq)
    stat = torch.empty(B, nh, L, 2, device="cuda")
    grads = [torch.empty_like(mq) for _ in range(6)]
    drop = DropCfg(0.5, 1, 1, True).next("attn", nh, L, H)
    ws = torch.empty(max(lib.adt_wattention_scratch_bytes(B, L, H, nh, 1), 1), dtype=torch.uint8, device="cuda") if flash else None
    fa = Lb.fill(Lb.adt_wattention_args(), mq=mq, cq=cq, mk=mk, ck=ck, mv=mv, cv=cv, mctx=mctx, cctx=cctx, lse=stat, key_ids=ids, B=B, L=L,
                 H=H, nh=nh, drop=drop, tc_scratch=ws)
    ba = Lb.fill(Lb.adt_wattention_args(), mq=mq, cq=cq, mk=mk, ck=ck, mv=mv, cv=cv, lse=stat, key_ids=ids, dmctx=dm, dcctx=dc, dmq=grads[0],
                 dcq=grads[1], dmk=grads[2], dck=grads[3], dmv=grads[4], dcv=grads[5], B=B, L=L, H=H, nh=nh, drop=drop, tc_scratch=ws,
                 mctx_in=mctx, cctx_in=cctx)
    st = _st(mq.device)
    fwd = lib.adt_wattention_flash_fwd if flash else lib.adt_wattention_fwd
    bwd = lib.adt_wattention_flash_bwd if flash else lib.adt_wattention_bwd
    Lb.check(fwd(ctypes.byref(fa), st), "fwd")
    Lb.check(bwd(ctypes.byref(ba), st), "bwd")
    return timed(lambda: fwd(ctypes.byref(fa), st), iters), timed(lambda: bwd(ctypes.byref(ba), st), iters)


def batch(rng, B, L, I):
    seq = np.zeros((B, L), np.int64)
    for b in range(B):
        n = int(rng.integers(L // 4, L + 1))
        seq[b, L - n:] = rng.integers(1, I + 1, size=n)
    dec = np.zeros_like(seq)
    dec[:, 1:] = seq[:, :-1]
    pos = np.roll(seq, -1, axis=1) * (seq > 0)
    neg = rng.integers(1, I + 1, size=(B, L)) * (pos > 0)
    return seq, dec, pos, neg


def train_step(B, L, H, nh, iters, precision=1, p=0.5, I=12101):
    from adt_b200.dp import FlatOptimizer
    from adt_b200.stosa import DisenDistSAModel
    args = types.SimpleNamespace(item_size=I + 2, num_users=B, maxlen=L, hidden_units=H, num_heads=nh, num_layers=1, dropout=p,
                                 attention_dropout=p, initializer_range=0.02, pvn_weight=0.005)
    torch.manual_seed(0)
    m = DisenDistSAModel(args).cuda().train()
    m.precision = precision
    opt = FlatOptimizer(m, lr=1e-3)
    seq, dec, pos, neg = (torch.from_numpy(a).cuda() for a in batch(np.random.default_rng(1), B, L, I))

    def step():
        opt.zero_grad()
        loss = m.fused_loss(seq, dec, pos, neg, [0.0021], [0.0009])[0]
        loss.backward()
        opt.step()
    torch.cuda.reset_peak_memory_stats()
    ms = timed(step, iters)
    return {"ms_per_step": ms, "seqs_per_sec": B / ms * 1e3, "peak_gib": torch.cuda.max_memory_allocated() / 2 ** 30}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--skip-steps", action="store_true")
    a = ap.parse_args()
    print(json.dumps({"what": "device", **gpu_info()}), flush=True)
    for B, L in SHAPES:
        for H, nh in HEADS:
            fms, bms = core(B, L, H, nh, a.iters)
            ff, bf = flops(B, L, H, nh)
            print(json.dumps({"what": "wflash_core", "B": B, "L": L, "H": H, "nh": nh, "hd": H // nh, "fwd_ms": fms, "bwd_ms": bms,
                              "fwd_tflops": ff / fms * 1e-9, "bwd_tflops": bf / bms * 1e-9, "fwd_share_of_2250": ff / fms * 1e3 / PEAK_BF16,
                              "bwd_share_of_2250": bf / bms * 1e3 / PEAK_BF16}), flush=True)
    B, L, H, nh = 256, 200, 64, 4
    r = dict(zip(("resident_fwd_ms", "resident_bwd_ms"), core(B, L, H, nh, a.iters, flash=False)))
    r.update(zip(("flash_fwd_ms", "flash_bwd_ms"), core(B, L, H, nh, a.iters)))
    print(json.dumps({"what": "both_paths", "B": B, "L": L, "H": H, "nh": nh, **r}), flush=True)
    if a.skip_steps:
        return
    for B, L in SHAPES:
        for H, nh in HEADS:
            print(json.dumps({"what": "train_step", "B": B, "L": L, "H": H, "nh": nh, "precision": 1, "dropout": 0.5,
                              **train_step(B, L, H, nh, a.iters)}), flush=True)


if __name__ == "__main__":
    main()
