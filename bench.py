#!/usr/bin/env python
"""bench.py -- headline benchmark of the ADT hot path (BASELINE.json: SASRec train seqs/sec + full-catalog eval
users/sec) on N B200s of one node.

    python bench.py [--gpus N --steps K --warmup W]                 our CUDA path
    python bench.py --impl reference [...]                           the UNMODIFIED reference on the host CPU cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   (N > 1, one rank per GPU)

A "step" = one SASRec-ADT optimisation step (forward, fused losses, backward, sort+segmented embedding
backward, clip + Adam) over one synthetic batch of the C2 shape (configs[1]: ~12k items, maxlen 50, hidden 64,
2 heads, 2 blocks, 256 sequences per GPU, dropout 0.5).  Prints ONE JSON line on rank 0:

  value / e2e / roofline / cpu_baseline      the training half of the metric (C2)
  eval {value, e2e, roofline, cpu_baseline}  the evaluation half (full-catalog top-10 of 512 users per batch, C2)
  fp32 {...}                                 the step with fp32 FFMA GEMM cores (the reference's precision), device + e2e
  c1 {...}                                   configs[0]'s shape (ml-1m: L 200, H 256) through the same trainer
  c3 {...}                                   configs[2]: Bert4Rec-ADT cloze training step (ml-20m shape), linear layers on tcgen05
  c5 {...}                                   catalog scoring at 1M items (H 64 / 256): tensor-pipe roofline
  reference_gpu_eager {...}                  the unmodified reference in PyTorch eager on the same B200 (the kernel bar)
  evolution {...}                            evolution.py's population evaluation on the supernet, candidates dealt to the ranks
  selfcheck {...}                            N > 1: data-parallel and item-sharded results against the 1-GPU fixture
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from adt_b200 import synth  # noqa: E402
from adt_b200.lambdas import get_lambdas  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2")
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16"],
                    help="GEMM cores of the block kernels: fp32 FFMA (reference precision) or bf16 tensor cores with fp32 accumulate")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget-s", type=float, default=12.0)
    ap.add_argument("--skip", default="", help="comma list of optional sections to skip: c1,c5,refgpu,fp32,selfcheck,eval")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the training step of the timed loop behind `value` as it computes from the seeded initial weights, on "
                         "the batch and dropout stream of that loop's last step (loss, gradient norm, clipped gradients), as "
                         "DIR/<name>.npy, to compare two builds output for output")
    return ap.parse_args()


def dump_outputs(path, arrays, limit=64 << 20, min_rows=4096):
    """{name: array} -> path/<name>.npy, float64 arrays as float64 and everything else as float32.  When the arrays come to more
    than `limit` bytes, every array of more than `min_rows` rows keeps a fixed, seeded sample of its rows, in row order, sized so
    that the sampled arrays take at most half the limit; path/<name>.rows.npy lists the rows kept."""
    arrays = {k: np.asarray(v, dtype=np.float64 if np.asarray(v).dtype == np.float64 else np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        if total > limit and a.ndim and len(a) > min_rows:
            rows = np.sort(np.random.default_rng(0).choice(len(a), int(len(a) * (limit // 2) / total), replace=False))
            np.save(os.path.join(path, f"{k}.rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(path, f"{k}.npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": float(d["hbm_gbs"]), "bf16": float(d.get("bf16_tflops", 1590.0)), "bf16_sustained": float(d.get("bf16_tflops_sustained", 1400.0)),
                "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "bf16": 1590.0, "bf16_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.samples, self.stop, self.index = [], False, index
        self.th = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.th.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 2 + i and s[2 + i].lower().startswith("active") for s in self.samples)]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons}


def init_state_dict(cfg, seed=23):
    """random-init weights of the architecture, the way sasrec/main.py:93-99 does it (xavier_normal_ on >=2-D)."""
    import types
    from adt_b200.model import SASRecADT
    torch.manual_seed(seed)
    args = types.SimpleNamespace(device="cpu", num_heads=cfg["nh"], maxlen=cfg["L"], num_layers=cfg["nl"], hidden_units=cfg["H"],
                                 dropout=cfg["p"])
    m = SASRecADT(1, cfg["items"], args)
    for _, prm in m.named_parameters():
        try:
            torch.nn.init.xavier_normal_(prm.data)
        except Exception:
            pass
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def workload_name(name, cfg):
    return (f"SASRec-ADT {name}: train step (items={cfg['items']}, maxlen={cfg['L']}, hidden={cfg['H']}, heads={cfg['nh']}, "
            f"blocks={cfg['nl']}, batch={cfg['B']}/GPU, dropout={cfg['p']}) + full-catalog eval (512 users/batch, top-10)")


def config_dict(args, cfg, world):
    """the SAME dict for both arms (the driver compares the arms on it)"""
    return {"workload": workload_name(args.config, cfg), "parallelism": f"dp{world}", "global_batch": world * cfg["B"],
            "l2": "flushed between timed steps (256 MB write)", "timing": "per-step CUDA events on the launch stream, max over ranks"}


# ------------------------------------------------------------------------------------------------ the reference on host cores / eager GPU
def time_reference_train(cfg, device, steps, warmup, budget_s=None):
    """the UNMODIFIED reference model (oracle/_ref, staged from /root/reference/sasrec) + the loss/clip/Adam lines of
    main.py:146-173 with torch's own dropout.  -> (seqs_per_sec, median ms_per_step, n timed steps)"""
    from oracle import ref_runner as R
    l1, l2 = get_lambdas(cfg["dataset"])
    tr = R.RefTrainer(cfg, l1, l2, device=device, state_dict=init_state_dict(cfg))
    rng = np.random.default_rng(23)
    pool = [synth.make_batch(rng, cfg) for _ in range(4)]
    sync = torch.cuda.synchronize if device != "cpu" else (lambda: None)
    ts, t_begin, i = [], time.time(), 0
    while True:
        sync()
        t0 = time.time()
        tr.step(*pool[i % len(pool)])
        sync()
        dt = time.time() - t0
        if i >= warmup:
            ts.append(dt)
        i += 1
        if len(ts) >= steps:
            break
        if budget_s is not None and time.time() - t_begin > budget_s and len(ts) >= 2:
            break
    ms = 1e3 * float(np.median(ts))
    return cfg["B"] / (ms / 1e3), ms, len(ts)


def time_reference_eval(cfg, device, batches, warmup=1, budget_s=None, U=512):
    """predict(full=True) + the masking / argpartition / argsort lines of evaluate_loader_full (utils.py:718-731)."""
    from oracle import ref_runner as R
    ev = R.RefEvaluator(cfg, device=device, state_dict=init_state_dict(cfg))
    erng = np.random.default_rng(99)
    eseq, _, eip, eix = synth.make_eval_batch(erng, cfg, U)
    sync = torch.cuda.synchronize if device != "cpu" else (lambda: None)
    ts, t_begin, i = [], time.time(), 0
    while True:
        sync()
        t0 = time.time()
        ev.topk(eseq, eip, eix, k=40)
        sync()
        dt = time.time() - t0
        if i >= warmup:
            ts.append(dt)
        i += 1
        if len(ts) >= batches:
            break
        if budget_s is not None and time.time() - t_begin > budget_s and len(ts) >= 2:
            break
    ms = 1e3 * float(np.median(ts))
    return U / (ms / 1e3), ms, len(ts)


def run_reference(args, cfg, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on all host threads, rank 0 only."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    v, ms, n = time_reference_train(cfg, "cpu", steps=args.steps, warmup=args.warmup)
    ev, ems, en = time_reference_eval(cfg, "cpu", batches=max(3, min(args.steps, 10)), warmup=1)
    sample = f"{n} full optimisation steps (after {args.warmup} warm-up) of {cfg['B']}-sequence batches, median; torch dropout, {cores} threads"
    line = {"metric": "train_seqs_per_sec", "value": v, "unit": "seqs/s", "n_gpus": args.gpus, "steps": n, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "impl": "reference", "config": config_dict(args, cfg, world),
            "cpu_baseline": {"value": v, "unit": "seqs/s", "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": v, "unit": "seqs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "eval": {"metric": "eval_users_per_sec", "value": ev, "unit": "users/s", "ms_per_batch": ems, "batches": en,
                     "what": "predict(full=True) + seen-mask + argpartition(40) + argsort, 512 users per batch (utils.py:718-731)"},
            "reference_source": "oracle/_ref (unmodified /root/reference/sasrec/{model,modules}.py) + main.py:146-173 loss/clip/Adam lines"}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ our arm: helpers
def make_model(cfg, dev):
    import types
    from adt_b200.model import SASRecADT
    margs = types.SimpleNamespace(device=dev, num_heads=cfg["nh"], maxlen=cfg["L"], num_layers=cfg["nl"], hidden_units=cfg["H"],
                                  dropout=cfg["p"])
    model = SASRecADT(1, cfg["items"], margs)
    model.load_state_dict(init_state_dict(cfg))
    return model.to(dev).train()


class Ctx:
    pass


def timed_steps(cx, tr, batches, K, e2e_host=None, reps=3):
    """device-resident timing (per-step CUDA events, L2 flushed between steps) and, optionally, the end-to-end loop from pinned host
    ids with the loss read back every step.  -> (total_ms, e2e_ms or None, last_loss)"""
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    cx.barrier()
    for k in range(K):
        cx.flush.zero_()
        evs[k][0].record()
        tr.step(*batches[k % len(batches)])
        evs[k][1].record()
    cx.barrier()
    total_ms = float(sum(a.elapsed_time(b) for a, b in evs))
    e2e_ms, last_loss = None, None
    if e2e_host is not None:
        rr = []
        for _ in range(reps):
            cx.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(K):
                tr.step(*e2e_host[k % len(e2e_host)])
                last_loss = tr.loss()
            e1.record()
            cx.barrier()
            rr.append(e0.elapsed_time(e1))
        e2e_ms = float(np.median(rr))
    return total_ms, e2e_ms, last_loss


def reduce_max(cx, *vals):
    t = torch.tensor([float(v) for v in vals], dtype=torch.float64, device=cx.dev)
    if cx.world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return t.tolist()


def kernel_breakdown(cx, tr, batches, KT):
    """per-kernel live timing (events inside the library, eager launches) -> {name: {avg_us, launches, ms_total}}"""
    lib = cx.lib
    names_buf = ctypes.create_string_buffer(4096)
    tot = (ctypes.c_float * 64)()
    cnt = (ctypes.c_int * 64)()
    tr.use_graph = False
    tr.step(*batches[0])
    torch.cuda.synchronize()
    lib.adt_timing_enable(1)
    for k in range(KT):
        cx.flush.zero_()
        tr.step(*batches[k % len(batches)])
    n = lib.adt_timing_collect(names_buf, 4096, tot, cnt, 64)
    lib.adt_timing_enable(0)
    tr.use_graph = True
    knames = names_buf.value.decode().split("\n")[:n]
    return {knames[i]: {"ms_total": tot[i], "launches": cnt[i], "avg_us": 1e3 * tot[i] / max(cnt[i], 1)} for i in range(n)}


def alg_bytes_table(cfg):
    """ALGORITHMIC bytes per launch, SURVEY.md 8(d) per-unit figures x the rows one launch processes (DESIGN.md section 4)"""
    M, H, nh, e = cfg["B"] * cfg["L"], cfg["H"], cfg["nh"], 4
    return {
        "enc_block_fwd": M * (2 * H * e + nh * nh * e), "enc_block_bwd": M * (3 * H * e + nh * nh * e),
        # decoder block, SURVEY 8d: fwd 3 L H e (x, feats in; out), bwd 5 L H e (dout, x, feats in; dx, dfeats out), split over its two launches
        "dec_block_fwd_p1": M * 1 * H * e, "dec_block_fwd_p2": M * 2 * H * e, "dec_block_bwd_p2": M * 3 * H * e, "dec_block_bwd_p1": M * 2 * H * e,
        "enc_post_bwd": M * (3 * H * e + nh * nh * e), "dec_post_bwd": M * 5 * H * e // 2, "attn_bwd": M * 7 * H * e, "attn_fwd": M * 4 * H * e,
        "pre_bwd": M * 5 * H * e, "mid_bwd": M * 8 * H * e, "enc_post_fwd": M * (2 * H * e + nh * nh * e), "dec_post_fwd": M * 3 * H * e,
        "pre_fwd": M * 4 * H * e, "mid_fwd": M * 6 * H * e,
        "embed_fwd": M * (2 * H * e + 4), "final_fwd": M * (H * e + 2 * (H * e + 4) + 8), "final_bwd": M * (3 * H * e + 2 * (H * e + 4)),
    }


def step_alg(cfg):
    """whole-step algorithmic work per sequence (SURVEY 8d): FLOPs = 3[nl(32 L H^2 + 12 L^2 H) + 4 L H]; bytes: per-block figures + embeddings"""
    L_, H, nh, nl, e = cfg["L"], cfg["H"], cfg["nh"], cfg["nl"], 4
    flops = 3 * (nl * (32 * L_ * H * H + 12 * L_ * L_ * H) + 4 * L_ * H)
    by = nl * ((2 * L_ * H * e + L_ * nh * nh * e) + (3 * L_ * H * e + L_ * nh * nh * e) + 3 * L_ * H * e + 5 * L_ * H * e)
    by += 2 * L_ * (2 * H * e + 4) + (L_ * H * e + 2 * L_ * (H * e + 4) + 8 * L_) + 4 * L_ * (2 * H * e + 8)
    by += 7 * (cfg["items"] + 1) * H * 4 / cfg["B"]
    return flops, by


def train_section(cx, args, cfg, name, precision, K, W, with_e2e=True, with_kernels=True, pool=8):
    from adt_b200.trainer import FusedTrainer
    model = make_model(cfg, cx.dev)
    l1, l2 = get_lambdas(cfg["dataset"])
    tr = FusedTrainer(model, l1, l2, weight_decay=cfg["wd"], lr=1e-3, betas=(0.9, 0.98), clip=5.0, seed=23, use_graph=True, precision=precision)
    rng = np.random.default_rng(23 + cx.rank)
    host = [[torch.from_numpy(a).pin_memory() for a in synth.make_batch(rng, cfg)] for _ in range(pool)]
    resident = [[a.to(cx.dev) for a in b] for b in host]
    for i in range(max(W, 3)):
        tr.step(*resident[i % pool])
    cx.barrier()
    total_ms, e2e_ms, last_loss = timed_steps(cx, tr, resident, K, host if with_e2e else None)
    total_ms, e2e_ms_r = reduce_max(cx, total_ms, e2e_ms or 0.0)
    B = cfg["B"]
    out = {"value": cx.world * B * K / (total_ms / 1e3), "ms_per_step": total_ms / K, "steps": K, "dtype": precision,
           "launch": tr.launch_mode, "loss": last_loss}
    if with_e2e:
        out["e2e"] = {"value": cx.world * B * K / (e2e_ms_r / 1e3), "unit": "seqs/s", "h2d_bytes_per_step": 4 * B * cfg["L"] * 4,
                      "d2h_bytes_per_step": 8 * (8 + 2 * cfg["nl"]) + 8, "ms_per_step": e2e_ms_r / K,
                      "timing": "median of 3 repetitions of the K-step region (each step: pinned H2D of the ids + loss read-back)"}
    try:
        out["gpu_launches_per_step"] = tr.kernel_nodes()
    except Exception as e:   # noqa: BLE001
        out["gpu_launches_per_step"] = None
        out["launch_count_error"] = str(e)
    flops, by = step_alg(cfg)
    pk = peaks()
    sps = out["value"] / cx.world
    out["step_roofline"] = {"hbm_frac": sps * by / 1e9 / pk["hbm"], "tensor_frac": sps * flops / 1e12 / pk["bf16_sustained"],
                            "alg_bytes_per_seq": by, "alg_flops_per_seq": flops, "peaks": pk["src"]}
    if with_kernels:
        kern = kernel_breakdown(cx, tr, resident, min(K, 20))
        out["kernels"] = kern
    if with_e2e and with_kernels and name == "C2":
        # end to end WITHOUT any host batch: the batch is assembled on the device from resident user histories (SURVEY 8f-1:
        # adt_assemble_train_batch = WarpDataset.sample_data + random_neq), then the same step, loss read back every step
        from adt_b200.sampler import DeviceSampler
        n_users = 4096
        tr_h, va_h, te_h = synth.make_histories(np.random.default_rng(5), cfg, n_users)
        ds = DeviceSampler(tr_h, va_h, te_h, n_users, cfg["items"], cfg["L"], device=cx.dev, seed=23)
        users = [torch.from_numpy(np.random.default_rng(7 + cx.rank + i).integers(1, n_users + 1, size=B).astype(np.int32)).to(cx.dev) for i in range(8)]
        bufs = [torch.empty(B, cfg["L"], dtype=torch.int32, device=cx.dev) for _ in range(4)]
        for i in range(3):
            tr.step(*ds.train_batch(users[i % 8], epoch=i, out=bufs))
        rr = []
        for _ in range(3):
            cx.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(K):
                tr.step(*ds.train_batch(users[k % 8], epoch=k, out=bufs))
                last_loss = tr.loss()
            e1.record()
            cx.barrier()
            rr.append(e0.elapsed_time(e1))
        (dms,) = reduce_max(cx, float(np.median(rr)))
        out["e2e_device_batches"] = {"value": cx.world * B * K / (dms / 1e3), "unit": "seqs/s", "ms_per_step": dms / K, "h2d_bytes_per_step": 0,
                                     "what": "batch assembled on the GPU (history CSR resident, Philox negatives) + step + loss read-back; "
                                             "the reference feeds this step from 4 CPU DataLoader workers"}
    out["_tr"], out["_model"] = tr, model
    return out


def dump_step(cx, cfg, precision, K, W, pool=8):
    """--dump-outputs: the step of train_section's device-resident timed loop (the K steps behind `value`; same trainer settings,
    CUDA graph and precision) taken once more by a fresh trainer, from the seeded initial weights, on the batch and with the dropout
    stream of that loop's last step.  The trainer sums weight gradients with fp32 atomics, so weights trained for many steps differ
    from run to run by more than rounding: Adam scales each element's update by that element's own gradient, and an element whose
    exact gradient is zero (the key bias under softmax) moves by about lr in a direction set by rounding.  One step from fixed
    weights depends on the arguments only, up to rounding.
    -> {name: array}: loss, gradient norm, and every parameter's gradient after clipping, as Adam applied it."""
    from adt_b200.trainer import FusedTrainer
    model = make_model(cfg, cx.dev)
    l1, l2 = get_lambdas(cfg["dataset"])
    tr = FusedTrainer(model, l1, l2, weight_decay=cfg["wd"], lr=1e-3, betas=(0.9, 0.98), clip=5.0, seed=23, use_graph=True, precision=precision)
    rng = np.random.default_rng(23 + cx.rank)
    batches = [synth.make_batch(rng, cfg) for _ in range(pool)]     # the batches train_section draws
    tr.t = W + K - 1                                  # dropout stream of the last device-resident timed step
    tr.step(*[torch.from_numpy(a).to(cx.dev) for a in batches[(K - 1) % pool]])
    outs = {"train_loss": np.float64(tr.loss()), "train_grad_norm": np.float64(tr.grad_norm())}
    outs.update({f"grad.{n}": tr.eng.grad_view(n).cpu().numpy() for n, _ in tr.eng.order})
    return outs


def dominant_roofline(cfg, kern, config_name):
    ab = alg_bytes_table(cfg)
    pk = peaks()
    tot = max(sum(v["ms_total"] for v in kern.values()), 1e-9)
    top = max(kern, key=lambda k_: kern[k_]["ms_total"])
    ach = ab[top] / (kern[top]["avg_us"] * 1e-6) / 1e9 if top in ab else None
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if config_name == "C2" and os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f)["bytes_per_launch"].get(top)
    M = cfg["B"] * cfg["L"]
    ctas = (M + 63) // 64
    return {"bound": "hbm", "kernel": top, "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": (ach / pk["hbm"]) if ach else None,
            "traffic": traffic, "alg_bytes": ab.get(top), "peak_source": pk["src"], "avg_us": kern[top]["avg_us"],
            "share_of_step": kern[top]["ms_total"] / tot,
            "note": f"{config_name}: M = {M} rows per launch ({cfg['B']} sequences x {cfg['L']} positions), H = {cfg['H']}"}


def eval_section(cx, args, cfg, model, K):
    """full-catalog evaluation users/sec: encoder forward + catalog scoring + fused top-10 + fused HIT/NDCG/MRR, 512 users per batch.
    N > 1: catalogs below CatalogScorer.shard_min_items are not sharded -- every rank evaluates ITS OWN users (weak scaling)."""
    from adt_b200.evaluate import CatalogScorer, GraphedScorer
    model.eval()
    U = 512
    pool = 4
    scorer = CatalogScorer(model, K=10)
    erng = np.random.default_rng(99 + (0 if scorer.sharded else cx.rank))
    bt = [synth.make_eval_batch(erng, cfg, U) for _ in range(pool)]
    max_seen = max(len(b[3]) for b in bt)
    gs = GraphedScorer(scorer, U, cfg["L"], max_seen=max_seen)
    dev_b = [[torch.from_numpy(np.ascontiguousarray(a)).to(cx.dev) for a in b] for b in bt]
    pin_b = [[torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in b] for b in bt]
    for i in range(3):
        gs.topk(dev_b[i % pool][0], dev_b[i % pool][2], dev_b[i % pool][3], dev_b[i % pool][1])
    gs.metrics()
    cx.barrier()
    KE = max(10, min(K, 50))
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(KE)]
    for k in range(KE):
        b = dev_b[k % pool]
        cx.flush.zero_()
        evs[k][0].record()
        gs.topk(b[0], b[2], b[3], b[1])
        evs[k][1].record()
    cx.barrier()
    dev_ms = float(sum(a.elapsed_time(b) for a, b in evs))
    metrics = gs.metrics()
    # end to end: pinned host ids / CSR / answers in, top-10 ids [U,10] back on the host, every batch
    out_host = torch.empty(U, 10, dtype=torch.int32).pin_memory()
    rr = []
    for _ in range(3):
        cx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(KE):
            b = pin_b[k % pool]
            _, ids = gs.topk(b[0], b[2], b[3], b[1])
            out_host.copy_(ids, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        e1.record()
        cx.barrier()
        rr.append(e0.elapsed_time(e1))
    e2e_ms = float(np.median(rr))
    dev_ms, e2e_ms = reduce_max(cx, dev_ms, e2e_ms)
    mult = 1 if scorer.sharded else cx.world       # user-parallel: every rank evaluated different users
    I1, H = cfg["items"] + 1, cfg["H"]
    flops = 2.0 * U * I1 * H
    pk = peaks()
    # the scoring kernel alone, timed live (events around the scorer call on precomputed features)
    feats = model.final_feats(dev_b[0][0])
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        scorer.topk_from_feats(feats, dev_b[0][2], dev_b[0][3])
    torch.cuda.synchronize()
    s0.record()
    for _ in range(10):
        scorer.topk_from_feats(feats, dev_b[0][2], dev_b[0][3])
    s1.record()
    torch.cuda.synchronize()
    score_us = 1e3 * s0.elapsed_time(s1) / 10
    tc = scorer._uses_tc(H, *scorer.bounds())
    h2d = sum(int(a.numel()) * 4 for a in pin_b[0])
    model.train()
    return {"metric": "eval_users_per_sec", "value": mult * U * KE / (dev_ms / 1e3), "unit": "users/s", "users_per_batch": U, "K": 10,
            "items": I1, "batches": KE, "ms_per_batch": dev_ms / KE,
            "launch": "one CUDA graph per batch (encoder + scoring + top-K + metric sums" + (" + all-gather + merge)" if scorer.sharded else ")"),
            "partition": "item-sharded" if scorer.sharded else ("users split across ranks (catalog below shard_min_items)" if cx.world > 1 else "single GPU"),
            "e2e": {"value": mult * U * KE / (e2e_ms / 1e3), "unit": "users/s", "ms_per_batch": e2e_ms / KE, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": U * 10 * 4, "what": "pinned host ids + seen CSR + answers in, [U,10] item ids back on the host, every batch"},
            "roofline": {"bound": "tensor", "kernel": "score_tc_kernel (tcgen05)" if tc else "score_topk_kernel (exact fp32 FFMA: catalog below tc_min_items)",
                         "achieved": flops / (score_us * 1e-6) / 1e12, "peak": pk["bf16"], "unit": "TFLOP/s",
                         "frac": flops / (score_us * 1e-6) / 1e12 / pk["bf16"], "traffic": None, "avg_us": score_us,
                         "alg_flops": flops, "peak_source": pk["src"],
                         "note": "2*U*(I+1)*H flops of one 512-user batch / scoring time; a 12k-item catalog is 1.55 MFLOP per user: latency bound, see c5 for the 1M-item roofline"},
            "metrics": metrics, "fallback_users": scorer.fallback_users}


def c5_section(cx, args):
    """catalog scoring at 1M items (configs[4]): 512 users x 1,000,001 items, H 64 and 256, top-10, tensor-core path with the exact
    re-score; item-sharded across the ranks when N > 1."""
    import types
    from adt_b200.evaluate import CatalogScorer
    pk = peaks()
    out = {}
    I = 1_000_000
    U = 512
    for H in (64, 256):
        g = torch.Generator(device="cpu").manual_seed(5 + H)
        E = (torch.randn(I + 1, H, generator=g) * (2.0 / (I + 1 + H)) ** 0.5 * 30).to(cx.dev)
        feats = torch.randn(U, H, generator=g).to(cx.dev)
        fake = types.SimpleNamespace(item_emb=types.SimpleNamespace(weight=E), hidden=H)
        sc = CatalogScorer(fake, K=10)
        sc.refresh_table()
        for _ in range(3):
            sc.topk_from_feats(feats)
        cx.barrier()
        n = 10
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for k in range(n):
            evs[k][0].record()
            s_, i_ = sc.topk_from_feats(feats)
            evs[k][1].record()
        cx.barrier()
        ms = float(sum(a.elapsed_time(b) for a, b in evs)) / n
        (ms,) = reduce_max(cx, ms)
        flops = 2.0 * U * (I + 1) * H
        # spot check against the exact fp32 kernel (ids identical)
        ex = CatalogScorer(fake, K=10, use_tensor_cores=False)
        se, ie = ex.topk_from_feats(feats)
        same = bool(torch.equal(i_, ie))
        out[f"U{U}_I1M_H{H}"] = {"ms": ms, "users_per_sec": U / (ms / 1e3), "tflops": flops / (ms * 1e-3) / 1e12,
                                 "tensor_frac": flops / (ms * 1e-3) / 1e12 / pk["bf16"], "partition": "item-sharded" if sc.sharded else "single GPU",
                                 "ids_equal_exact_fp32": same, "fallback_users": sc.fallback_users,
                                 "catalog_larger_than_l2": True}
        del E, sc, ex, fake
        torch.cuda.empty_cache()
    out["peak_tflops"] = pk["bf16"]
    out["what"] = "adt_score_topk_tc + exact re-score + masked exact re-run, features resident; whole call timed per batch (catalog >> 126 MB L2)"
    return out


def c3_section(cx):
    """configs[2]: Bert4Rec-ADT cloze training step at the ml-20m shape (B 256/GPU, L 200, H 256, 4 heads, inner 1024, 26,744 items,
    mask_prob 0.2): fused loss (vocabulary head on the labelled positions only) + backward + flat clip/Adam, linear layers on tcgen05
    (adt_gemm_tc), batches generated on the device (adt_cloze_batch).  Data parallel over the ranks (one all-reduce of the flat gradient)."""
    import types
    from adt_b200.bert4rec import BertModel
    from adt_b200.dp import FlatOptimizer
    from adt_b200.sampler import ClozeSampler
    B, L_, H, nh, nl, I, inner = 256, 200, 256, 4, 2, 26744, 1024
    args = types.SimpleNamespace(device=cx.dev, num_heads=nh, maxlen=L_, num_layers=nl, hidden_units=H, dropout=0.1, attention_dropout=0.1,
                                 inner_units=inner, type_vocab_size=2)
    torch.manual_seed(0)
    m = BertModel(100, I, args).to(cx.dev).train()
    m.precision = 1
    rng = np.random.default_rng(23 + cx.rank)
    n_users = 512
    hist = {u: [int(x) for x in rng.integers(1, I + 1, size=int(np.clip(rng.geometric(1.0 / 144) + 2, 3, 400)))] for u in range(1, n_users + 1)}
    cs = ClozeSampler(hist, n_users, I, L_, mask_prob=0.2, dupe_factor=2, prop_sliding_window=0.5, device=cx.dev, seed=23)
    opt = FlatOptimizer(m, lr=1e-3, clip=5.0)
    order = torch.from_numpy(rng.permutation(len(cs))).to(cx.dev)
    state = {"i": 0}

    def step():
        idx = order[(state["i"] * B) % (len(cs) - B):][:B]
        state["i"] += 1
        src, dec, lab = cs.batch(idx, epoch=state["i"])
        opt.zero_grad()
        loss = m.fused_loss(src, dec, lab, [0.01, 0.01], [0.001, 0.001])
        loss.backward()
        opt.step()
        return loss
    for _ in range(3):
        step()
    cx.barrier()
    K3 = 8
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K3):
        loss = step()
    e1.record()
    cx.barrier()
    (ms,) = reduce_max(cx, e0.elapsed_time(e1) / K3)
    out = {"workload": "Bert4Rec-ADT C3: cloze train step (items=26744, maxlen=200, hidden=256, heads=4, inner=1024, blocks=2, batch=256/GPU, mask_prob=0.2)",
           "value": cx.world * B / (ms / 1e3), "unit": "seqs/s", "ms_per_step": ms, "steps": K3, "dtype": "bf16", "loss": float(loss),
           "launch": "eager launches (autograd-composed ops); batches from adt_cloze_batch", "round1_ms_per_step_fp32_cores": 86.0}
    del m, opt, cs
    torch.cuda.empty_cache()
    return out


def refgpu_section(cx, cfg):
    """the unmodified reference (PyTorch eager, fp32) on the same B200: SURVEY 8d's 'honest kernel bar'"""
    try:
        v, ms, n = time_reference_train(cfg, "cuda", steps=10, warmup=3)
        ev, ems, en = time_reference_eval(cfg, "cuda", batches=10, warmup=2)
        return {"train_seqs_per_sec": v, "train_ms_per_step": ms, "eval_users_per_sec": ev, "eval_ms_per_batch": ems,
                "what": "oracle/_ref SASRecADT + main.py:146-173 lines, device='cuda', torch eager fp32, host ids in, loss.item() per step"}
    except Exception as e:   # noqa: BLE001
        return {"unavailable": str(e)[:200]}


def evolution_section(cx, cfg):
    """evolution.py's population evaluation on the frozen supernet (SURVEY 8e row 3 / 8f-2): candidates dealt round-robin to the ranks,
    validation batches assembled once on the device, fused rank metrics; serial (one candidate at a time) vs 4 candidates in flight."""
    import types
    from adt_b200.supernet import SuperSASRecModel
    from adt_b200.sampler import DeviceSampler
    from adt_b200.evolution import PopulationEvaluator
    rec_choice = [0, 0.0001, 0.0005, 0.001, 0.005, 0.01]          # sasrec/evolution.py:95-96
    ind_choice = [0, 0.0001, 0.0005, 0.001, 0.0015, 0.002]
    n_users, n_val, C = 4096, 2048, 100
    tr_h, va_h, te_h = synth.make_histories(np.random.default_rng(5), cfg, n_users)
    torch.manual_seed(3)
    args = types.SimpleNamespace(device=cx.dev, num_heads=cfg["nh"], maxlen=cfg["L"], num_layers=cfg["nl"], hidden_units=cfg["H"], dropout=cfg["p"])
    m = SuperSASRecModel(n_users, cfg["items"], rec_choice, ind_choice, args).to(cx.dev).eval()
    m.precision = 1          # bf16 GEMM cores for the fitness pass (ranking metrics; BASELINE tolerance 2e-2): one launch per candidate block
    ds = DeviceSampler(tr_h, va_h, te_h, n_users, cfg["items"], cfg["L"], device=cx.dev, seed=23)
    users = np.arange(1, n_val + 1, dtype=np.int32)
    batches = [ds.eval_batch(users[i:i + 512], mode="val", n_candidates=C) for i in range(0, n_val, 512)]
    rng = np.random.default_rng(11)
    n_cand = 8 * cx.world
    cands = [list(rng.random(2 * cfg["nl"]) * 0.98) for _ in range(n_cand)]
    res = {}
    fit = None
    for name, inflight in (("serial", 1), ("in_flight_4", 4)):
        pe = PopulationEvaluator(m, batches, rec_choice, ind_choice, in_flight=inflight)
        pe.evaluate(cands[:cx.world * 2])
        cx.barrier()
        t0 = time.time()
        fit = pe.evaluate(cands)
        cx.barrier()
        dt = time.time() - t0
        (dt,) = reduce_max(cx, dt)
        res[name] = {"candidates_per_sec": n_cand / dt, "seconds": dt}
    res.update({"candidates": n_cand, "val_users": n_val, "sampled_negatives": C, "ranks": cx.world,
                "best_auc": float(np.max(fit[:, 0])), "what": "set_choice + supernet encoder (4 blended candidate blocks per layer) + "
                "gather-dot / rank / AUC-NDCG-HR sums per 512-user batch; candidates c -> rank c mod G"})
    return res


def selfcheck_section(cx):
    """N > 1: (a) the data-parallel step on the c2mini_p5 fixture (6 sequences split across 2 ranks... all ranks take a slice) against
    the unmodified reference's loss / updated weights; (b) item-sharded top-K against the single-GPU exact scorer."""
    from adt_b200 import testing as T
    from adt_b200.trainer import FusedTrainer
    from adt_b200.evaluate import CatalogScorer
    res = {}
    g = T.load_golden("c2mini_p5")
    B = g["seq"].shape[0]
    if B % cx.world == 0:
        per = B // cx.world
        sl = slice(cx.rank * per, (cx.rank + 1) * per)
        l1, l2, wd = [float(x) for x in g["lambdas1"]], [float(x) for x in g["lambdas2"]], float(g["wd"])
        m = T.model_from_golden(g).train()
        tr = FusedTrainer(m, l1, l2, weight_decay=wd, seed=int(g["drop_seed"]))
        tr.t = int(g["drop_step"])
        tr.step(g["seq"][sl], g["dec"][sl], g["pos"][sl], g["neg"][sl])
        loss = tr.loss()
        gn = tr.grad_norm()
        e_loss = abs(loss - float(g["loss"])) / abs(float(g["loss"]))
        e_gn = abs(gn - float(g["gnorm"])) / abs(float(g["gnorm"]))
        res["dp_parity"] = {"loss_rel_err": e_loss, "grad_norm_rel_err": e_gn, "ok": bool(e_loss < 1e-5 and e_gn < 1e-4), "ranks": cx.world,
                            "fixture": "tests/golden/sasrec_c2mini_p5.npz (unmodified reference; its 6 sequences split across the ranks, "
                                       "loss and global gradient norm of the all-reduced step against the reference's)"}
    else:
        # the fixture's 6 sequences do not split over this many ranks: tile them cyclically to world * per sequences and compare the
        # N-rank step with the SINGLE-rank step (a one-member process group) on the same global batch -- same Philox streams, because
        # a rank's dropout counters start at its global row offset
        per = -(-B // cx.world)
        idx = [(cx.rank * per + i) % B for i in range(per)]
        gidx = [(r * per + i) % B for r in range(cx.world) for i in range(per)]
        solo = [torch.distributed.new_group(ranks=[r]) for r in range(cx.world)][cx.rank]
        l1, l2, wd = [float(x) for x in g["lambdas1"]], [float(x) for x in g["lambdas2"]], float(g["wd"])
        out = []
        for pg, ii in ((None, idx), (solo, gidx)):
            m = T.model_from_golden(g).train()
            tr = FusedTrainer(m, l1, l2, weight_decay=wd, seed=int(g["drop_seed"]), process_group=pg)
            tr.t = int(g["drop_step"])
            tr.step(g["seq"][ii], g["dec"][ii], g["pos"][ii], g["neg"][ii])
            out.append((tr.loss(), tr.grad_norm()))
        (loss, gn), (loss1, gn1) = out
        e_loss, e_gn = abs(loss - loss1) / abs(loss1), abs(gn - gn1) / abs(gn1)
        res["dp_parity"] = {"loss_rel_err": e_loss, "grad_norm_rel_err": e_gn, "ok": bool(e_loss < 1e-5 and e_gn < 1e-4), "ranks": cx.world,
                            "fixture": f"tests/golden/sasrec_c2mini_p5.npz tiled to {len(gidx)} sequences ({per} per rank): loss and global gradient "
                                       "norm of the all-reduced N-rank step against the single-rank step on the same global batch"}
    # item-sharded top-K: every rank scores the same users against its shard; merged ids must equal the unsharded exact result
    import types
    gen = torch.Generator(device="cpu").manual_seed(11)
    I, H, U = 70_001, 64, 256
    E = (torch.randn(I, H, generator=gen) * 0.1).to(cx.dev)
    feats = torch.randn(U, H, generator=gen).to(cx.dev)
    ans = torch.randint(1, I, (U,), generator=gen).int().to(cx.dev)
    fake = types.SimpleNamespace(item_emb=types.SimpleNamespace(weight=E), hidden=H)
    acc_s = torch.zeros(6, dtype=torch.float64, device=cx.dev)
    acc_1 = torch.zeros(6, dtype=torch.float64, device=cx.dev)
    sh = CatalogScorer(fake, K=10, shard=True, tc_min_items=0)
    s_s, i_s = sh.topk_from_feats(feats, answers=ans, metric_acc=acc_s)
    one = CatalogScorer(fake, K=10, shard=False, use_tensor_cores=False)
    s_1, i_1 = one.topk_from_feats(feats, answers=ans, metric_acc=acc_1)
    res["shard_eval_parity"] = {"ids_equal": bool(torch.equal(i_s, i_1)), "scores_equal": bool(torch.equal(s_s, s_1)),
                                "metrics_equal": bool(torch.equal(acc_s, acc_1)), "shards": cx.world, "items": I, "users": U,
                                "ok": bool(torch.equal(i_s, i_1) and torch.equal(acc_s, acc_1))}
    return res


# ------------------------------------------------------------------------------------------------ our arm
def main():
    args = parse()
    cfg = synth.CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return
    from adt_b200 import _lib as L
    skip = set(x for x in args.skip.split(",") if x)
    torch.cuda.set_device(local)
    cx = Ctx()
    cx.dev = torch.device("cuda", local)
    cx.world, cx.rank = world, rank
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=cx.dev)
    cx.lib = L.lib()
    cx.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=cx.dev)   # > 126 MB L2

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
    cx.barrier = barrier

    def trace(msg):
        if os.environ.get("ADT_BENCH_TRACE"):
            print(f"[bench rank {rank}] {msg}", file=sys.stderr, flush=True)

    K, W = args.steps, max(args.warmup, 3)
    trace("train")
    with ClockSampler(local) as clk:
        main_tr = train_section(cx, args, cfg, args.config, args.precision, K, W)
    clocks = clk.summary()
    model, tr = main_tr.pop("_model"), main_tr.pop("_tr")
    kern = main_tr.pop("kernels")
    roofline = dominant_roofline(cfg, kern, args.config)

    other = "fp32" if args.precision == "bf16" else "bf16"
    other_mode = None
    if "fp32" not in skip:
        trace("other precision")
        o = train_section(cx, args, cfg, args.config, other, min(K, 20), 3, with_e2e=True, with_kernels=False, pool=4)
        o.pop("_model"); o.pop("_tr")
        other_mode = o

    ev = None
    if "eval" not in skip:
        trace("eval")
        ev = eval_section(cx, args, cfg, model, K)

    c1 = None
    if "c1" not in skip and args.config != "C1":
        trace("c1")
        c1cfg = synth.CONFIGS["C1"]
        o = train_section(cx, args, c1cfg, "C1", args.precision, min(K, 10), 3, with_e2e=False, with_kernels=True, pool=2)
        o.pop("_model"); o.pop("_tr")
        k1 = o.pop("kernels")
        o["roofline"] = dominant_roofline(c1cfg, k1, "C1")
        o["kernels_us"] = {k_: round(v["avg_us"], 1) for k_, v in sorted(k1.items())}
        o["workload"] = workload_name("C1", c1cfg)
        c1 = o
        torch.cuda.empty_cache()

    c3 = None
    if "c3" not in skip:
        trace("c3")
        try:
            c3 = c3_section(cx)
        except Exception as e:   # noqa: BLE001
            c3 = {"error": str(e)[:300]}

    c5 = None
    if "c5" not in skip:
        trace("c5")
        try:
            c5 = c5_section(cx, args)
        except Exception as e:   # noqa: BLE001
            c5 = {"error": str(e)[:300]}

    evo = None
    if "evo" not in skip:
        trace("evolution")
        try:
            evo = evolution_section(cx, cfg)
        except Exception as e:   # noqa: BLE001
            evo = {"error": str(e)[:300]}

    selfcheck = None
    if world > 1 and "selfcheck" not in skip:
        trace("selfcheck")
        try:
            selfcheck = selfcheck_section(cx)
        except Exception as e:   # noqa: BLE001
            selfcheck = {"error": str(e)[:300]}

    refgpu = None
    if rank == 0 and world == 1 and "refgpu" not in skip:
        trace("reference on the GPU (eager)")
        refgpu = refgpu_section(cx, cfg)

    trace("cpu baseline")
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        try:
            v, ms, ns = time_reference_train(cfg, "cpu", steps=20, warmup=1, budget_s=args.cpu_budget_s)
            cpu = {"value": v, "unit": "seqs/s", "cores": cores, "kind": "reference", "ms_per_step": ms,
                   "sample": f"{ns} full optimisation steps of {cfg['B']}-sequence batches of the same workload (median, 1 warm-up, torch dropout)"}
            if ev is not None:
                e_v, e_ms, e_n = time_reference_eval(cfg, "cpu", batches=10, warmup=1, budget_s=args.cpu_budget_s / 2)
                ev["cpu_baseline"] = {"value": e_v, "unit": "users/s", "cores": cores, "kind": "reference", "ms_per_batch": e_ms,
                                      "sample": f"{e_n} batches of 512 users: predict(full=True) + mask + argpartition(40) + argsort (median, 1 warm-up)"}
        except Exception as e:   # noqa: BLE001
            cpu = {"unavailable": str(e)[:200]}

    if args.dump_outputs:
        trace("dump outputs")
        outs = dump_step(cx, cfg, args.precision, K, W)       # every rank: the step all-reduces when N > 1
        if rank == 0:
            dump_outputs(args.dump_outputs, outs)

    if rank == 0:
        lps = main_tr.get("gpu_launches_per_step")
        line = {
            "metric": "train_seqs_per_sec", "value": main_tr["value"], "unit": "seqs/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": main_tr["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.precision,
            "data": "synthetic", "config": config_dict(args, cfg, world), "launch": main_tr["launch"],
            "e2e": main_tr["e2e"], "e2e_device_batches": main_tr.get("e2e_device_batches"), "gpu_launches": (lps * K) if lps else None, "gpu_launches_per_step": lps,
            "gpu_launches_how": "kernel nodes of the captured step graph (cuGraphGetNodes) x timed steps",
            "loss": main_tr["loss"], "roofline": roofline, "step_roofline": main_tr["step_roofline"],
            "kernels_us": {k_: round(v["avg_us"], 2) for k_, v in sorted(kern.items())},
            "eval_users_per_sec": ev["value"] if ev else None, "eval": ev,
            ("fp32" if other == "fp32" else "bf16"): other_mode, "c1": c1, "c3": c3, "c5": c5, "evolution": evo, "selfcheck": selfcheck, "reference_gpu_eager": refgpu,
            "cpu_baseline": cpu, "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # the step / evaluation graphs hold captured NCCL work: tearing the communicator down underneath them can block at interpreter
        # exit, so every rank synchronises, agrees that the line is out, and leaves without running destructors
        torch.cuda.synchronize()
        torch.distributed.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
