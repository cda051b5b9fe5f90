"""Flat-buffer optimiser step + data-parallel gradient exchange for the autograd-composed models (Bert4Rec-ADT, STOSA-ADT,
supernet): the reference's `clip_grad_norm_` + `torch.optim.Adam` (bert4rec/trainer.py:27,129-131; stosa/trainer.py:36,
535-537; sasrec/evolution.py:111,316-318) as three launches of libadt_b200.so over ONE flat parameter / gradient / state
buffer, with a single NCCL all-reduce(avg) of the flat gradient when a process group is active (SURVEY 8e: training is
data parallel, model replicated, replicas stay bit-identical)."""
import ctypes
import torch

from . import _lib as L


class FlatOptimizer:
    """clip_grad_norm_ + torch.optim.Adam over ONE flat parameter / gradient / state buffer.

    torch semantics are kept per parameter: a parameter that received no gradient in this backward (`.grad is None` in the
    reference -- the 32 inactive candidate blocks of every supernet layer, sasrec/evolution.py:111,316-318) is skipped entirely
    (no moment decay, no weight decay, no step increment, no all-reduce traffic) and every parameter keeps its own Adam step
    count.  Which parameters were touched is recorded on the host by post-accumulate-grad hooks (no device synchronisation);
    while every step touches every parameter the plain one-launch kernel runs."""

    CHUNK = 8192

    def __init__(self, model, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, clip=None, process_group=None):
        self.model = model
        self.params = [p for p in model.parameters() if p.requires_grad]
        if not self.params or self.params[0].device.type != "cuda":
            raise L.AdtError("adt_b200.FlatOptimizer needs the model on a CUDA device (no CPU fallback)")
        dev = self.params[0].device
        offs, total = [], 0
        for p in self.params:
            offs.append(total)
            total += (p.numel() + 3) // 4 * 4            # 16-byte aligned segments
        self.offs = offs
        self.pflat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.gflat = torch.zeros_like(self.pflat)
        self.m, self.v = torch.zeros_like(self.pflat), torch.zeros_like(self.pflat)
        self._touched = set()
        for i, (p, o) in enumerate(zip(self.params, offs)):
            n = p.numel()
            self.pflat[o:o + n].copy_(p.data.reshape(-1))
            p.data = self.pflat[o:o + n].view(p.shape)   # parameters become views of the flat buffer
            p.grad = self.gflat[o:o + n].view(p.shape)   # autograd accumulates straight into the flat gradient
            p.register_post_accumulate_grad_hook(lambda _p, i=i: self._touched.add(i))
        self.lr, self.betas, self.eps, self.wd = float(lr), betas, float(eps), float(weight_decay)
        self.clip = float(clip) if clip else 0.0
        self.pg = process_group
        self.world = 1
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
        self.t = 0
        self.gn = torch.zeros(1, dtype=torch.float64, device=dev)
        self.lib = L.lib()
        self.uniform = True                                # every step so far touched every parameter
        self.seg_step = torch.zeros(len(self.params), dtype=torch.int32, device=dev)
        self._plans = {}                                   # frozenset(active) -> device work list
        self.last_active = None

    def zero_grad(self):
        self.gflat.zero_()
        self._touched.clear()

    def grad_norm(self):
        """global gradient norm seen by the last step (before clipping)."""
        return float(self.gn.sqrt())

    # ------------------------------------------------------------------ segmented path
    def active_ranges(self, active):
        """merge the flat-buffer spans of the active parameters into maximal contiguous [start, end) element ranges"""
        rng = []
        for i in sorted(active):
            s, e = self.offs[i], self.offs[i] + (self.params[i].numel() + 3) // 4 * 4
            if rng and rng[-1][1] == s:
                rng[-1][1] = e
            else:
                rng.append([s, e])
        return rng

    def _plan(self, active):
        key = frozenset(active)
        pl = self._plans.get(key)
        if pl is None:
            dev = self.pflat.device
            st, ln, sg = [], [], []
            for i in sorted(active):
                o, n = self.offs[i], self.params[i].numel()
                for c in range(0, n, self.CHUNK):
                    st.append(o + c); ln.append(min(self.CHUNK, n - c)); sg.append(i)
            pl = (torch.tensor(st, dtype=torch.int64, device=dev), torch.tensor(ln, dtype=torch.int32, device=dev),
                  torch.tensor(sg, dtype=torch.int32, device=dev), torch.tensor(sorted(active), dtype=torch.int32, device=dev), len(st),
                  self.active_ranges(active))
            if len(self._plans) > 256:
                self._plans.clear()
            self._plans[key] = pl
        return pl

    def step(self, step_dev=None):
        """step_dev: optional int32 device tensor holding Adam's t (already incremented) -- used under CUDA-graph replay."""
        st = ctypes.c_void_p(torch.cuda.current_stream(self.pflat.device).cuda_stream)
        if self._touched or self.last_active is None:
            active = set(self._touched) if self._touched else set(range(len(self.params)))
        else:
            active = self.last_active                     # graph replay / hooks did not fire: same topology as the last eager step
        self.last_active = active
        full = len(active) == len(self.params)
        if not full:
            self.uniform = False
        n = self.pflat.numel()
        if self.world > 1:
            if full:
                torch.distributed.all_reduce(self.gflat, op=torch.distributed.ReduceOp.AVG, group=self.pg)
            else:       # only the active slices travel (SURVEY 8e: supernet warm-up all-reduces the 4*nl active blocks)
                rng = self._plan(active)[5]
                pack = torch.cat([self.gflat[s:e] for s, e in rng])
                torch.distributed.all_reduce(pack, op=torch.distributed.ReduceOp.AVG, group=self.pg)
                o = 0
                for s, e in rng:
                    self.gflat[s:e].copy_(pack[o:o + e - s]); o += e - s
        self.gn.zero_()
        L.check(self.lib.adt_sumsq(L.ptr(self.gflat), ctypes.c_int64(n), L.ptr(self.gn), st), "adt_sumsq")
        self.t += 1
        self.model._adt_param_version = getattr(self.model, "_adt_param_version", 0) + 1   # raw-pointer update: see CatalogScorer.ensure_table
        a = L.fill(L.adt_adam_args(), p=self.pflat, g=self.gflat, m=self.m, v=self.v, n=n, lr=self.lr, beta1=self.betas[0],
                   beta2=self.betas[1], eps=self.eps, weight_decay=self.wd, step=self.t, max_norm=self.clip, gnormsq=self.gn,
                   step_dev=step_dev)
        if self.uniform:
            self.seg_step.add_(1)
            L.check(self.lib.adt_adam(ctypes.byref(a), st), "adt_adam")
            return
        cs, cl, cg, act, nch, _ = self._plan(active)
        g = L.fill(L.adt_adam_segments(), chunk_start=cs, chunk_len=cl, chunk_seg=cg, n_chunks=nch, seg_step=self.seg_step,
                   active_seg=act, n_active=len(active))
        L.check(self.lib.adt_adam_segmented(ctypes.byref(a), ctypes.byref(g), st), "adt_adam_segmented")


class GraphedStep:
    """One optimisation step of an autograd-composed model (Bert4Rec-ADT, STOSA-ADT) captured ONCE as a CUDA graph and replayed:
    zero_grad -> loss_fn(*static inputs) -> backward -> FlatOptimizer.step.  Dropout's step index and Adam's t advance through
    device-side counters, so replay k reproduces eager step k.  Single-process only (the NCCL all-reduce of the data-parallel
    path is issued eagerly by FlatOptimizer; use the eager loop there).  Build it BEFORE any eager forward/backward of the same
    parameters on the default stream: autograd binds each leaf's gradient accumulator to the stream of its first forward, and
    work on the legacy default stream cannot be captured (the warm-up here runs on a side stream for that reason).

        gs = GraphedStep(model, opt, lambda seq, dec, pos, neg: model.fused_loss(seq, dec, pos, neg, l1, l2)[0])
        loss = gs.step(seq, dec, pos, neg)          # int arrays [B, L]; returns a device scalar (no sync)
    """

    def __init__(self, model, opt, loss_fn, warmup=2):
        if opt.world > 1:
            raise L.AdtError("GraphedStep is single-process; run the eager FlatOptimizer loop under data parallelism")
        self.model, self.opt, self.loss_fn, self.warmup = model, opt, loss_fn, warmup
        self.graph, self.static, self.loss = None, None, None
        dev = opt.pflat.device
        self.counters = torch.zeros(2, dtype=torch.int32, device=dev)     # [0] dropout step offset, [1] Adam t
        self.steps = 0

    def _one(self):
        opt = self.opt
        opt.zero_grad()
        loss = self.loss_fn(*self.static)
        loss.backward()
        self.counters[1:2].add_(1)
        opt.step(step_dev=self.counters[1:2])
        self.counters[0:1].add_(1)
        return loss.detach()

    def _capture(self, arrays):
        m, opt, dev = self.model, self.opt, self.opt.pflat.device
        self.static = [torch.zeros(tuple(a.shape), dtype=torch.int32, device=dev) for a in arrays]
        for d, a in zip(self.static, arrays):
            d.copy_(_to_i32(a, dev))
        m.step_dev = self.counters[0:1]
        snap = (opt.pflat.clone(), opt.m.clone(), opt.v.clone(), self.counters.clone(), m.drop_step, opt.t, opt.seg_step.clone())
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                      # warm-up outside capture (lazy allocations, function attributes)
            for _ in range(self.warmup):
                self._one()
        torch.cuda.current_stream(dev).wait_stream(side)

        def restore():
            opt.pflat.copy_(snap[0]); opt.m.copy_(snap[1]); opt.v.copy_(snap[2]); self.counters.copy_(snap[3])
            m.drop_step, opt.t = snap[4], snap[5]
            opt.seg_step.copy_(snap[6])          # per-parameter step counts (segmented Adam) advanced during the warm-up too
        restore()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = self._one()
        restore()                                          # capture does not execute; keep host-side counters explicit

    def step(self, *arrays):
        if self.graph is None:
            self._capture(arrays)
        dev = self.opt.pflat.device
        for d, a in zip(self.static, arrays):
            d.copy_(_to_i32(a, dev), non_blocking=True)
        self.graph.replay()
        self.steps += 1
        # the replayed Adam kernel wrote the parameters through raw pointers, which moves no tensor version: announce it like
        # FlatOptimizer.step does, so derived data (scorer bf16 copies, STOSA's ranked catalog) is rebuilt before its next use
        self.model._adt_param_version = getattr(self.model, "_adt_param_version", 0) + 1
        return self.loss


def _to_i32(a, dev):
    import numpy as np
    if isinstance(a, torch.Tensor):
        return a.to(device=dev, dtype=torch.int32, non_blocking=True)
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev, non_blocking=True)
