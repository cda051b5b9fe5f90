"""One runner of the SASRec-ADT encoder and decoder blocks through the block C ABI (adt_enc_block_fwd / _bwd, adt_dec_block_fwd / _bwd),
for the block tests.

Inputs are seeded on the host (fp32), so the same dictionary feeds the kernels and the fp64 references of block_ref.py.  Every output
and scratch buffer starts as NaN (bytes 0xff in the bf16 scratch areas), so a row a kernel fails to write shows up; every accumulated
output (g_*, dfeats, nll_acc, mse_acc) starts at known non-zero values, and run() returns initial value + contribution minus the
initial value, i.e. the contribution.  The names of the kernels each call launched are collected with adt_timing_enable /
adt_timing_collect, so a test can pin the route a case takes."""
import ctypes

import numpy as np
import torch

from block_ref import DEC_PARAMS, ENC_PARAMS


class Case:
    """B sequences of L positions, hidden size H, nh heads; pad[b] = left padding of sequence b (L: an empty sequence); dropout p with
    the data-parallel batch offset b0 and an optional device step counter sdev added to the step at run time"""

    def __init__(self, B, L, H, nh, pad, mask_mode=0, p=0.5, b0=0, sdev=None, precision=1, seed=0):
        assert len(pad) == B
        self.B, self.L, self.H, self.nh, self.pad, self.mask_mode, self.p = B, L, H, nh, list(pad), mask_mode, p
        self.b0, self.sdev, self.precision, self.seed = b0, sdev, precision, seed

    def __repr__(self):
        return f"{self.B}x{self.L} H{self.H}/{self.nh} mask{self.mask_mode} p{self.p} prec{self.precision}"


SEED, STEP, ENC_SITES, DEC_SITES = 77, 5, (0, 1, 2), (3, 4, 5, 6)


def inputs(c):
    """{"enc": ..., "dec": ...}: host fp32 tensors of both blocks and the scalars their references need"""
    from oracle.sasrec_oracle import Drop
    B, L, H, nh = c.B, c.L, c.H, c.nh
    M = B * L
    g = torch.Generator().manual_seed(1000 + 7 * L + 13 * H + nh + c.seed)
    rnd = lambda *s, sc=1.0: sc * torch.randn(*s, generator=g)
    ids = torch.zeros(B, L, dtype=torch.int32)
    for b in range(B):
        ids[b, c.pad[b]:] = torch.randint(1, 100, (L - c.pad[b],), generator=g, dtype=torch.int32)
    drop = Drop(c.p, SEED, STEP + (c.sdev or 0), c.b0)
    base = dict(B=B, L=L, H=H, nh=nh, ids=ids, mask_mode=c.mask_mode, drop=drop)

    def lin(n_out, n_in):
        return rnd(n_out, n_in, sc=n_in ** -0.5), rnd(n_out, sc=0.1)

    def ln():
        return 1.0 + rnd(H, sc=0.1), rnd(H, sc=0.1)

    enc = dict(base, x=rnd(M, H), sites=ENC_SITES)
    enc["ln1_w"], enc["ln1_b"] = ln()
    enc["in_w"], enc["in_b"] = lin(3 * H, H)
    enc["out_w"], enc["out_b"] = lin(H, H)
    enc["ln2_w"], enc["ln2_b"] = ln()
    enc["w1"], enc["b1"] = lin(H, H)
    enc["w2"], enc["b2"] = lin(H, H)
    enc["sp_w"], enc["sp_b"] = rnd(nh, H // nh, sc=0.3), rnd(nh, sc=0.1)
    enc.update(dout=rnd(M, H), dx_extra=rnd(M, H), drec=rnd(M, nh, nh, sc=0.1), nll_coef=0.3)
    dec = dict(base, x=rnd(M, H), feats=rnd(M, H), sites=DEC_SITES)
    dec["ln_w"], dec["ln_b"] = ln()
    for pre in ("s_", "e_"):
        dec[pre + "in_w"], dec[pre + "in_b"] = lin(3 * H, H)
        dec[pre + "out_w"], dec[pre + "out_b"] = lin(H, H)
    dec["w1"], dec["b1"] = lin(H, H)
    dec["w2"], dec["b2"] = lin(H, H)
    dec.update(dout=rnd(M, H), enc_in=rnd(M, H), mse_coef=0.7)
    return {"enc": enc, "dec": dec}


def _sizes(c):
    from adt_b200 import _lib as L_
    q = L_.fill(L_.adt_workspace_query(), B=c.B, L=c.L, H=c.H, nh=c.nh, nl=1, K=1, n_splits=1)
    sz = L_.adt_workspace_sizes()
    L_.check(L_.lib().adt_workspace_bytes(ctypes.byref(q), ctypes.byref(sz)), "adt_workspace_bytes")
    return sz


class _Timed:
    """kernel names launched inside the with-block"""

    def __enter__(self):
        from adt_b200 import _lib as L_
        L_.lib().adt_timing_enable(1)
        self.names = []
        return self

    def __exit__(self, *exc):
        from adt_b200 import _lib as L_
        lib = L_.lib()
        buf, tot, cnt = ctypes.create_string_buffer(8192), (ctypes.c_float * 64)(), (ctypes.c_int * 64)()
        n = lib.adt_timing_collect(buf, 8192, tot, cnt, 64)
        lib.adt_timing_enable(0)
        self.names[:] = buf.value.decode().split("\n")[:n]


class Mirror:
    """one flat fp32 parameter buffer (segments on 8-element boundaries) and its RN bf16 copy: the adt_wmirror of the trainer"""

    def __init__(self, tensors, dev):
        offs, n = [], 0
        for t in tensors:
            offs.append(n)
            n += (t.numel() + 7) // 8 * 8
        self.flat = torch.zeros(n, dtype=torch.float32, device=dev)
        self.views = []
        for t, o in zip(tensors, offs):
            v = self.flat[o:o + t.numel()].view(t.shape)
            v.copy_(t)
            self.views.append(v)
        self.bf16 = self.flat.to(torch.bfloat16)


def run(c, inp, phases=(0, 0, 0), wm=False, extras=True):
    """both blocks forward + backward on the device.  phases = (encoder forward, decoder forward, decoder backward): 0 runs the whole
    call, 12 runs phase 1 then phase 2 (forward), 21 phase 2 then phase 1 (decoder backward).  wm: pass an adt_wmirror of the
    parameters.  extras: the trainer's extra arguments (nll_acc / nll_coef / drec / dx_extra, enc_in / mse_acc / mse_coef / denc).
    Returns {"enc/<name>" | "dec/<name>": array} with block_ref's names, and {"names/<call>": [kernel names]}."""
    from adt_b200 import _lib as L_
    lib, dev = L_.lib(), torch.device("cuda")
    B, Lq, H, nh = c.B, c.L, c.H, c.nh
    M, prec = B * Lq, c.precision
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = torch.Generator().manual_seed(5)
    keep = []                       # the C structs hold raw pointers: the tensors behind them must outlive the calls
    nan = lambda *s: torch.full(s, float("nan"), dtype=torch.float32, device=dev)
    sz = _sizes(c)

    def area(n):
        if not n:
            return None
        t = torch.full((int(n),), 0xFF, dtype=torch.uint8, device=dev)
        keep.append(t)
        return t

    fs = area(sz.fwd_scratch if prec and H >= 128 else 0)
    wg = area(sz.wgrad_scratch if prec and H >= 128 else 0)
    asc = area(sz.attn_scratch)
    step_dev = torch.tensor([c.sdev], dtype=torch.int32, device=dev) if c.sdev is not None else None

    def drop(kind, site):
        d = L_.adt_dropout()
        d.enabled, d.p, d.seed, d.step, d.site = int(c.p > 0), c.p, SEED, STEP, site
        d.base = c.b0 * (nh * Lq if kind == "attn" else Lq * H)
        d.step_dev = step_dev.data_ptr() if step_dev is not None else None
        return d

    def acc(*s):
        """accumulated output: starts at known values; returns (device tensor, initial host copy)"""
        t = 0.25 * torch.randn(*s, generator=g)
        return t.to(dev), t

    out, init, names = {}, {}, {}

    def dev_params(blk, keys):
        ts = [inp[blk][k].to(dev) for k in keys]
        if wm:
            m = Mirror(ts, dev)
            keep.append(m)
            ts = m.views
            w = L_.adt_wmirror()
            w.base32, w.bf16 = m.flat.data_ptr(), m.bf16.data_ptr()
        else:
            w = L_.adt_wmirror()
        keep.extend(ts)
        return dict(zip(keys, ts)), w

    def grads(blk, keys):
        gs = {}
        for k in keys:
            gs[k], init[f"{blk}/g_{k}"] = acc(*inp[blk][k].shape)
            out[f"{blk}/g_{k}"] = gs[k]
        keep.extend(gs.values())
        return gs

    def call(fn, a, tag):
        with _Timed() as t:
            L_.check(getattr(lib, fn)(ctypes.byref(a), stream), fn)
        names[tag] = names.get(tag, []) + t.names

    def dbl(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        keep.append(t)
        return t

    # ---- encoder block
    e = inp["enc"]
    P, wme = dev_params("enc", ENC_PARAMS)
    x, ids = e["x"].to(dev), e["ids"].to(dev)
    keep.extend([x, ids])
    mw = lambda pre: L_.fill(L_.adt_mha_w(), in_w=P[pre + "in_w"], in_b=P[pre + "in_b"], out_w=P[pre + "out_w"], out_b=P[pre + "out_b"])
    attn = mw("")
    ffn = L_.fill(L_.adt_ffn_w(), w1=P["w1"], b1=P["b1"], w2=P["w2"], b2=P["b2"])
    sv = {k: nan(M, H) for k in ("q", "k", "v", "ctx", "y", "h1", "out")}
    sv["lse"], sv["rec"] = nan(B, nh, Lq), nan(M, nh, nh)
    nll = dbl(1.5) if extras else None
    da, d1, d2 = drop("attn", ENC_SITES[0]), drop("row", ENC_SITES[1]), drop("row", ENC_SITES[2])
    common = dict(x=x, ids=ids, ln1_w=P["ln1_w"], ln1_b=P["ln1_b"], attn=attn, ln2_w=P["ln2_w"], ln2_b=P["ln2_b"], ffn=ffn,
                  sparse_w=P["sp_w"], sparse_b=P["sp_b"], B=B, L=Lq, H=H, nh=nh, mask_mode=c.mask_mode, drop_attn=da, drop_ffn1=d1,
                  drop_ffn2=d2, precision=prec, wm=wme, attn_scratch=asc)
    for ph in ((1, 2) if phases[0] == 12 else (phases[0],)):
        a = L_.fill(L_.adt_enc_block_fwd_args(), nll_acc=nll, training=1, tc_scratch=fs, phase=ph, **common, **sv)
        call("adt_enc_block_fwd", a, "enc_fwd")
    sc = {k: nan(M, H) for k in ("dq", "dk", "dv", "dctx", "dy", "dx")}
    G = grads("enc", ENC_PARAMS)
    gm = lambda pre: L_.fill(L_.adt_mha_g(), in_w=G[pre + "in_w"], in_b=G[pre + "in_b"], out_w=G[pre + "out_w"], out_b=G[pre + "out_b"])
    ext = dict(dx_extra=e["dx_extra"].to(dev), drec=e["drec"].to(dev), nll_coef=e["nll_coef"]) if extras else dict(nll_coef=0.0)
    keep.extend(v for v in ext.values() if torch.is_tensor(v))
    dout = e["dout"].to(dev)
    keep.append(dout)
    a = L_.fill(L_.adt_enc_block_bwd_args(), dout=dout, wgrad_scratch=wg, g_ln1_w=G["ln1_w"], g_ln1_b=G["ln1_b"],
                g_attn=gm(""), g_ln2_w=G["ln2_w"], g_ln2_b=G["ln2_b"],
                g_ffn=L_.fill(L_.adt_ffn_g(), w1=G["w1"], b1=G["b1"], w2=G["w2"], b2=G["b2"]), g_sparse_w=G["sp_w"], g_sparse_b=G["sp_b"],
                **common, **{k: sv[k] for k in ("q", "k", "v", "ctx", "lse", "y", "h1")}, **sc, **ext)
    call("adt_enc_block_bwd", a, "enc_bwd")
    out.update({"enc/" + k: v for k, v in sv.items()})
    out.update({"enc/dx": sc["dx"], "enc/dctx": sc["dctx"], "enc/dy": sc["dy"]})
    if extras:
        out["enc/nll_acc"], init["enc/nll_acc"] = nll, torch.tensor([1.5], dtype=torch.float64)

    # ---- decoder block
    d = inp["dec"]
    P, wmd = dev_params("dec", DEC_PARAMS)
    x, feats = d["x"].to(dev), d["feats"].to(dev)
    slf, enc = mw("s_"), mw("e_")
    ffn = L_.fill(L_.adt_ffn_w(), w1=P["w1"], b1=P["b1"], w2=P["w2"], b2=P["b2"])
    sv = {k: nan(M, H) for k in ("d", "q1", "k1", "v1", "ctx1", "a", "q2", "k2", "v2", "ctx2", "c", "h1", "out")}
    sv["lse1"], sv["lse2"] = nan(B, nh, Lq), nan(B, nh, Lq)
    enc_in = d["enc_in"].to(dev) if extras else None
    mse = dbl(2.5) if extras else None
    ds, de = drop("attn", DEC_SITES[0]), drop("attn", DEC_SITES[1])
    d1, d2 = drop("row", DEC_SITES[2]), drop("row", DEC_SITES[3])
    common = dict(x=x, feats=feats, ids=ids, ln_w=P["ln_w"], ln_b=P["ln_b"], slf=slf, enc=enc, ffn=ffn, enc_in=enc_in, B=B, L=Lq, H=H,
                  nh=nh, mask_mode=c.mask_mode, drop_slf=ds, drop_enc=de, drop_ffn1=d1, drop_ffn2=d2, precision=prec, wm=wmd,
                  attn_scratch=asc)
    for ph in ((1, 2) if phases[1] == 12 else (phases[1],)):
        a = L_.fill(L_.adt_dec_block_fwd_args(), mse_acc=mse, training=1, tc_scratch=fs, phase=ph, **common, **sv)
        call("adt_dec_block_fwd", a, "dec_fwd")
    sc = {k: nan(M, H) for k in ("dq", "dk", "dv", "dctx", "dd", "dq2", "dk2", "dv2", "dctx2", "dx")}
    dfeats, init["dec/dfeats"] = acc(M, H)
    denc = nan(M, H) if extras else None
    G = grads("dec", DEC_PARAMS)
    dout = d["dout"].to(dev)
    keep.extend([x, feats, enc_in, dout, dfeats])
    for ph in ((2, 1) if phases[2] == 21 else (phases[2],)):
        a = L_.fill(L_.adt_dec_block_bwd_args(), mse_coef=d["mse_coef"] if extras else 0.0, dout=dout, denc=denc,
                    wgrad_scratch=wg, g_ln_w=G["ln_w"], g_ln_b=G["ln_b"], g_slf=gm("s_"), g_enc=gm("e_"),
                    g_ffn=L_.fill(L_.adt_ffn_g(), w1=G["w1"], b1=G["b1"], w2=G["w2"], b2=G["b2"]), dfeats=dfeats, phase=ph,
                    **common, **sv, **sc)
        call("adt_dec_block_bwd", a, "dec_bwd")
    out.update({"dec/" + k: v for k, v in sv.items()})
    out.update({"dec/dx": sc["dx"], "dec/dctx": sc["dctx"], "dec/dctx2": sc["dctx2"], "dec/dd": sc["dd"], "dec/dfeats": dfeats})
    if extras:
        out["dec/denc"], out["dec/mse_acc"] = denc, mse
        init["dec/mse_acc"] = torch.tensor([2.5], dtype=torch.float64)
    torch.cuda.synchronize()
    del keep
    res = {}
    for k, v in out.items():
        v = v.cpu()
        if k in init:
            v = v.double() - init[k].double()
        res[k] = v.numpy()
    res.update({"names/" + k: v for k, v in names.items()})
    return res
