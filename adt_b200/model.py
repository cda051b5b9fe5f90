"""SASRecADT on B200: the reference's nn.Module surface over the hand-written CUDA path.

Mirrors /root/reference/sasrec/model.py:8-97 (constructor arguments, `forward`, `predict`, parameter names and
shapes, so reference checkpoints load both ways and main.py/evolution.py can drive it unchanged), but every
device op is a call into libadt_b200.so (include/adt_b200.h).  Two ways in:

  * compat:  `model(u, seq, dec, pos, neg)` returns autograd-connected tensors exactly like the reference,
             so the caller's loss lines (sasrec/main.py:147-171) work as they are;
  * fused :  `model.engine.train_step(...)` (see trainer.py) runs forward, the fused loss epilogues, backward, the
             sort-then-segmented embedding backward and clip+Adam without autograd.

There is no CPU path: constructing the engine without the CUDA library / a CUDA device raises.
"""
import math
import numpy as np
import torch
import torch.nn as nn

from . import _lib as L


def _as_ids(a, dev):
    """host numpy / torch integer array [B,L] -> contiguous int32 device tensor."""
    if isinstance(a, torch.Tensor):
        return a.to(device=dev, dtype=torch.int32, non_blocking=True).contiguous()
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev, non_blocking=True)


def _check_ids(t, item_num, what):
    """ids feed raw-pointer kernels: an id outside [0, item_num] would be a silent out-of-bounds read where torch raises."""
    if t.numel():
        lo, hi = int(t.min()), int(t.max())
        if lo < 0 or hi > item_num:
            raise IndexError(f"{what}: item ids must lie in [0, {item_num}], got [{lo}, {hi}]")


class _MHA(nn.Module):
    """parameter holder with nn.MultiheadAttention's names/inits (sasrec/modules.py:168-218)."""

    def __init__(self, H):
        super().__init__()
        self.in_proj_weight = nn.Parameter(torch.empty(3 * H, H))
        self.in_proj_bias = nn.Parameter(torch.zeros(3 * H))
        self.out_proj = nn.Linear(H, H)
        nn.init.xavier_uniform_(self.in_proj_weight)
        nn.init.constant_(self.out_proj.bias, 0.0)


class _FFN(nn.Module):
    """PointWiseFeedForward parameters (sasrec/modules.py:618-627): Conv1d k=1 weights are [H,H,1]."""

    def __init__(self, H):
        super().__init__()
        self.conv1 = nn.Conv1d(H, H, kernel_size=1)
        self.conv2 = nn.Conv1d(H, H, kernel_size=1)


class _EncoderLayer(nn.Module):
    def __init__(self, H, nh):
        super().__init__()
        self.attention_layernorm = nn.LayerNorm(H, eps=1e-8)
        self.attention_layer = _MHA(H)
        self.forward_layernorm = nn.LayerNorm(H, eps=1e-8)
        self.forward_layer = _FFN(H)
        self.sparse = nn.Linear(H // nh, nh)


class _DecoderLayer(nn.Module):
    def __init__(self, H, nh):
        super().__init__()
        self.layer_norm = nn.LayerNorm(H, eps=1e-8)
        self.slf_attn = _MHA(H)
        self.enc_attn = _MHA(H)
        self.pos_ffn = _FFN(H)
        self.pos_ffn_layernorm = nn.LayerNorm(H, eps=1e-8)  # present but never applied (modules.py:663,673)


class _Encoder(nn.Module):
    def __init__(self, nl, H, nh):
        super().__init__()
        self.encoder_layers = nn.ModuleList(_EncoderLayer(H, nh) for _ in range(nl))


class _Decoder(nn.Module):
    def __init__(self, nl, H, nh):
        super().__init__()
        self.decoder_layers = nn.ModuleList(_DecoderLayer(H, nh) for _ in range(nl))


def _mha_w(m):
    return L.fill(L.adt_mha_w(), in_w=m.in_proj_weight, in_b=m.in_proj_bias, out_w=m.out_proj.weight, out_b=m.out_proj.bias)


def _ffn_w(m):
    return L.fill(L.adt_ffn_w(), w1=m.conv1.weight, b1=m.conv1.bias, w2=m.conv2.weight, b2=m.conv2.bias)


class Engine:
    """Owns workspaces and drives the C-ABI calls for one model on one device."""

    SITE_ENC_EMB = 0

    def __init__(self, model):
        self.m = model
        self.lib = L.lib()  # raises if the CUDA library is missing
        self.ws = {}
        self.drop_seed = 0
        self.drop_step = 0
        self.batch_offset = 0      # first global sample index of this rank (data parallel)
        self.global_rows = None    # M of the global batch (None -> local)
        self.gflat = None
        self.side_stream = None    # optional second stream: decoder work that is independent of the encoder runs beside it
        self.step_dev = None       # optional int32 device tensor: [0] is added to the dropout step at run time
        self.precision = 0         # 0: fp32 FFMA GEMM cores (reference precision) ; 1: bf16 tensor-core cores, fp32 accumulate
        self.use_mirror = True     # keep a bf16 mirror of the dense weights for the sequence-resident kernels (bf16 mode only)
        self.pflat = None
        self.mirror, self._mirror_key = None, None

    # ------------------------------------------------------------------ parameters / flat buffers
    def dev(self):
        return self.m.item_emb.weight.device

    def trainable(self):
        """(name, param) of every parameter that receives a gradient (pos_ffn_layernorm never does)."""
        return [(n, p) for n, p in self.m.named_parameters() if "pos_ffn_layernorm" not in n]

    def ensure_flat(self):
        """Re-home all trainable parameters as views of one flat fp32 buffer [dense..., item_emb] (16B aligned
        segments) with a matching flat gradient buffer: one allreduce / one Adam launch covers everything."""
        named = self.trainable()
        order = [x for x in named if x[0] != "item_emb.weight"] + [x for x in named if x[0] == "item_emb.weight"]
        offs, off = {}, 0
        for n, p in order:
            offs[n] = off
            off += (p.numel() + 7) // 8 * 8          # 8-element segments: 16-byte aligned in the bf16 mirror too (cp.async)
        dev = self.dev()
        ok = self.gflat is not None and self.pflat.device == dev and self.pflat.numel() == off and all(
            p.data_ptr() == self.pflat.data_ptr() + 4 * offs[n] for n, p in order)
        if not ok:
            pflat = torch.zeros(off, dtype=torch.float32, device=dev)
            for n, p in order:
                seg = pflat[offs[n]:offs[n] + p.numel()].view(p.shape)
                seg.copy_(p.data)
                p.data = seg
            self.pflat, self.gflat = pflat, torch.zeros_like(pflat)
            self.adam_m, self.adam_v = torch.zeros_like(pflat), torch.zeros_like(pflat)
            self.adam_t = 0
            self.offs, self.order = offs, order
            self.table_off = offs["item_emb.weight"]
            # bf16 mirror of the dense parameters (everything before the item table): the sequence-resident block kernels cp.async
            # their weight tiles from it; the fused trainer's Adam kernel keeps it current, everybody else through ensure_mirror()
            self.mirror = torch.zeros(self.table_off, dtype=torch.bfloat16, device=dev)
            self._mirror_key = None
        return self.offs

    def _param_key(self):
        return (self.pflat.data_ptr(), getattr(self.m, "_adt_param_version", 0), sum(p._version for _, p in self.order))

    def refresh_mirror(self):
        n = self.table_off
        L.check(self.lib.adt_to_bf16(L.ptr(self.pflat), L.ptr(self.mirror), L.ctypes.c_int64(n // 8), L.ctypes.c_int32(8), None, self._stream()),
                "adt_to_bf16")
        self._mirror_key = self._param_key()

    def ensure_mirror(self):
        """make the bf16 weight mirror current (host-side version check; not callable during graph capture).  Models that were
        never given a flat parameter buffer get one here (parameters become views of it; values unchanged)."""
        if not self.use_mirror:
            return
        self.ensure_flat()
        if self._mirror_key != self._param_key():
            self.refresh_mirror()

    def mirror_marked_current(self):
        """the fused trainer's Adam kernel has just rewritten the mirror together with the parameters"""
        self._mirror_key = self._param_key()

    def wm(self):
        """adt_wmirror for the kernels: the mirror when it is known to be current, else NULL (kernels convert from fp32)"""
        w = L.adt_wmirror()
        if self.use_mirror and self.gflat is not None and self._mirror_key is not None and (
                torch.cuda.is_current_stream_capturing() or self._mirror_key == self._param_key()):
            w.base32, w.bf16 = self.pflat.data_ptr(), self.mirror.data_ptr()
        return w

    def seq_kernels(self, Lq):
        m = self.m
        return bool(self.lib.adt_seq_kernels_apply(int(Lq), int(m.hidden), int(m.num_heads), int(self.precision)))

    def mirror_kernels(self, Lq):
        """kernels that read the bf16 weight mirror serve this shape: the sequence-resident block kernels, or the tcgen05 forward path of
        wide models (which otherwise converts every weight per call)"""
        return self.seq_kernels(Lq) or (bool(self.precision) and self.m.hidden >= 128)

    def grad_view(self, name):
        p = dict(self.order)[name]
        o = self.offs[name]
        return self.gflat[o:o + p.numel()].view(p.shape)

    # ------------------------------------------------------------------ workspaces
    def workspace(self, B, Lq):
        key = (B, Lq)
        w = self.ws.get(key)
        if w is not None:
            return w
        m, dev = self.m, self.dev()
        H, nh, nl = m.hidden, m.num_heads, m.num_layers
        M = B * Lq
        f = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
        w = {"B": B, "L": Lq, "M": M, "gen": 0}
        q = L.fill(L.adt_workspace_query(), B=B, L=Lq, H=H, nh=nh, nl=nl, K=1, n_splits=1)
        sz = L.adt_workspace_sizes()
        L.check(self.lib.adt_workspace_bytes(L.ctypes.byref(q), L.ctypes.byref(sz)), "adt_workspace_bytes")
        w["sizes"] = {k: int(getattr(sz, k)) for k, _ in sz._fields_}
        w["x"] = [f(M, H) for _ in range(nl + 1)]        # encoder stream: x[0]=embedding, x[l+1]=block l output
        w["xd"] = [f(M, H) for _ in range(nl + 1)]       # decoder stream
        w["enc"] = [{k: f(M, H) for k in ("q", "k", "v", "ctx", "y", "h1")} | {"lse": f(B, nh, Lq), "rec": f(M, nh, nh)}
                    for _ in range(nl)]
        w["dec"] = [{k: f(M, H) for k in ("d", "q1", "k1", "v1", "ctx1", "a", "q2", "k2", "v2", "ctx2", "c", "h1")} |
                    {"lse1": f(B, nh, Lq), "lse2": f(B, nh, Lq)} for _ in range(nl)]
        w["feats"], w["pos_logits"], w["neg_logits"] = f(M, H), f(M), f(M)
        w["acc"] = torch.zeros(8 + 2 * nl, dtype=torch.float64, device=dev)
        # backward scratch
        w["zero4"] = torch.empty(4, M, H, dtype=torch.float32, device=dev)   # dk, dv, dk2, dv2 scratch
        for k in ("dq", "dctx", "dres", "dq2", "dctx2", "dfeats", "dxa", "dxb", "dxd_a", "dxd_b"):
            w[k] = f(M, H)
        w["denc"] = [f(M, H) for _ in range(nl)]
        w["side"] = {k: f(M, H) for k in ("dq", "dk", "dv", "dctx", "dres")}   # decoder block 0 backward, run beside the encoder backward
        w["cpos"], w["cneg"] = f(M), f(M)
        # bf16 operand copies of the hoisted weight gradients (H >= 128 in the bf16 mode; one more for the side-stream half of decoder block 0)
        nwg = w["sizes"]["wgrad_scratch"] if self.precision else 0
        w["wg"] = torch.empty(nwg, dtype=torch.uint8, device=dev) if nwg else None
        w["side"]["wg"] = torch.empty(nwg, dtype=torch.uint8, device=dev) if nwg else None
        # bf16 operands of the tcgen05 forward path (same condition; the side-stream half of decoder block 0 owns a second one)
        nfs = w["sizes"]["fwd_scratch"] if self.precision else 0
        w["fs"] = torch.empty(nfs, dtype=torch.uint8, device=dev) if nfs else None
        w["side"]["fs"] = torch.empty(nfs, dtype=torch.uint8, device=dev) if nfs else None
        # bf16 operands of the fused flash attention (L > 256; again one more for the side-stream half of decoder block 0)
        nas = w["sizes"]["attn_scratch"]
        w["as"] = torch.empty(nas, dtype=torch.uint8, device=dev) if nas else None
        w["side"]["as"] = torch.empty(nas, dtype=torch.uint8, device=dev) if nas else None
        N = 4 * M
        i32 = lambda n: torch.empty(n, dtype=torch.int32, device=dev)
        w["keys"], w["vals"], w["keys_tmp"], w["vals_tmp"] = i32(N), i32(N), i32(N), i32(N)
        assert w["sizes"]["sort_keys"] == 16 * N
        w["hist"] = i32(w["sizes"]["sort_hist"] // 4)
        nb = w["sizes"]["scatter_flags"] // 4
        assert w["sizes"]["scatter_rows"] == 2 * nb * H * 4
        w["head"], w["tail"], w["has_tail"] = f(nb, H), f(nb, H), i32(nb)
        self.ws[key] = w
        return w

    # ------------------------------------------------------------------ dropout sites (SURVEY.md A.8 order)
    def _drop(self, site, kind, training, B, Lq):
        m = self.m
        d = L.adt_dropout()
        d.enabled = 1 if (training and m.dropout_p > 0.0) else 0
        d.p = float(m.dropout_p)
        d.seed = int(self.drop_seed)
        d.step = int(self.drop_step)
        d.step_dev = self.step_dev.data_ptr() if self.step_dev is not None else None
        d.site = int(site)
        per = m.num_heads * Lq if kind == "attn" else Lq * m.hidden   # attention sites: ROW offset ; row sites: element offset
        d.base = int(self.batch_offset) * per
        return d

    def _sites(self):
        nl = self.m.num_layers
        s = {"enc_emb": 0, "dec_emb": 1 + 3 * nl}
        for l in range(nl):
            s[("enc", l)] = (1 + 3 * l, 2 + 3 * l, 3 + 3 * l)
            b = 2 + 3 * nl + 4 * l
            s[("dec", l)] = (b, b + 1, b + 2, b + 3)
        return s

    def _stream(self):
        return L.ctypes.c_void_p(torch.cuda.current_stream(self.dev()).cuda_stream)

    # ------------------------------------------------------------------ forward
    def embed(self, ids, out, site, training, B, Lq):
        m = self.m
        a = L.fill(L.adt_embed_fwd_args(), ids=ids, item_emb=m.item_emb.weight, pos_emb=m.pos_emb.weight, x=out, B=B, L=Lq, H=m.hidden,
                   drop=self._drop(site, "row", training, B, Lq))
        L.check(self.lib.adt_embed_fwd(L.ctypes.byref(a), self._stream()), "adt_embed_fwd")

    def encode(self, seq, training, w, nll=False, last_phase=0, out_last=None):
        """embedding + encoder blocks (+ last LayerNorm into w['feats'] when pos is None handled by caller).
        last_phase=1 stops the LAST block after its attention (see encode_last); out_last: [B,H] buffer that receives the LAST
        block's output at the last position only (sequence-resident kernels)."""
        m = self.m
        B, Lq = w["B"], w["L"]
        sites = self._sites()
        wm = self.wm()
        self.embed(seq, w["x"][0], sites["enc_emb"], training, B, Lq)
        for l, layer in enumerate(m.encoder.encoder_layers):
            sv = w["enc"][l]
            sa, s1, s2 = sites[("enc", l)]
            last = l == m.num_layers - 1
            a = L.fill(L.adt_enc_block_fwd_args(), x=w["x"][l], ids=seq, phase=(last_phase if l == m.num_layers - 1 else 0),
                       wm=wm, out_last=(out_last if last else None), tc_scratch=w.get("fs"), attn_scratch=w.get("as"),
                       ln1_w=layer.attention_layernorm.weight, ln1_b=layer.attention_layernorm.bias, attn=_mha_w(layer.attention_layer),
                       ln2_w=layer.forward_layernorm.weight, ln2_b=layer.forward_layernorm.bias, ffn=_ffn_w(layer.forward_layer),
                       sparse_w=layer.sparse.weight, sparse_b=layer.sparse.bias,
                       q=sv["q"], k=sv["k"], v=sv["v"], ctx=sv["ctx"], lse=sv["lse"], y=sv["y"], h1=sv["h1"],
                       out=(None if (last and out_last is not None) else w["x"][l + 1]), rec=(sv["rec"] if training or out_last is None else None),
                       nll_acc=(w["acc"][3 + m.num_layers + l:] if (nll and m.num_heads > 1) else None),
                       B=B, L=Lq, H=m.hidden, nh=m.num_heads, training=int(training), mask_mode=0, precision=self.precision,
                       drop_attn=self._drop(sa, "attn", training, B, Lq), drop_ffn1=self._drop(s1, "row", training, B, Lq),
                       drop_ffn2=self._drop(s2, "row", training, B, Lq))
            L.check(self.lib.adt_enc_block_fwd(L.ctypes.byref(a), self._stream()), "adt_enc_block_fwd")

    def encode_last(self, seq, w):
        """eval-mode encoder + last LayerNorm for the LAST position of every sequence only (model.py:86-89 reads
        log_feats[:, -1, :]).  Blocks 0..nl-2 run in full; the last block still projects and attends over all rows (its
        keys/values are needed), but its row-wise tail (out-projection, residual, LayerNorms, FFN, pad mask) and the final
        LayerNorm run on the B last rows instead of B*L.  Returns feats [B, H] (a workspace buffer)."""
        m = self.m
        B, Lq, H, nl = w["B"], w["L"], m.hidden, m.num_layers
        ws = self.workspace(B, 1)
        if self.seq_kernels(Lq):
            # sequence-resident kernels: every block is one launch over whole sequences; the last one writes position L-1 only
            self.encode(seq, False, w, out_last=ws["x"][nl])
            self.final(ws, None, None, with_loss=False)
            return ws["feats"]
        self.encode(seq, False, w, last_phase=1)
        layer, sv, svs = m.encoder.encoder_layers[nl - 1], w["enc"][nl - 1], ws["enc"][nl - 1]
        ws["x"][nl - 1].copy_(w["x"][nl - 1].view(B, Lq, H)[:, Lq - 1])      # strided gathers of the last position
        svs["ctx"].copy_(sv["ctx"].view(B, Lq, H)[:, Lq - 1])
        ids_last = seq[:, Lq - 1].contiguous()
        nodrop = self._drop(0, "row", False, B, 1)
        # beyond H = 256 only the tcgen05 block path serves, at any row count: it runs phase 2 on the B last rows from its own scratch
        tc = {"wm": self.wm(), "tc_scratch": ws["fs"]} if H > 256 else {}
        a = L.fill(L.adt_enc_block_fwd_args(), x=ws["x"][nl - 1], ids=ids_last, phase=2, **tc,
                   ln1_w=layer.attention_layernorm.weight, ln1_b=layer.attention_layernorm.bias, attn=_mha_w(layer.attention_layer),
                   ln2_w=layer.forward_layernorm.weight, ln2_b=layer.forward_layernorm.bias, ffn=_ffn_w(layer.forward_layer),
                   sparse_w=layer.sparse.weight, sparse_b=layer.sparse.bias,
                   q=svs["q"], k=svs["k"], v=svs["v"], ctx=svs["ctx"], lse=svs["lse"], y=svs["y"], h1=svs["h1"],
                   out=ws["x"][nl], rec=svs["rec"], nll_acc=None,
                   B=B, L=1, H=H, nh=m.num_heads, training=0, mask_mode=0, precision=self.precision,
                   drop_attn=nodrop, drop_ffn1=nodrop, drop_ffn2=nodrop)
        L.check(self.lib.adt_enc_block_fwd(L.ctypes.byref(a), self._stream()), "adt_enc_block_fwd")
        self.final(ws, None, None, with_loss=False)
        return ws["feats"]

    def final(self, w, pos, neg, with_loss):
        m = self.m
        ln = m.last_layernorm if m.has_last_ln else None
        a = L.fill(L.adt_final_fwd_args(), x=w["x"][m.num_layers], ln_w=ln.weight if ln is not None else None,
                   ln_b=ln.bias if ln is not None else None, item_emb=m.item_emb.weight, pos=pos, neg=neg, feats=w["feats"],
                   pos_logits=w["pos_logits"], neg_logits=w["neg_logits"], acc=w["acc"] if with_loss else None, M=w["M"], H=m.hidden)
        L.check(self.lib.adt_final_logits_loss_fwd(L.ctypes.byref(a), self._stream()), "adt_final_logits_loss_fwd")

    def decode(self, dec, training, w, fused_mse, phases=(0,)):
        """phases=(0,): embedding + all decoder blocks.  phases=(1,): embedding + LN/self-attention of block 0 only (needs
        nothing from the encoder); phases=(2,): the rest.  (1,) then (2,) equals (0,)."""
        m = self.m
        B, Lq, nl = w["B"], w["L"], m.num_layers
        sites = self._sites()
        if phases[0] != 2:
            self.embed(dec, w["xd"][0], sites["dec_emb"], training, B, Lq)
        for j, layer in enumerate(m.decoder.decoder_layers):
            if phases[0] == 1 and j > 0:
                break
            sv = w["dec"][j]
            ss, se, s1, s2 = sites[("dec", j)]
            a = L.fill(L.adt_dec_block_fwd_args(), x=w["xd"][j], feats=w["feats"], ids=dec, wm=self.wm(),
                       tc_scratch=(w["side"]["fs"] if phases[0] == 1 else w["fs"]),     # phase 1 runs beside the encoder on the side stream
                       attn_scratch=(w["side"]["as"] if phases[0] == 1 else w["as"]),
                       ln_w=layer.layer_norm.weight, ln_b=layer.layer_norm.bias, slf=_mha_w(layer.slf_attn), enc=_mha_w(layer.enc_attn),
                       ffn=_ffn_w(layer.pos_ffn), enc_in=w["x"][nl - 1 - j] if fused_mse else None,
                       out=w["xd"][j + 1], mse_acc=(w["acc"][3 + j:] if fused_mse else None),
                       B=B, L=Lq, H=m.hidden, nh=m.num_heads, training=int(training), mask_mode=0, precision=self.precision,
                       drop_slf=self._drop(ss, "attn", training, B, Lq), drop_enc=self._drop(se, "attn", training, B, Lq),
                       drop_ffn1=self._drop(s1, "row", training, B, Lq), drop_ffn2=self._drop(s2, "row", training, B, Lq),
                       phase=(phases[0] if j == 0 else 0),
                       **{k: sv[k] for k in ("d", "q1", "k1", "v1", "ctx1", "lse1", "a", "q2", "k2", "v2", "ctx2", "lse2", "c", "h1")})
            L.check(self.lib.adt_dec_block_fwd(L.ctypes.byref(a), self._stream()), "adt_dec_block_fwd")

    def forward(self, seq, dec, pos, neg, training, fused_loss):
        """Full forward of model.py:67-81.  fused_loss=True also accumulates BCE / MSE / NLL sums into w['acc']."""
        B, Lq = seq.shape
        w = self.workspace(B, Lq)
        w["gen"] += 1          # every forward of this shape overwrites the saved activations (see _CompatForward.backward)
        if fused_loss:
            w["acc"].zero_()
        side = self.side_stream
        if side is None:
            self.encode(seq, training, w, nll=fused_loss)
            self.final(w, pos, neg, with_loss=fused_loss)
            self.decode(dec, training, w, fused_mse=fused_loss)
            return w
        # the decoder's embedding + first self-attention do not depend on the encoder: run them beside it
        cur = torch.cuda.current_stream(self.dev())
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            self.decode(dec, training, w, fused_mse=fused_loss, phases=(1,))
        self.encode(seq, training, w, nll=fused_loss)
        self.final(w, pos, neg, with_loss=fused_loss)       # writes the encoder features the cross-attention reads
        cur.wait_stream(side)
        self.decode(dec, training, w, fused_mse=fused_loss, phases=(2,))
        return w

    # ------------------------------------------------------------------ backward
    def sort_ids(self, seq, dec, pos, neg, w):
        a = L.fill(L.adt_embed_sort_args(), seq=seq, dec=dec, pos=pos, neg=neg, M=w["M"], max_id=self.m.item_num,
                   keys=w["keys"], vals=w["vals"], keys_tmp=w["keys_tmp"], vals_tmp=w["vals_tmp"], hist=w["hist"])
        L.check(self.lib.adt_embed_sort(L.ctypes.byref(a), self._stream()), "adt_embed_sort")

    def backward(self, seq, dec, pos, neg, w, grads, lambdas1=None, lambdas2=None, ext=None, n_valid=None):
        """Backward of the whole step into `grads` (name -> tensor, ACCUMULATED).
        fused mode : lambdas1/lambdas2 given -> BCE (mean over n_valid), lambda1*MSE and lambda2*NLL adjoints are
                     generated inside the kernels (main.py:152-169 incl. the stale-index quirk B1).
        compat mode: ext = dict(dpl, dnl, denc_in[list], ddec_out[list, per decoder layer], drec[list]) external grads.
        Sorting of the lookup ids must have been issued (sort_ids)."""
        m = self.m
        B, Lq, M, H, nh, nl = w["B"], w["L"], w["M"], m.hidden, m.num_heads, m.num_layers
        Mg = self.global_rows or M
        sites = self._sites()
        fused = lambdas1 is not None
        ext = ext or {}
        g = grads
        mg = lambda pre: L.fill(L.adt_mha_g(), in_w=g[pre + "in_proj_weight"], in_b=g[pre + "in_proj_bias"],
                                out_w=g[pre + "out_proj.weight"], out_b=g[pre + "out_proj.bias"])
        fg = lambda pre: L.fill(L.adt_ffn_g(), w1=g[pre + "conv1.weight"], b1=g[pre + "conv1.bias"], w2=g[pre + "conv2.weight"],
                                b2=g[pre + "conv2.bias"])
        z4 = w["zero4"]
        side = self.side_stream
        w["dfeats"].zero_()
        # ---- decoder blocks, last to first
        dxd, bufs = None, [w["dxd_a"], w["dxd_b"]]
        for j in reversed(range(nl)):
            layer, sv = m.decoder.decoder_layers[j], w["dec"][j]
            pre = f"decoder.decoder_layers.{j}."
            ss, se, s1, s2 = sites[("dec", j)]
            dout = dxd
            eo = ext.get("ddec_out")
            if eo is not None and eo[j] is not None:
                dout = eo[j] if dout is None else dout + eo[j]
            i_enc = nl - 1 - j
            out_dx = bufs[j % 2]
            split = side is not None and j == 0
            sb = w["side"] if split else None
            a = L.fill(L.adt_dec_block_bwd_args(), x=w["xd"][j], feats=w["feats"], ids=dec, wm=self.wm(),
                       ln_w=layer.layer_norm.weight, ln_b=layer.layer_norm.bias, slf=_mha_w(layer.slf_attn), enc=_mha_w(layer.enc_attn),
                       ffn=_ffn_w(layer.pos_ffn), out=w["xd"][j + 1], enc_in=w["x"][i_enc] if fused else None,
                       mse_coef=(float(lambdas1[i_enc]) * 2.0 / (Mg * H)) if fused else 0.0,
                       dout=dout, denc=w["denc"][i_enc] if fused else None,
                       dq=sb["dq"] if split else w["dq"], dk=sb["dk"] if split else z4[0], dv=sb["dv"] if split else z4[1],
                       dctx=sb["dctx"] if split else w["dctx"], dd=sb["dres"] if split else w["dres"],
                       dq2=w["dq2"], dk2=z4[2], dv2=z4[3], dctx2=w["dctx2"], phase=2 if split else 0, wgrad_scratch=w["wg"], attn_scratch=w["as"],
                       dfeats=w["dfeats"], dx=out_dx, g_ln_w=g[pre + "layer_norm.weight"], g_ln_b=g[pre + "layer_norm.bias"],
                       g_slf=mg(pre + "slf_attn."), g_enc=mg(pre + "enc_attn."), g_ffn=fg(pre + "pos_ffn."),
                       B=B, L=Lq, H=H, nh=nh, mask_mode=0, precision=self.precision,
                       drop_slf=self._drop(ss, "attn", True, B, Lq), drop_enc=self._drop(se, "attn", True, B, Lq),
                       drop_ffn1=self._drop(s1, "row", True, B, Lq), drop_ffn2=self._drop(s2, "row", True, B, Lq),
                       **{k: sv[k] for k in ("d", "q1", "k1", "v1", "ctx1", "lse1", "a", "q2", "k2", "v2", "ctx2", "lse2", "c", "h1")})
            L.check(self.lib.adt_dec_block_bwd(L.ctypes.byref(a), self._stream()), "adt_dec_block_bwd")
            if split:   # self-attention + LN adjoints of block 0 feed only the decoder embedding: beside the encoder backward
                cur = torch.cuda.current_stream(self.dev())
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    a.phase = 1
                    a.wgrad_scratch = sb["wg"].data_ptr() if sb["wg"] is not None else None
                    a.attn_scratch = sb["as"].data_ptr() if sb["as"] is not None else None
                    L.check(self.lib.adt_dec_block_bwd(L.ctypes.byref(a), self._stream()), "adt_dec_block_bwd")
            dxd = out_dx
        dx_dec_emb = dxd
        # ---- last LayerNorm + logits + BCE
        ln = m.last_layernorm if m.has_last_ln else None
        if n_valid is None:
            n_valid = w["acc"][2:3]
        a = L.fill(L.adt_final_bwd_args(), x=w["x"][nl], ln_w=ln.weight if ln is not None else None, item_emb=m.item_emb.weight,
                   pos=pos, neg=neg, pos_logits=w["pos_logits"], neg_logits=w["neg_logits"], dfeats_in=w["dfeats"], n_valid=n_valid,
                   bce_weight=1.0 if fused else 0.0, dpl_ext=ext.get("dpl"), dnl_ext=ext.get("dnl"), dx=w["dxa"], cpos=w["cpos"],
                   cneg=w["cneg"], g_ln_w=g["last_layernorm.weight"] if ln is not None else None,
                   g_ln_b=g["last_layernorm.bias"] if ln is not None else None, M=M, H=H)
        L.check(self.lib.adt_final_logits_loss_bwd(L.ctypes.byref(a), self._stream()), "adt_final_logits_loss_bwd")
        # ---- encoder blocks, last to first
        dx, other = w["dxa"], w["dxb"]
        for l in reversed(range(nl)):
            layer, sv = m.encoder.encoder_layers[l], w["enc"][l]
            pre = f"encoder.encoder_layers.{l}."
            sa, s1, s2 = sites[("enc", l)]
            ei = ext.get("denc_in")
            dout = dx   # already contains the external grad wrt x[l+1] (added as dx_extra of block l+1)
            dx_extra = w["denc"][l] if fused else (ei[l] if ei is not None else None)
            dr = ext.get("drec")
            a = L.fill(L.adt_enc_block_bwd_args(), x=w["x"][l], ids=seq, wm=self.wm(),
                       ln1_w=layer.attention_layernorm.weight, ln1_b=layer.attention_layernorm.bias, attn=_mha_w(layer.attention_layer),
                       ln2_w=layer.forward_layernorm.weight, ln2_b=layer.forward_layernorm.bias, ffn=_ffn_w(layer.forward_layer),
                       sparse_w=layer.sparse.weight, sparse_b=layer.sparse.bias,
                       q=sv["q"], k=sv["k"], v=sv["v"], ctx=sv["ctx"], lse=sv["lse"], y=sv["y"], h1=sv["h1"],
                       dout=dout, dx_extra=dx_extra, drec=dr[l] if dr is not None else None,
                       nll_coef=(float(lambdas2[nl - 1]) / (Mg * nh)) if (fused and nh > 1) else 0.0,
                       dq=w["dq"], dk=z4[0], dv=z4[1], dctx=w["dctx"], dy=w["dres"], dx=other, wgrad_scratch=w["wg"], attn_scratch=w["as"],
                       g_ln1_w=g[pre + "attention_layernorm.weight"], g_ln1_b=g[pre + "attention_layernorm.bias"],
                       g_attn=mg(pre + "attention_layer."), g_ln2_w=g[pre + "forward_layernorm.weight"],
                       g_ln2_b=g[pre + "forward_layernorm.bias"], g_ffn=fg(pre + "forward_layer."),
                       g_sparse_w=g[pre + "sparse.weight"], g_sparse_b=g[pre + "sparse.bias"],
                       B=B, L=Lq, H=H, nh=nh, mask_mode=0, precision=self.precision,
                       drop_attn=self._drop(sa, "attn", True, B, Lq), drop_ffn1=self._drop(s1, "row", True, B, Lq),
                       drop_ffn2=self._drop(s2, "row", True, B, Lq))
            L.check(self.lib.adt_enc_block_bwd(L.ctypes.byref(a), self._stream()), "adt_enc_block_bwd")
            dx, other = other, dx
        # ---- embeddings: sorted segmented scatter-add into the table, batch reduction into pos_emb
        if side is not None:
            torch.cuda.current_stream(self.dev()).wait_stream(side)
        a = L.fill(L.adt_embed_bwd_args(), keys=w["keys"], vals=w["vals"], seq=seq, dec=dec, B=B, L=Lq, H=H,
                   dx_enc=dx, dx_dec=dx_dec_emb, feats=w["feats"], cpos=w["cpos"], cneg=w["cneg"],
                   drop_enc=self._drop(sites["enc_emb"], "row", True, B, Lq), drop_dec=self._drop(sites["dec_emb"], "row", True, B, Lq),
                   d_item_emb=g["item_emb.weight"], d_pos_emb=g["pos_emb.weight"], head=w["head"], tail=w["tail"], has_tail=w["has_tail"])
        L.check(self.lib.adt_embed_bwd(L.ctypes.byref(a), self._stream()), "adt_embed_bwd")

    def loss_from_acc(self, w, lambdas1, lambdas2, weight_decay, emb_norm, acc=None):
        """Assemble main.py:152-170's scalar from the accumulators (host side, float64)."""
        m = self.m
        if acc is None:
            acc = w["acc"].tolist()
        Mg = self.global_rows or w["M"]
        nl, H, nh = m.num_layers, m.hidden, m.num_heads
        n = max(acc[2], 1.0)
        total = acc[0] / n + acc[1] / n
        for j in range(nl):
            total += lambdas1[nl - 1 - j] * acc[3 + j] / (Mg * H)
        if nh > 1:
            for l in range(nl):
                total += lambdas2[nl - 1] * acc[3 + nl + l] / (Mg * nh)
        return total + weight_decay * emb_norm


class _CompatForward(torch.autograd.Function):
    """autograd bridge for the reference-style `forward` (main.py:146-171 builds the loss itself)."""

    @staticmethod
    def forward(ctx, model, seq, dec, pos, neg, *params):
        eng = model.engine
        training = model.training
        w = eng.forward(seq, dec, pos, neg, training, fused_loss=False)
        if training:
            eng.sort_ids(seq, dec, pos, neg, w)
        ctx.model, ctx.ids, ctx.w = model, (seq, dec, pos, neg), w
        ctx.gen, ctx.drop_step = w["gen"], eng.drop_step
        nl, nh = model.num_layers, model.num_heads
        B, Lq = seq.shape
        H = model.hidden
        outs = [w["pos_logits"].view(B, Lq).clone(), w["neg_logits"].view(B, Lq).clone()]
        outs += [w["x"][l].view(B, Lq, H).clone() for l in range(nl)]
        outs += [w["xd"][j + 1].view(B, Lq, H).clone() for j in range(nl)]
        outs += [w["enc"][l]["rec"].view(B, Lq, nh, nh).clone() for l in range(nl)]
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gouts):
        model, w = ctx.model, ctx.w
        eng = model.engine
        nl = model.num_layers
        seq, dec, pos, neg = ctx.ids
        names = [n for n, _ in model.named_parameters()]
        grads = {n: torch.zeros_like(p) for n, p in model.named_parameters()}
        H = model.hidden
        c = lambda t: None if t is None else t.contiguous().float()
        c2 = lambda t: None if t is None else t.contiguous().float().view(-1, H)
        ext = {"dpl": c(gouts[0]), "dnl": c(gouts[1]), "denc_in": [c2(t) for t in gouts[2:2 + nl]],
               "ddec_out": [c2(t) for t in gouts[2 + nl:2 + 2 * nl]], "drec": [c(t) for t in gouts[2 + 2 * nl:2 + 3 * nl]]}
        if model.num_heads == 1:
            ext["drec"] = None
        if w["gen"] != ctx.gen:
            raise L.AdtError("SASRecADT: the saved activations of this forward were overwritten by a later forward/predict of the same "
                             "[B, L] shape before backward() ran (the engine keeps ONE workspace per shape): call backward() first")
        cur_step, eng.drop_step = eng.drop_step, ctx.drop_step      # the adjoints re-draw the masks of THIS forward
        try:
            eng.backward(seq, dec, pos, neg, w, grads, ext=ext)
        finally:
            eng.drop_step = cur_step
        return (None, None, None, None, None) + tuple(grads[n] for n in names)


class SASRecADT(nn.Module):
    """Drop-in for /root/reference/sasrec/model.py:7 `SASRecADT(user_num, item_num, args)`."""

    has_last_ln = True
    check_ids = True      # host-side range check of the ids (one min/max reduction per call); the fused trainer never pays it

    def __init__(self, user_num, item_num, args):
        super().__init__()
        self.user_num, self.item_num = user_num, item_num
        self.dev = args.device
        self.num_heads, self.maxlen, self.num_layers = args.num_heads, args.maxlen, args.num_layers
        self.hidden, self.dropout_p = args.hidden_units, float(args.dropout)
        H = args.hidden_units
        self.item_emb = nn.Embedding(item_num + 1, H, padding_idx=0)
        self.pos_emb = nn.Embedding(args.maxlen, H)
        self.emb_dropout = nn.Dropout(p=args.dropout)
        self.encoder = _Encoder(args.num_layers, H, args.num_heads)
        self.decoder = _Decoder(args.num_layers, H, args.num_heads)
        if self.has_last_ln:
            self.last_layernorm = nn.LayerNorm(H, eps=1e-8)
        self.args = args
        self._engine = None

    @property
    def engine(self):
        if self._engine is None:
            if self.item_emb.weight.device.type != "cuda":
                raise L.AdtError("adt_b200.SASRecADT runs on CUDA only (no CPU fallback): call .to('cuda') first")
            self._engine = Engine(self)
        return self._engine

    # -- reference API -------------------------------------------------------------------------
    def forward(self, user_ids, log_seqs, dec_seqs, pos_seqs, neg_seqs):
        """model.py:67-81 -> (pos_logits, neg_logits, enc_inputs[nl], dec_outputs[nl] reversed, rec_ind[nl])."""
        dev = self.item_emb.weight.device
        seq, dec, pos, neg = (_as_ids(a, dev) for a in (log_seqs, dec_seqs, pos_seqs, neg_seqs))
        if self.check_ids:
            for t, what in ((seq, "log_seqs"), (dec, "dec_seqs"), (pos, "pos_seqs"), (neg, "neg_seqs")):
                _check_ids(t, self.item_num, what)
        params = [p for _, p in self.named_parameters()]
        outs = _CompatForward.apply(self, seq, dec, pos, neg, *params)
        eng = self.engine
        if self.training and eng.step_dev is None:
            eng.drop_step += 1     # a fresh dropout stream for every training forward (the fused trainer advances step_dev instead)
        nl = self.num_layers
        B, Lq = seq.shape
        enc_in = list(outs[2:2 + nl])
        dec_out = list(outs[2 + nl:2 + 2 * nl])
        dec_out.reverse()  # modules.py:756
        # modules.py:517-518 views the [L,B,H] context buffer as [B,L,nh,hd]: a pure row permutation of the true rows
        rec = [r.transpose(0, 1).contiguous().view(B, Lq, self.num_heads, self.num_heads) for r in outs[2 + 2 * nl:2 + 3 * nl]]
        return outs[0], outs[1], enc_in, dec_out, rec

    @torch.no_grad()
    def predict(self, user_ids, log_seqs, item_indices, full=False):
        """model.py:83-97: logits of the last position against candidates ([B,C], or one shared 1-D list [C] as utils.evaluate /
        evaluate_valid pass it) or against the whole table [B,I+1].  Scoring runs in libadt_b200.so (adt_score_full /
        adt_candidate_scores), not in a torch matmul."""
        dev = self.item_emb.weight.device
        seq = _as_ids(log_seqs, dev)
        if self.check_ids:
            _check_ids(seq, self.item_num, "log_seqs")
        final = self.final_feats(seq)
        return score_candidates(self.item_emb.weight, final, item_indices, full, check=self.check_ids)

    @torch.no_grad()
    def final_feats(self, seq):
        """eval-mode encoder -> features of the last position [B,H] (model.py:86-89)."""
        eng = self.engine
        B, Lq = seq.shape
        w = eng.workspace(B, Lq)
        if eng.precision and eng.mirror_kernels(Lq) and not torch.cuda.is_current_stream_capturing():
            eng.ensure_mirror()
        if Lq > 1 and self.num_layers >= 1:
            return eng.encode_last(seq, w).clone()
        eng.encode(seq, False, w)
        eng.final(w, None, None, with_loss=False)
        return w["feats"].view(B, Lq, self.hidden)[:, -1, :].contiguous()


@torch.no_grad()
def score_candidates(E, final, item_indices, full, check=True, want_rank=False, metric_acc=None):
    """shared tail of predict(): final [B,H] against the table E [I+1,H].  Returns logits [B,C] / [B,I+1]
    (and the rank of column 0 when want_rank)."""
    lib = L.lib()
    dev = E.device
    B, H = final.shape
    st = L.ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    final = final.contiguous()
    if full:
        out = torch.empty(B, E.shape[0], dtype=torch.float32, device=dev)
        L.check(lib.adt_score_full(L.ptr(final), L.ctypes.c_int32(B), L.ctypes.c_int32(H), L.ptr(E), L.ctypes.c_int32(E.shape[0]),
                                   L.ctypes.c_int32(0), L.ptr(out), L.ctypes.c_int64(E.shape[0]), st), "adt_score_full")
        return out
    idx = _as_ids(item_indices, dev)
    if check:
        _check_ids(idx, E.shape[0] - 1, "item_indices")
    if idx.dim() == 1:
        stride, C = 0, idx.shape[0]
    else:
        if idx.shape[0] != B:
            raise ValueError(f"item_indices must be [C] or [{B}, C], got {tuple(idx.shape)}")
        stride, C = idx.shape[1], idx.shape[1]
    out = torch.empty(B, C, dtype=torch.float32, device=dev)
    rank = torch.empty(B, dtype=torch.int32, device=dev) if want_rank else None
    a = L.fill(L.adt_candidate_scores_args(), feats=final, item_emb=E, idx=idx, scores=out, rank=rank, metric_acc=metric_acc,
               idx_stride=stride, U=B, H=H, C=C, n_rows=E.shape[0])
    L.check(lib.adt_candidate_scores(L.ctypes.byref(a), st), "adt_candidate_scores")
    return (out, rank) if want_rank else out
