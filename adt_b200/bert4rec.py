"""Bert4Rec-ADT on B200 (SURVEY 8a row a19): the reference's BertModel surface composed from libadt_b200.so ops.

Mirrors /root/reference/bert4rec/model/bert.py:8-116 (constructor args, `forward(src_ids, dec_ids, seq_pos_ids,
seq_sent_ids, deq_pos_ids, deq_sent_ids)`, `predict`, parameter names/shapes) and model/modules.py (BertEmbedding,
post-LN encoder/decoder layers with separate q/k/v/out Linear, GELU FFN, per-head classifier).  Bidirectional
attention with the key-padding mask runs in the same attention kernel as SASRec (mask_mode 1).

`fused_loss` is the B200 training entry: the vocabulary head and the cross entropy are evaluated ONLY on the positions
that carry a label (~mask_prob of them) instead of the reference's [B*L, V] logits tensor (bert.py:80-90 +
trainer.py:112-115), in column blocks of the tied item table.  From FUSED_HEAD_MIN_VOCAB items on (bf16 mode, sm_100) the head and the
cross entropy run fused (ops.linear_cross_entropy): the scores stay on chip, only a per-row log-sum-exp is kept for the backward.
"""
import ctypes
import math
import numpy as np
import torch
import torch.nn as nn

from . import _lib as L
from .blocks import DropCfg
from .ops import AttnFn, DrlFn, Gather3Fn, linear, linear_cross_entropy, no_drop

# vocabulary size (itemnum + 100) from which fused_loss runs the fused tcgen05 head + cross entropy (adt_linear_ce_*) instead of the
# [R, V] logits + MaskedCE: at C3 (V 26,844) the materialising path is what runs; at 1M items its [R, V] fp32 tensors no longer fit
FUSED_HEAD_MIN_VOCAB = 65536


def _ids(a, dev):
    if isinstance(a, torch.Tensor):
        return a.to(device=dev, dtype=torch.int32).contiguous()
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)


class _BertEmbedding(nn.Module):
    def __init__(self, vocab, type_vocab, maxlen, H, dropout):
        super().__init__()
        self.word_emb = nn.Embedding(vocab, H, padding_idx=0)
        self.pos_emb = nn.Embedding(maxlen, H, padding_idx=0)
        self.sent_emb = nn.Embedding(type_vocab, H, padding_idx=0)
        self.layer_norm = nn.LayerNorm(H, eps=1e-5)
        self.dropout = nn.Dropout(p=dropout)

    def get_item_emb(self):
        return self.word_emb.weight


class _MHA(nn.Module):
    def __init__(self, H):
        super().__init__()
        self.query_transfer, self.key_transfer = nn.Linear(H, H), nn.Linear(H, H)
        self.value_transfer, self.out_transfer = nn.Linear(H, H), nn.Linear(H, H)


class _DRL(nn.Module):
    def __init__(self, H, p):
        super().__init__()
        self.dropout = nn.Dropout(p=p)
        self.layer_norm = nn.LayerNorm(H, eps=1e-5)


class _FFN(nn.Module):
    def __init__(self, H, inner):
        super().__init__()
        self.act = nn.GELU()
        self.fc1, self.fc2 = nn.Linear(H, inner), nn.Linear(inner, H)


class _EncLayer(nn.Module):
    def __init__(self, H, nh, inner, pa):
        super().__init__()
        self.multi_head_attention = _MHA(H)
        self.drop_residual_normalize_layer_after_multi = _DRL(H, pa)
        self.ffn = _FFN(H, inner)
        self.drop_residual_normalize_layer_final = _DRL(H, pa)
        self.head_classifier = nn.Linear(H // nh, nh)


class _DecLayer(nn.Module):
    def __init__(self, H, nh, inner, pa):
        super().__init__()
        self.dec_multi_head_attention = _MHA(H)
        self.drop_residual_normalize_layer_after_multi = _DRL(H, pa)
        self.src_dec_attention = _MHA(H)
        self.drop_residual_normalize_layer_after_src_dec = _DRL(H, pa)
        self.ffn = _FFN(H, inner)
        self.drop_residual_normalize_layer_final = _DRL(H, pa)


class _Stack(nn.Module):
    def __init__(self, name, layers):
        super().__init__()
        setattr(self, name, nn.ModuleList(layers))


class BertModel(nn.Module):
    def __init__(self, usernum, itemnum, args):
        super().__init__()
        self.usernum, self.itemnum = usernum, itemnum
        self.maxlen, self.num_heads, self.num_layers = args.maxlen, args.num_heads, args.num_layers
        self.dev = args.device
        self.dropout = float(args.dropout)
        self.attention_dropout = float(args.attention_dropout)
        self.hidden_units = H = args.hidden_units
        nh, inner = args.num_heads, args.inner_units
        self.item_emb = _BertEmbedding(itemnum + 100, args.type_vocab_size, args.maxlen, H, args.dropout)
        self.encoder = _Stack("encoder_layers", [_EncLayer(H, nh, inner, args.attention_dropout) for _ in range(args.num_layers)])
        self.decoder = _Stack("decoder_layers", [_DecLayer(H, nh, inner, args.attention_dropout) for _ in range(args.num_layers)])
        self.mask_trans_feat = nn.Linear(H, H)
        self.act = nn.GELU()
        self.mask_bias = nn.Parameter(torch.zeros(itemnum + 100))
        self.mask_layer_norm = nn.LayerNorm(H, eps=1e-5)
        self.drop_seed, self.drop_step, self.precision = 0, 0, 0
        self.step_dev = None      # optional device-side dropout step counter (adt_b200.dp.GraphedStep)
        self._scorers = {}        # (K, device) -> CatalogScorer of full_sort_topk (keeps its bf16 table and scratch between calls)
        L.lib()

    # ------------------------------------------------------------------------------------------
    def _check(self):
        if self.mask_bias.device.type != "cuda":
            raise L.AdtError("adt_b200.BertModel runs on CUDA only (no CPU fallback): call .to('cuda') first")

    def _drop(self, dc, kind, p, Lq):
        """next dropout site with probability p (two different p's on this path: dropout / attention_dropout)."""
        old = dc.p
        dc.p = p
        d = dc.next(kind, self.num_heads, Lq, self.hidden_units)
        dc.p = old
        return d

    def _mha(self, m, q_in, kv_in, key_ids, B, Lq, dc):
        H, nh, pr = self.hidden_units, self.num_heads, self.precision
        scale = 1.0 / math.sqrt(H // nh)
        q = linear(q_in, m.query_transfer.weight, m.query_transfer.bias, 0, scale, pr)
        k = linear(kv_in, m.key_transfer.weight, m.key_transfer.bias, 0, 1.0, pr)
        v = linear(kv_in, m.value_transfer.weight, m.value_transfer.bias, 0, 1.0, pr)
        d = self._drop(dc, "attn", self.attention_dropout, Lq)
        ctx = AttnFn.apply(q, k, v, key_ids, (B, Lq, nh, 1), d, dc.training, pr)
        return linear(ctx, m.out_transfer.weight, m.out_transfer.bias, 0, 1.0, pr), ctx

    def _drl(self, m, out, prev, dc, Lq):
        d = self._drop(dc, "row", self.attention_dropout, Lq)
        return DrlFn.apply(out, prev, m.layer_norm.weight, m.layer_norm.bias, 0, 1e-5, d)

    def _ffn(self, m, x):
        h = linear(x, m.fc1.weight, m.fc1.bias, 2, 1.0, self.precision)
        return linear(h, m.fc2.weight, m.fc2.bias, 0, 1.0, self.precision)

    def _embed(self, ids, pos_ids, sent_ids, dc, Lq):
        e = self.item_emb
        s = Gather3Fn.apply(ids, pos_ids, sent_ids, e.word_emb.weight, e.pos_emb.weight, e.sent_emb.weight)
        d = self._drop(dc, "row", self.dropout, Lq)
        return DrlFn.apply(s, None, e.layer_norm.weight, e.layer_norm.bias, 1, 1e-5, d)

    def _encode(self, src, pos_ids, sent_ids, dc):
        B, Lq = src.shape
        nh, H = self.num_heads, self.hidden_units
        x = self._embed(src, pos_ids, sent_ids, dc, Lq)
        enc_inputs, inds = [], []
        for layer in self.encoder.encoder_layers:
            enc_inputs.append(x)
            m, ctx = self._mha(layer.multi_head_attention, x, x, src, B, Lq, dc)
            h = self._drl(layer.drop_residual_normalize_layer_after_multi, m, x, dc, Lq)
            x = self._drl(layer.drop_residual_normalize_layer_final, self._ffn(layer.ffn, h), h, dc, Lq)
            logit = linear(ctx.view(B * Lq * nh, H // nh), layer.head_classifier.weight, layer.head_classifier.bias, 0, 1.0, 0)
            inds.append(torch.log_softmax(logit.view(B, Lq, nh, nh), dim=3))   # modules.py:213
        return x, enc_inputs, inds

    def _decode(self, dec, pos_ids, sent_ids, feats, src, dc):
        B, Lq = dec.shape
        y = self._embed(dec, pos_ids, sent_ids, dc, Lq)
        outs = []
        for layer in self.decoder.decoder_layers:
            m, _ = self._mha(layer.dec_multi_head_attention, y, y, dec, B, Lq, dc)
            y = self._drl(layer.drop_residual_normalize_layer_after_multi, m, y, dc, Lq)
            m, _ = self._mha(layer.src_dec_attention, y, feats, src, B, Lq, dc)
            y = self._drl(layer.drop_residual_normalize_layer_after_src_dec, m, y, dc, Lq)
            y = self._drl(layer.drop_residual_normalize_layer_final, self._ffn(layer.ffn, y), y, dc, Lq)
            outs.append(y)
        outs.reverse()
        return outs

    def _head_hidden(self, rows):
        """bert.py:81-86 on a set of rows [R,H]: Linear -> GELU -> LayerNorm."""
        h = linear(rows, self.mask_trans_feat.weight, self.mask_trans_feat.bias, 2, 1.0, self.precision)
        return DrlFn.apply(h, None, self.mask_layer_norm.weight, self.mask_layer_norm.bias, 0, 1e-5, no_drop())

    def downstream(self, feats_rows):
        """bert.py:80-90 -> logits [R, V] (tied item table + mask_bias)."""
        h = self._head_hidden(feats_rows)
        return linear(h, self.item_emb.word_emb.weight, self.mask_bias, 0, 1.0, self.precision)

    def _body(self, src_ids, dec_ids, seq_pos_ids, seq_sent_ids, deq_pos_ids, deq_sent_ids):
        self._check()
        dev = self.mask_bias.device
        src, dec = _ids(src_ids, dev), _ids(dec_ids, dev)
        sp, ss, dp, ds = (_ids(a, dev) for a in (seq_pos_ids, seq_sent_ids, deq_pos_ids, deq_sent_ids))
        dc = DropCfg(self.dropout, self.drop_seed, self.drop_step, self.training, step_dev=self.step_dev)
        feats, enc_inputs, inds = self._encode(src, sp, ss, dc)
        dec_outs = self._decode(dec, dp, ds, feats, src, dc)
        if self.training:
            self.drop_step += 1
        return feats, enc_inputs, dec_outs, inds

    def forward(self, src_ids, dec_ids, seq_pos_ids, seq_sent_ids, deq_pos_ids, deq_sent_ids):
        """bert.py:92-108 -> (logits [B,L,V], enc_inputs, dec_outputs reversed, ind_outputs)."""
        feats, enc_inputs, dec_outs, inds = self._body(src_ids, dec_ids, seq_pos_ids, seq_sent_ids, deq_pos_ids, deq_sent_ids)
        B, Lq = np.shape(src_ids)[0], np.shape(src_ids)[1]
        H = self.hidden_units
        logits = self.downstream(feats).view(B, Lq, -1)
        return logits, [e.view(B, Lq, H) for e in enc_inputs], [d.view(B, Lq, H) for d in dec_outs], inds

    def fused_loss(self, src_ids, dec_ids, labels, lambda1, lambda2):
        """trainer.py:112-128 with the vocabulary head evaluated only where labels != 0.  Returns the scalar loss
        (autograd-connected); `loss.backward()` then runs the CUDA adjoints."""
        import torch.nn.functional as F
        dev = self.mask_bias.device
        B, Lq = np.shape(src_ids)
        pos_ids = torch.arange(Lq, dtype=torch.int32, device=dev).repeat(B, 1)
        sent = torch.zeros(B, Lq, dtype=torch.int32, device=dev)
        feats, enc_inputs, dec_outs, inds = self._body(src_ids, dec_ids, pos_ids, sent, pos_ids, sent)
        lab = (labels.to(dev) if isinstance(labels, torch.Tensor) else torch.as_tensor(np.asarray(labels)).to(dev)).view(-1).long()
        rows = torch.nonzero(lab != 0, as_tuple=False).flatten()
        if self._fused_head(rows.numel()):
            h = self._head_hidden(feats.index_select(0, rows))
            total = linear_cross_entropy(h, self.item_emb.word_emb.weight, self.mask_bias, lab[rows].int())
        else:
            logits = self.downstream(feats.index_select(0, rows))
            total = MaskedCE.apply(logits, lab[rows].int())
        nh = self.num_heads
        for i in range(self.num_layers):
            if lambda1[i] != 0:
                total = total + lambda1[i] * F.mse_loss(enc_inputs[i], dec_outs[i])
        if nh > 1:
            label = torch.arange(nh, device=dev).repeat(B * Lq, 1)
            for l in range(self.num_layers):
                if lambda2[l] != 0:
                    total = total + lambda2[l] * F.nll_loss(inds[l].reshape(B * Lq, nh, nh), label)
        return total

    def _fused_head(self, R):
        """fused_loss's choice of vocabulary head: the fused tcgen05 head + cross entropy in the bf16 mode on sm_100 from
        FUSED_HEAD_MIN_VOCAB on; the [R, V] logits + MaskedCE otherwise (precision 0 is the parity mode and stays there)."""
        dev = self.mask_bias.device
        return (self.precision == 1 and R > 0 and self.mask_bias.shape[0] >= FUSED_HEAD_MIN_VOCAB
                and torch.cuda.get_device_capability(dev) == (10, 0))

    # ---- full-catalog evaluation -------------------------------------------------------------
    def scoring_catalog(self):
        """what full-catalog ranking scores (adt_b200.evaluate.catalog_of): score[u, i] = <final_feats[u], E_word[i]> + mask_bias[i]
        over the real items i = 1..itemnum only -- the padding row 0 and the extra vocabulary rows (mask token itemnum+1 ...) of the
        tied table are never ranked."""
        from .evaluate import Catalog
        I = self.itemnum
        return Catalog(self.item_emb.word_emb.weight.detach()[1:I + 1], self.mask_bias.detach()[1:I + 1], 1, self.hidden_units)

    @torch.no_grad()
    def final_feats(self, seqs, seq_pos_ids=None, seq_sent_ids=None):
        """[U, H] rows the catalog is scored against: encoder in evaluation mode (no dropout, the ops of `predict`), last position,
        then the head's Linear -> GELU -> LayerNorm (bert.py:81-86).  Position / sentence ids default to 0..L-1 and 0 as in training.
        No host synchronisation, so a CUDA graph can capture it (GraphedScorer)."""
        self._check()
        dev = self.mask_bias.device
        src = _ids(seqs, dev)
        B, Lq = src.shape
        sp = _ids(seq_pos_ids, dev) if seq_pos_ids is not None else torch.arange(Lq, dtype=torch.int32, device=dev).repeat(B, 1)
        ss = _ids(seq_sent_ids, dev) if seq_sent_ids is not None else torch.zeros(B, Lq, dtype=torch.int32, device=dev)
        feats, _, _ = self._encode(src, sp, ss, DropCfg(0.0, 0, 0, False))
        return self._head_hidden(feats.view(B, Lq, -1)[:, -1, :].contiguous())

    @torch.no_grad()
    def full_sort_topk(self, seqs, seen_indptr=None, seen_idx=None, K=40, answers=None, metric_acc=None):
        """full-catalog top-K (the bert.py:80-90 score of every item 1..itemnum) -> (scores [U,K] fp32, ids [U,K] int32), best first,
        ties by ascending id, seen ids (CSR, ascending per user) excluded.  `seqs` is what `predict` takes (history with the mask token
        last).  Same contract as CatalogScorer.topk, including the fused HIT/NDCG/MRR sums into metric_acc."""
        from .evaluate import CatalogScorer
        key = (int(K), self.mask_bias.device)
        if key not in self._scorers:
            self._scorers[key] = CatalogScorer(self, K=K)
        return self._scorers[key].topk(seqs, seen_indptr, seen_idx, answers, metric_acc)

    @torch.no_grad()
    def predict(self, user_ids, seqs, seq_pos_ids, seq_sent_ids, candidates):
        """bert.py:110-116 (the head only on the last position -- the reference runs it on all L and keeps the last)."""
        self._check()
        dev = self.mask_bias.device
        src, sp, ss = _ids(seqs, dev), _ids(seq_pos_ids, dev), _ids(seq_sent_ids, dev)
        B, Lq = src.shape
        feats, _, _ = self._encode(src, sp, ss, DropCfg(0.0, 0, 0, False))
        last = feats.view(B, Lq, -1)[:, -1, :].contiguous()
        logits = self.downstream(last)
        return logits.gather(1, torch.as_tensor(candidates).to(dev).long())


class MaskedCE(torch.autograd.Function):
    """mean cross entropy over the gathered label rows (nn.CrossEntropyLoss(ignore_index=0), trainer.py:45,115)."""

    @staticmethod
    def forward(ctx, logits, labels):
        R, V = logits.shape
        lse = torch.empty(R, dtype=torch.float32, device=logits.device)
        acc = torch.zeros(1, dtype=torch.float64, device=logits.device)
        st = ctypes.c_void_p(torch.cuda.current_stream(logits.device).cuda_stream)
        L.check(L.lib().adt_softmax_ce_fwd(L.ptr(logits), L.ptr(labels), L.ptr(lse), L.ptr(acc), ctypes.c_int32(R), ctypes.c_int32(V), st),
                "adt_softmax_ce_fwd")
        ctx.save_for_backward(logits, labels, lse)
        return (acc / max(R, 1)).float().squeeze(0)

    @staticmethod
    def backward(ctx, g):
        logits, labels, lse = ctx.saved_tensors
        R, V = logits.shape
        d = logits.clone()
        st = ctypes.c_void_p(torch.cuda.current_stream(logits.device).cuda_stream)
        L.check(L.lib().adt_softmax_ce_bwd(L.ptr(d), L.ptr(labels), L.ptr(lse), ctypes.c_float(1.0 / max(R, 1)), ctypes.c_int32(R),
                                           ctypes.c_int32(V), st), "adt_softmax_ce_bwd")
        return d * g, None
