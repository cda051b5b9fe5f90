"""TEST INFRASTRUCTURE ONLY (oracle) -- never imported by the product path.

CPU restatement (plain PyTorch) of the reference's STOSA-ADT hot path (SURVEY 8a row a20).  Pinned against the UNMODIFIED
reference (/root/reference/stosa/models.py `DisenDistSAModel` + the loss lines of stosa/trainer.py, run by
oracle/make_golden_stosa.py) through tests/golden/stosa_*.npz.

Reference map (file:line under /root/reference/stosa):
  wdist() / wdist_matmul()  modules.py:22-28 / 30-43
  embed_mean()/embed_cov()  models.py:183-210      (LN(eps=1e-12) -> dropout -> ELU ; cov: ELU(dropout(LN)) + 1)
  attention()               modules.py:222-275 (self) and :312-361 (encoder-decoder); its core (scores .. P^2 cv) is attention_core()
  init_state()              models.py:262-270 (a fresh state dict at any shape)
  intermediate()            modules.py:474-494     (dense 4H, ELU, dense, dropout, LN(+input))
  enc_layer()/dec_layer()   modules.py:509-525 / 527-541 (the decoder's self attention output is DISCARDED, :537-538)
  finetune()                models.py:212-260
  loss()                    trainer.py:358-378 (bpr_optimization) + :517-533 (reconstruction / independence / pvn terms)
  predict_full()            trainer.py:464-479 ; full_sort_topk() :604-614
Dropout sites follow the reference's call order: enc mean emb, enc cov emb, dec mean emb, dec cov emb ; per encoder layer
(attention probs, mean out, cov out, mean FFN, cov FFN) ; per decoder layer (3 sites of the discarded self attention,
attention probs, mean out, cov out, mean FFN, cov FFN).  A site number is only consumed when its probability is > 0.
"""
import math
import numpy as np
import torch
import torch.nn.functional as F

from .sasrec_oracle import Drop
from .bert_oracle import _Sites, _drop

MASK = float(-2 ** 32 + 1)


class SCfg:
    def __init__(self, item_size, num_users, maxlen, hidden, heads, layers, dropout=0.0, attention_dropout=0.0, pvn_weight=0.005):
        self.item_size, self.num_users, self.maxlen, self.hidden, self.heads, self.layers = item_size, num_users, maxlen, hidden, heads, layers
        self.dropout, self.attention_dropout, self.pvn_weight = dropout, attention_dropout, pvn_weight


def init_state(cfg, seed, std=0.02, dtype=torch.float32):
    """a freshly initialised DisenDistSAModel state dict (names, order and shapes of the reference's state_dict; models.py:262-270:
    Linear and Embedding weights ~ N(0.01, std) including the padding row, Linear biases 0, LayerNorm 1 / 0), drawn from `seed`."""
    H, nh = cfg.hidden, cfg.heads
    g = torch.Generator().manual_seed(int(seed))
    sd = {}

    def normal(name, *shape):
        sd[name] = torch.empty(*shape, dtype=torch.float32).normal_(mean=0.01, std=std, generator=g).to(dtype)

    def linear(pre, n_out, n_in):
        normal(pre + ".weight", n_out, n_in)
        sd[pre + ".bias"] = torch.zeros(n_out, dtype=dtype)

    def layer_norm(pre):
        sd[pre + ".weight"], sd[pre + ".bias"] = torch.ones(H, dtype=dtype), torch.zeros(H, dtype=dtype)

    def dist_attention(pre):
        for n in ("mean_query", "cov_query", "mean_key", "cov_key", "mean_value", "cov_value", "mean_dense", "cov_dense"):
            linear(f"{pre}.{n}", H, H)
        layer_norm(pre + ".LayerNorm")

    def intermediate(pre):
        linear(pre + ".dense_1", 4 * H, H)
        linear(pre + ".dense_2", H, 4 * H)
        layer_norm(pre + ".LayerNorm")

    for which in ("mean", "cov"):
        normal(f"item_{which}_embeddings.weight", cfg.item_size, H)
    for which in ("mean", "cov"):
        normal(f"position_{which}_embeddings.weight", cfg.maxlen, H)
    normal("user_margins.weight", cfg.num_users, 1)
    for l in range(cfg.layers):
        pre = f"item_encoder.layer.{l}"
        dist_attention(pre + ".attention")
        intermediate(pre + ".mean_intermediate")
        intermediate(pre + ".cov_intermediate")
        linear(pre + ".mean_independence_layer", nh, H // nh)
        linear(pre + ".cov_independence_layer", nh, H // nh)
    for l in range(cfg.layers):
        pre = f"item_decoder.layer.{l}"
        dist_attention(pre + ".dec_attention")
        dist_attention(pre + ".enc_attention")
        intermediate(pre + ".mean_intermediate")
        intermediate(pre + ".cov_intermediate")
    layer_norm("LayerNorm")
    layer_norm("decLayerNorm")
    return sd


def wdist(m1, c1, m2, c2):
    s1, s2 = torch.sqrt(torch.clamp(c1, min=1e-24)), torch.sqrt(torch.clamp(c2, min=1e-24))
    return ((m1 - m2) ** 2).sum(-1) + ((s1 - s2) ** 2).sum(-1)


def wdist_matmul(m1, c1, m2, c2):
    ret = -2 * m1 @ m2.transpose(-1, -2) + (m1 ** 2).sum(-1, keepdim=True) + (m2 ** 2).sum(-1, keepdim=True).transpose(-1, -2)
    s1, s2 = torch.sqrt(torch.clamp(c1, min=1e-24)), torch.sqrt(torch.clamp(c2, min=1e-24))
    return ret + (-2 * s1 @ s2.transpose(-1, -2) + c1.sum(-1, keepdim=True) + c2.sum(-1, keepdim=True).transpose(-1, -2))


def ln(sd, pre, x):
    return F.layer_norm(x, (x.shape[-1],), sd[pre + "weight"], sd[pre + "bias"], 1e-12)


def embed(sd, which, ids, cfg, drop, sites):
    L = ids.shape[1]
    e = F.embedding(ids, sd[f"item_{which}_embeddings.weight"], padding_idx=0) + sd[f"position_{which}_embeddings.weight"][:L][None]
    e = _drop(ln(sd, "LayerNorm.", e), drop, cfg.dropout, sites)
    return F.elu(e) if which == "mean" else F.elu(e) + 1


def attention_scores(mq, cq, mk, ck, mask):
    """modules.py:240-249: masked, scaled scores [B,nh,L,L] of the head-split streams [B,nh,L,hd].

    The additive mask is applied with the reference's fp32 semantics in any working dtype: a masked entry becomes
    float32(score) + float32(MASK).  In fp32 every |score| < 256 is absorbed into MASK (ulp 512), so a query row whose keys are all
    masked (left padding) is uniform over its L keys; in plain fp64 the scores would survive and that row would not be uniform.
    For fp32 inputs this is bit-identical to `score + mask`."""
    s = -wdist_matmul(mq, cq, mk, ck) / math.sqrt(mq.shape[-1])
    return torch.where(mask != 0, (s.float() + mask.float()).to(s.dtype), s)


def attention_core(mq, cq, mk, ck, mv, cv, mask, drop_p, drop, sites):
    """modules.py:240-254 on the projected head-split streams [B,nh,L,hd] (cov streams already ELU+1) -> (mean context, cov context),
    each [B,L,nh,hd]: scores, mask, softmax, dropout, P mv, P^2 cv."""
    p = _drop(torch.softmax(attention_scores(mq, cq, mk, ck, mask), dim=-1), drop, drop_p, sites)
    mctx = (p @ mv).permute(0, 2, 1, 3).contiguous()
    cctx = ((p ** 2) @ cv).permute(0, 2, 1, 3).contiguous()
    return mctx, cctx


def attention(sd, pre, qm, qc, km, kc, mask, cfg, drop, sites):
    """-> (mean', cov', mean context [B,L,nh,hd], cov context)."""
    B, L, H = qm.shape
    nh, hd = cfg.heads, H // cfg.heads
    lin = lambda n, x: F.linear(x, sd[pre + n + ".weight"], sd[pre + n + ".bias"])
    sp = lambda x: x.view(B, L, nh, hd).permute(0, 2, 1, 3)
    mq, mk, mv = sp(lin("mean_query", qm)), sp(lin("mean_key", km)), sp(lin("mean_value", km))
    cq, ck, cv = sp(F.elu(lin("cov_query", qc)) + 1), sp(F.elu(lin("cov_key", kc)) + 1), sp(F.elu(lin("cov_value", kc)) + 1)
    mctx, cctx = attention_core(mq, cq, mk, ck, mv, cv, mask, cfg.attention_dropout, drop, sites)
    mh = ln(sd, pre + "LayerNorm.", _drop(lin("mean_dense", mctx.view(B, L, H)), drop, cfg.dropout, sites) + qm)
    ch = ln(sd, pre + "LayerNorm.", _drop(lin("cov_dense", cctx.view(B, L, H)), drop, cfg.dropout, sites) + qc)
    return mh, ch, mctx, cctx


def intermediate(sd, pre, x, cfg, drop, sites):
    h = F.linear(F.elu(F.linear(x, sd[pre + "dense_1.weight"], sd[pre + "dense_1.bias"])), sd[pre + "dense_2.weight"], sd[pre + "dense_2.bias"])
    return ln(sd, pre + "LayerNorm.", _drop(h, drop, cfg.dropout, sites) + x)


def masks(ids):
    """models.py:214-233: additive (1 - nonpad_key * causal) * (-2^32+1), [B,1,L,L]."""
    L = ids.shape[1]
    causal = torch.tril(torch.ones(L, L, dtype=torch.long))[None, None]
    m = (ids > 0).long()[:, None, None, :] * causal
    return (1.0 - m.float()) * MASK


def forward(sd, cfg, ids, dec_ids, drop=None):
    drop = drop or Drop(train=False)
    sites = _Sites()
    emask, dmask = masks(ids), masks(dec_ids)
    m, c = embed(sd, "mean", ids, cfg, drop, sites), embed(sd, "cov", ids, cfg, drop, sites)
    dm, dc = embed(sd, "mean", dec_ids, cfg, drop, sites), embed(sd, "cov", dec_ids, cfg, drop, sites)
    enc_inputs, recs = [], []
    for l in range(cfg.layers):
        pre = f"item_encoder.layer.{l}."
        enc_inputs.append((m, c))
        am, ac, rm, rc = attention(sd, pre + "attention.", m, c, m, c, emask, cfg, drop, sites)
        m = intermediate(sd, pre + "mean_intermediate.", am, cfg, drop, sites)
        c = F.elu(intermediate(sd, pre + "cov_intermediate.", ac, cfg, drop, sites)) + 1
        rm = F.linear(rm, sd[pre + "mean_independence_layer.weight"], sd[pre + "mean_independence_layer.bias"])
        rc = F.linear(rc, sd[pre + "cov_independence_layer.weight"], sd[pre + "cov_independence_layer.bias"])
        recs.append((F.log_softmax(rm, dim=3), F.log_softmax(rc, dim=3)))
    dec_outs = []
    for l in range(cfg.layers):
        pre = f"item_decoder.layer.{l}."
        # the decoder's self attention is evaluated and thrown away (modules.py:537-538): it only consumes dropout sites
        for p in (cfg.attention_dropout, cfg.dropout, cfg.dropout):
            sites.next(drop.train and p > 0.0)
        am, ac, _, _ = attention(sd, pre + "enc_attention.", dm, dc, m, c, emask, cfg, drop, sites)
        dm = intermediate(sd, pre + "mean_intermediate.", am, cfg, drop, sites)
        dc = F.elu(intermediate(sd, pre + "cov_intermediate.", ac, cfg, drop, sites)) + 1
        dec_outs.append((dm, dc))
    return {"mean": m, "cov": c, "enc_inputs": enc_inputs, "recs": recs, "dec_outputs": dec_outs}


def loss(sd, cfg, out, pos, neg, lambda1, lambda2):
    """trainer.py:358-378 + 517-533 -> (total, bpr, pvn, auc)."""
    H = cfg.hidden
    Em, Ec = sd["item_mean_embeddings.weight"], sd["item_cov_embeddings.weight"]
    pm, pc = F.embedding(pos, Em, padding_idx=0).view(-1, H), (F.elu(F.embedding(pos, Ec, padding_idx=0)) + 1).view(-1, H)
    nm, nc = F.embedding(neg, Em, padding_idx=0).view(-1, H), (F.elu(F.embedding(neg, Ec, padding_idx=0)) + 1).view(-1, H)
    sm, sc = out["mean"].reshape(-1, H), out["cov"].reshape(-1, H)
    dp, dn, dpn = wdist(sm, sc, pm, pc), wdist(sm, sc, nm, nc), wdist(pm, pc, nm, nc)
    t = (pos > 0).view(-1).float()
    bpr = torch.sum(F.softplus(-(dn - dp + 1e-24)) * t) / t.sum()      # == -log(sigmoid(.)) where that is finite
    pvn = cfg.pvn_weight * torch.sum(torch.clamp(dp - dpn, 0) * t) / t.sum()
    auc = torch.sum(((torch.sign(dn - dp) + 1) / 2) * t) / t.sum()
    total = bpr
    dec = list(reversed(out["dec_outputs"]))
    for l in range(cfg.layers):
        total = total + lambda1[l] * F.mse_loss(out["enc_inputs"][l][0], dec[l][0]) + lambda1[l] * F.mse_loss(out["enc_inputs"][l][1], dec[l][1])
    B, L = pos.shape
    nh = cfg.heads
    label = torch.arange(nh).repeat(B * L, 1)
    for l in range(cfg.layers):
        total = total + lambda2[l] * F.nll_loss(out["recs"][l][0].reshape(B * L, nh, nh), label) \
            + lambda2[l] * F.nll_loss(out["recs"][l][1].reshape(B * L, nh, nh), label)
    return total + pvn, bpr, pvn, auc


@torch.no_grad()
def predict_full(sd, cfg, ids):
    """trainer.py:464-479 on the last position: distance matrix [U, item_size] (smaller is better)."""
    out = forward(sd, cfg, ids, ids, Drop(train=False))
    um, uc = out["mean"][:, -1, :], out["cov"][:, -1, :]
    return wdist_matmul(um, uc, sd["item_mean_embeddings.weight"], F.elu(sd["item_cov_embeddings.weight"]) + 1)


def full_sort_topk(dist, seen, K=40):
    """trainer.py:604-614: seen -> 1e24, K smallest in ascending order (ties by id)."""
    d = np.array(dist, dtype=np.float32, copy=True)
    for u, s in enumerate(seen):
        d[u, list(s)] = 1e24
    order = np.lexsort((np.broadcast_to(np.arange(d.shape[1]), d.shape), d), axis=1)
    return order[:, :K]
