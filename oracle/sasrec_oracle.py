"""TEST INFRASTRUCTURE ONLY (oracle) -- never imported by the product path.

CPU restatement (plain PyTorch, fp32 or fp64) of the reference's SASRec-ADT hot
path.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference leg may import this file.

Pinned against the UNMODIFIED reference (run in the build container by
oracle/make_golden.py, which imports /root/reference/sasrec/model.py) through
the fixtures committed under tests/golden/sasrec_*.npz: see
tests/test_oracle_golden.py.  The reference ships no golden vectors of its own
for this path (SURVEY.md section 4), so that is the only pin there can be.

Reference map (file:line under /root/reference):
  embed()            sasrec/model.py:34-41 (and :53-58 for the decoder input)
  mha()              sasrec/modules.py:270-527 (vendored MHA), :53-64 (sdpa),
                     :122-130 (packed in-projection, q from Q / k,v from x)
  encoder_layer()    sasrec/modules.py:644-655
  decoder_layer()    sasrec/modules.py:666-677
  ffn()              sasrec/modules.py:629-633
  forward()          sasrec/model.py:67-81, :32-50, :52-65
  loss()             sasrec/main.py:147-170
  train_step()       sasrec/main.py:146-173 (clip_grad_norm_ 5.0, Adam b=(.9,.98))
  predict()          sasrec/model.py:83-97
  full_sort_topk()   sasrec/utils.py:718-731
  rank_metrics()     sasrec/utils.py:395-428
  full_sort_metrics  sasrec/utils.py:686-708, :530-569, :629-648
"""
import math
import numpy as np
import torch
import torch.nn.functional as F

from . import philox


class Cfg:
    def __init__(self, item_num, maxlen, hidden, heads, layers, dropout=0.0):
        self.item_num, self.maxlen, self.hidden = item_num, maxlen, hidden
        self.heads, self.layers, self.dropout = heads, layers, dropout


class Drop:
    """Dropout context: p, seed, step, batch offset b0.  site ids follow the
    reference's call order (SURVEY.md A.8)."""

    def __init__(self, p=0.0, seed=0, step=0, b0=0, train=True):
        self.p, self.seed, self.step, self.b0, self.train = p, seed, step, b0, train

    def active(self):
        return self.train and self.p > 0.0

    def mask(self, site, shape, dtype):
        """keep-mask * 1/(1-p) in natural layout `shape` ([B,L,H] row sites or [B,nh,L,L] attention-probability sites)."""
        n = int(np.prod(shape))
        if len(shape) == 4:
            B, nh, Lq, Lk = shape
            keep = philox.keep_mask_attn(B * nh * Lq, Lk, self.p, self.seed, self.step, site, row_offset=self.b0 * nh * Lq)
        else:
            per_b = n // shape[0]
            keep = philox.keep_mask(n, self.p, self.seed, self.step, site, offset=self.b0 * per_b)
        m = torch.from_numpy(keep.reshape(shape)).to(dtype)
        return m * torch.tensor(1.0 / (1.0 - self.p), dtype=torch.float32).to(dtype)

    def apply(self, x, site):
        if not self.active():
            return x
        return x * self.mask(site, tuple(x.shape), x.dtype)


def site_ids(layers):
    """site numbering = order of F.dropout calls in one reference forward."""
    s = {"enc_emb": 0}
    for l in range(layers):
        s[f"enc{l}_attn"], s[f"enc{l}_ffn1"], s[f"enc{l}_ffn2"] = 1 + 3 * l, 2 + 3 * l, 3 + 3 * l
    base = 1 + 3 * layers
    s["dec_emb"] = base
    for l in range(layers):
        b = base + 1 + 4 * l
        s[f"dec{l}_self"], s[f"dec{l}_cross"], s[f"dec{l}_ffn1"], s[f"dec{l}_ffn2"] = b, b + 1, b + 2, b + 3
    return s


def layer_norm(x, w, b, eps=1e-8):
    return F.layer_norm(x, (x.shape[-1],), w, b, eps)


def embed(sd, ids, drop, site):
    """x = dropout(E[ids]*sqrt(H) + P[0..L-1]) * (ids != 0)   -- model.py:34-41"""
    E, P = sd["item_emb.weight"], sd["pos_emb.weight"]
    H = E.shape[1]
    x = E[ids]
    x = x * torch.tensor(H ** 0.5, dtype=torch.float32).to(x.dtype)  # `seqs *= H**0.5` (scalar cast to tensor dtype)
    x = x + P[: ids.shape[1]].unsqueeze(0)
    x = drop.apply(x, site)
    return x * (ids != 0).unsqueeze(-1).to(x.dtype)


class Products:
    """The matrix products of a block: every x W^T + b and the attention core.  The default evaluates them as the reference does;
    a test may pass a subclass that evaluates them differently (for instance on bf16-rounded operands, as the tensor-core kernels
    do) while LayerNorm, biases, residuals, dropout and the independence head stay the oracle's own."""

    def linear(self, x, w, b):
        return F.linear(x, w, b)

    def attention(self, q, k, v, drop, site, causal=True):
        """q (already scaled by 1/sqrt(hd)), k, v: [B, nh, L, hd] -> softmax(q k^T + mask) v, [B, nh, L, hd]"""
        L = q.shape[2]
        s = q @ k.transpose(-1, -2)
        if causal:
            neg = torch.full((L, L), float("-inf"), dtype=s.dtype).triu(1)
            s = s + neg
        p = torch.softmax(s, dim=-1)
        p = drop.apply(p, site)
        return p @ v


PRODUCTS = Products()


def mha(q_in, kv_in, w_in, b_in, w_o, b_o, nh, drop, site, causal=True, prod=PRODUCTS):
    """Batch-first restatement of multi_head_attention_forward (modules.py:270-527).
    q is projected from q_in with rows [0:H) of w_in, k/v from kv_in with rows
    [H:3H).  Returns (out [B,L,H], ctx [B,L,H] head-concatenated)."""
    B, L, H = q_in.shape
    hd = H // nh
    q = prod.linear(q_in, w_in[:H], b_in[:H])
    k = prod.linear(kv_in, w_in[H:2 * H], b_in[H:2 * H])
    v = prod.linear(kv_in, w_in[2 * H:], b_in[2 * H:])
    q = q.view(B, L, nh, hd).transpose(1, 2) / math.sqrt(hd)  # modules.py:54
    k = k.view(B, L, nh, hd).transpose(1, 2)
    v = v.view(B, L, nh, hd).transpose(1, 2)
    ctx = prod.attention(q, k, v, drop, site, causal).transpose(1, 2).reshape(B, L, H)
    return prod.linear(ctx, w_o, b_o), ctx


def ffn(x, w1, b1, w2, b2, drop, site1, site2, prod=PRODUCTS):
    """dropout2(conv2(relu(dropout1(conv1(x))))) + x  -- modules.py:629-633 (Conv1d k=1 == Linear)"""
    h = prod.linear(x, w1.squeeze(-1), b1)
    h = torch.relu(drop.apply(h, site1))
    h = prod.linear(h, w2.squeeze(-1), b2)
    return drop.apply(h, site2) + x


def encoder_layer(sd, pre, x, keep, nh, drop, sites, l, prod=PRODUCTS):
    """modules.py:644-655.  Returns (out, rec_true [B,L,nh,nh], ctx)."""
    Qn = layer_norm(x, sd[pre + "attention_layernorm.weight"], sd[pre + "attention_layernorm.bias"])
    mha_out, ctx = mha(Qn, x, sd[pre + "attention_layer.in_proj_weight"], sd[pre + "attention_layer.in_proj_bias"],
                       sd[pre + "attention_layer.out_proj.weight"], sd[pre + "attention_layer.out_proj.bias"],
                       nh, drop, sites[f"enc{l}_attn"], prod=prod)
    B, L, H = x.shape
    rec_true = F.log_softmax(F.linear(ctx.view(B, L, nh, H // nh), sd[pre + "sparse.weight"], sd[pre + "sparse.bias"]), dim=3)
    y = Qn + mha_out
    z = layer_norm(y, sd[pre + "forward_layernorm.weight"], sd[pre + "forward_layernorm.bias"])
    out = ffn(z, sd[pre + "forward_layer.conv1.weight"], sd[pre + "forward_layer.conv1.bias"],
              sd[pre + "forward_layer.conv2.weight"], sd[pre + "forward_layer.conv2.bias"],
              drop, sites[f"enc{l}_ffn1"], sites[f"enc{l}_ffn2"], prod)
    return out * keep, rec_true, ctx


def misview(rec_true):
    """modules.py:517-518: the [L,B,H] context buffer is .view()ed as [B,L,nh,hd]
    without a transpose, so row r=n*L+l of rec_ind holds true row (l',n')=(r//B, r%B)."""
    B, L = rec_true.shape[:2]
    return rec_true.transpose(0, 1).contiguous().view(B, L, *rec_true.shape[2:])


def decoder_layer(sd, pre, xd, feats, keep_d, nh, drop, sites, l, prod=PRODUCTS):
    """modules.py:666-677 (pos_ffn_layernorm is never applied)."""
    d = layer_norm(xd, sd[pre + "layer_norm.weight"], sd[pre + "layer_norm.bias"])
    a, _ = mha(d, d, sd[pre + "slf_attn.in_proj_weight"], sd[pre + "slf_attn.in_proj_bias"],
               sd[pre + "slf_attn.out_proj.weight"], sd[pre + "slf_attn.out_proj.bias"], nh, drop, sites[f"dec{l}_self"],
               prod=prod)
    c, _ = mha(a, feats, sd[pre + "enc_attn.in_proj_weight"], sd[pre + "enc_attn.in_proj_bias"],
               sd[pre + "enc_attn.out_proj.weight"], sd[pre + "enc_attn.out_proj.bias"], nh, drop, sites[f"dec{l}_cross"],
               prod=prod)
    f = ffn(c, sd[pre + "pos_ffn.conv1.weight"], sd[pre + "pos_ffn.conv1.bias"],
            sd[pre + "pos_ffn.conv2.weight"], sd[pre + "pos_ffn.conv2.bias"], drop, sites[f"dec{l}_ffn1"], sites[f"dec{l}_ffn2"], prod)
    return (d + f) * keep_d


def encode(sd, cfg, seq, drop, last_ln=True):
    """model.py:32-50 -> (feats, enc_inputs, rec_true list, last encoder output)."""
    sites = site_ids(cfg.layers)
    x = embed(sd, seq, drop, sites["enc_emb"])
    keep = (seq != 0).unsqueeze(-1).to(x.dtype)
    enc_inputs, recs = [], []
    for l in range(cfg.layers):
        enc_inputs.append(x)
        x, rec, _ = encoder_layer(sd, f"encoder.encoder_layers.{l}.", x, keep, cfg.heads, drop, sites, l)
        recs.append(rec)
    feats = layer_norm(x, sd["last_layernorm.weight"], sd["last_layernorm.bias"]) if last_ln else x
    return feats, enc_inputs, recs, x


def forward(sd, cfg, seq, dec, pos, neg, drop=None):
    """model.py:67-81.  All ids are int64 tensors [B,L]."""
    drop = drop or Drop()
    sites = site_ids(cfg.layers)
    feats, enc_inputs, recs, _ = encode(sd, cfg, seq, drop)
    xd = embed(sd, dec, drop, sites["dec_emb"])
    keep_d = (dec != 0).unsqueeze(-1).to(xd.dtype)
    dec_outs = []
    for l in range(cfg.layers):
        xd = decoder_layer(sd, f"decoder.decoder_layers.{l}.", xd, feats, keep_d, cfg.heads, drop, sites, l)
        dec_outs.append(xd)
    dec_outs.reverse()  # modules.py:756
    E = sd["item_emb.weight"]
    pos_logits = (feats * E[pos]).sum(-1)
    neg_logits = (feats * E[neg]).sum(-1)
    return {"pos_logits": pos_logits, "neg_logits": neg_logits, "enc_inputs": enc_inputs, "dec_outputs": dec_outs,
            "rec_true": recs, "rec_ind": [misview(r) for r in recs], "feats": feats}


def loss(sd, cfg, out, pos, lambdas1, lambdas2, weight_decay):
    """main.py:147-170, including the stale-index quirk (lambdas2[nl-1] for every layer)."""
    valid = pos != 0
    pl, nl_ = out["pos_logits"][valid], out["neg_logits"][valid]
    total = F.binary_cross_entropy_with_logits(pl, torch.ones_like(pl)) + \
        F.binary_cross_entropy_with_logits(nl_, torch.zeros_like(nl_))
    parts = {"bce": total.detach().clone()}
    for i in range(cfg.layers):
        total = total + lambdas1[i] * F.mse_loss(out["enc_inputs"][i], out["dec_outputs"][i])
    if cfg.heads > 1:
        B, L = pos.shape
        label = torch.arange(cfg.heads).repeat(B * L, 1)
        for l in range(cfg.layers):
            total = total + lambdas2[cfg.layers - 1] * F.nll_loss(out["rec_ind"][l].reshape(B * L, cfg.heads, cfg.heads), label)
    total = total + weight_decay * torch.norm(sd["item_emb.weight"])
    return total, parts


def train_step(sd, cfg, batch, lambdas1, lambdas2, weight_decay, lr=1e-3, clip=5.0, drop=None,
               betas=(0.9, 0.98), adam_state=None):
    """One reference optimisation step (main.py:146-173).  `sd` tensors must be leaf
    tensors with requires_grad; updated in place.  Returns (loss, grads, grad_norm)."""
    seq, dec, pos, neg = batch
    params = [p for p in sd.values()]
    for p in params:
        p.grad = None
    out = forward(sd, cfg, seq, dec, pos, neg, drop)
    total, _ = loss(sd, cfg, out, pos, lambdas1, lambdas2, weight_decay)
    total.backward()
    # unused params (pos_ffn_layernorm.*) keep grad None exactly like the reference
    gnorm = torch.nn.utils.clip_grad_norm_([p for p in params if p.grad is not None], clip)
    grads = {k: (None if p.grad is None else p.grad.detach().clone()) for k, p in sd.items()}
    opt = adam_state if adam_state is not None else torch.optim.Adam(params, lr=lr, betas=betas)
    opt.step()
    return total.detach(), grads, gnorm, opt, out


@torch.no_grad()
def predict(sd, cfg, seq, item_indices=None, full=False):
    """model.py:83-97 (eval mode: no dropout)."""
    feats, _, _, _ = encode(sd, cfg, seq, Drop(train=False))
    final = feats[:, -1, :]
    embs = sd["item_emb.weight"] if full else sd["item_emb.weight"][item_indices]
    return embs.matmul(final.unsqueeze(-1)).squeeze(-1)


def full_sort_topk(scores, seen_rows, k=40):
    """utils.py:718-731 on a [U, I+1] score matrix (higher is better).
    seen_rows: list of 1-D int arrays of already-seen item ids per user.
    Returns int64 [U,k] ids, best first.  (Column 0 -- the padding item -- is
    never masked: quirk B12.)"""
    rank = -np.asarray(scores, dtype=np.float32).copy()
    for u, s in enumerate(seen_rows):
        rank[u, np.asarray(s, dtype=np.int64)] = 1e24
    ind = np.argpartition(rank, k)[:, :k]
    arr = rank[np.arange(len(rank))[:, None], ind]
    order = np.argsort(arr, kind="stable")
    return ind[np.arange(len(rank))[:, None], order]


def rank_metrics(pred, ks=(5, 10)):
    """utils.py:395-428 on pred = -logits [U, C] with the answer in column 0."""
    pred = torch.as_tensor(pred)
    rank = pred.argsort(dim=1).argsort(dim=1)[:, 0]
    U = pred.shape[0]
    HT, NDCG = {}, {}
    for k in ks:
        hit = rank[rank < k]
        HT[k] = hit.shape[0] / U
        NDCG[k] = float((1 / torch.log2(hit + 2.0)).sum()) / U
    r1 = rank.numpy() + 1
    C = 1 + pred.shape[1]  # quirk B7
    return (NDCG, HT), float(np.mean((C - r1) / (C - 1))), rank.numpy()


def full_sort_metrics(answers, pred_list):
    """utils.py:686-708 restated for one answer per user (HIT/NDCG@5,10 + MRR).
    cal_mrr is broken on numpy>=1.24 in the reference (np.float); restated as
    1/(first hit index+1), 0 when absent, mean over all users (utils.py:546-569)."""
    answers = np.asarray(answers).reshape(len(pred_list), -1)
    res = {}
    for k in (5, 10):
        hit = ndcg = 0.0
        for a, p in zip(answers, pred_list):
            aset = set(a.tolist())
            hit += len(aset & set(p[:k].tolist())) / float(len(aset))
            idcg = sum(1.0 / math.log(i + 2, 2) for i in range(min(k, len(a))))
            ndcg += sum(int(p[j] in aset) / math.log(j + 2, 2) for j in range(k)) / idcg
        res[f"HIT@{k}"], res[f"NDCG@{k}"] = hit / len(pred_list), ndcg / len(pred_list)
    mrr = 0.0
    for a, p in zip(answers, pred_list):
        w = np.where(np.isin(p, a))[0]
        if len(w):
            mrr += 1.0 / (w[0] + 1)
    res["MRR"] = mrr / len(pred_list)
    return res


def get_weight(choices, prob):
    """candidates_to_lambdas.py:3-9 / sasrec/evolution.py:124-137."""
    split = 1 / (len(choices) - 1)
    idx = 0
    while prob > split:
        idx += 1
        prob -= split
    rd = prob / split
    return choices[idx] * (1 - rd) + choices[idx + 1] * rd
