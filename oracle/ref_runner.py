"""TEST / BASELINE INFRASTRUCTURE ONLY -- never imported by the product path (adt_b200/).

Drives the UNMODIFIED reference model staged under oracle/_ref/ (oracle/build_ref.py) the way the reference's own
scripts do, so `bench.py --impl reference`, bench.py's `cpu_baseline` leg and the tests can time / compare against the
reference's real code path with torch's own dropout (no Philox injection, no oracle restatement in the timed region):

  RefTrainer.step()     sasrec/main.py:142-175  (forward -> BCE + lambda1*MSE + lambda2*NLL (stale index, quirk B1)
                                                 + wd*||E|| -> backward -> clip_grad_norm_ -> Adam(b=(.9,.98)))
  RefEvaluator.topk()   sasrec/utils.py:710-731 (predict(full=True) -> negate -> seen -> 1e24 -> argpartition 40 -> argsort)

The ~25 loss/optimiser lines sit inside main() in the reference and cannot be imported; they are restated here with the
same calls in the same order (bool-index gather, BCEWithLogitsLoss, F.mse_loss, F.nll_loss on the [B*L,nh,nh] view,
torch.norm, clip_grad_norm_, torch.optim.Adam).  `device` may be "cpu" (the reported CPU baseline) or "cuda" (PyTorch
eager on the B200: the kernel bar SURVEY 8d / BASELINE.md section 3 name).
"""
import importlib
import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
STAGED = os.path.join(HERE, "_ref", "sasrec")


def ref_dir():
    """sasrec/ of the reference checkout (oracle/build_ref.REF: $ADT_REFERENCE_DIR, by default /root/reference), else the copy
    oracle/build_ref.py staged.  The reference's sources are not part of this repository."""
    from oracle.build_ref import REF
    for d in (os.path.join(REF, "sasrec"), STAGED):
        if os.path.exists(os.path.join(d, "model.py")):
            return d
    raise RuntimeError(f"reference sources not found: no checkout at {REF} (set ADT_REFERENCE_DIR) and nothing staged in oracle/_ref")


def ref_modules():
    d = ref_dir()
    if d not in sys.path:
        sys.path.insert(0, d)
    return importlib.import_module("model")


def make_args(cfg, device):
    return types.SimpleNamespace(device=device, num_heads=cfg["nh"], maxlen=cfg["L"], num_layers=cfg["nl"], hidden_units=cfg["H"],
                                 dropout=cfg["p"])


def build_model(cfg, device="cpu", state_dict=None, seed=23):
    """SASRecADT(usernum, itemnum, args) + the xavier loop of main.py:93-99 (or a given state_dict)."""
    refmodel = ref_modules()
    torch.manual_seed(seed)
    m = refmodel.SASRecADT(1, cfg["items"], make_args(cfg, device)).to(device)
    if state_dict is None:
        for _, prm in m.named_parameters():
            try:
                torch.nn.init.xavier_normal_(prm.data)
            except Exception:   # noqa: BLE001 -- main.py:96-99 ignores the 1-D parameters the same way
                pass
    else:
        m.load_state_dict({k: v.to(device) for k, v in state_dict.items()})
    return m


class RefTrainer:
    def __init__(self, cfg, lambdas1, lambdas2, device="cpu", state_dict=None, lr=1e-3, clip=5.0):
        self.cfg, self.dev = cfg, device
        self.l1, self.l2 = list(lambdas1), list(lambdas2)
        self.model = build_model(cfg, device, state_dict).train()
        self.bce = torch.nn.BCEWithLogitsLoss()
        self.opt = torch.optim.Adam(self.model.parameters(), lr=lr, betas=(0.9, 0.98))     # main.py:122
        self.clip = clip

    def step(self, seq, dec, pos, neg):
        """one iteration of main.py:144-175 on host numpy id arrays [B,L]; returns loss.item()."""
        m, dev, cfg = self.model, self.dev, self.cfg
        nh, L = cfg["nh"], cfg["L"]
        pos_logits, neg_logits, enc_in, dec_out, rec = m(None, seq, dec, pos, neg)
        pos_labels, neg_labels = torch.ones(pos_logits.shape, device=dev), torch.zeros(neg_logits.shape, device=dev)
        self.opt.zero_grad()
        indices = np.where(pos != 0)
        loss = self.bce(pos_logits[indices], pos_labels[indices])
        loss += self.bce(neg_logits[indices], neg_labels[indices])
        i = 0
        if len(enc_in) != 0 and len(enc_in) == len(dec_out):
            for i in range(len(enc_in)):
                loss += self.l1[i] * F.mse_loss(enc_in[i], dec_out[i])
        if nh > 1:
            bs = rec[0].shape[0]
            label = torch.tile(torch.arange(nh), [bs * L, 1]).to(dev)
            for l in range(len(rec)):
                loss += self.l2[i] * F.nll_loss(rec[l].view(bs * L, nh, nh), label)       # stale i: main.py:167-169
        for prm in m.item_emb.parameters():
            loss += cfg["wd"] * torch.norm(prm)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), self.clip)
        self.opt.step()
        return loss.item()


class RefEvaluator:
    def __init__(self, cfg, device="cpu", state_dict=None, model=None):
        self.cfg, self.dev = cfg, device
        self.model = (model if model is not None else build_model(cfg, device, state_dict)).eval()

    @torch.no_grad()
    def topk(self, seq, seen_indptr, seen_idx, k=40):
        """evaluate_loader_full's per-batch lines (utils.py:718-731) with the seen-set given as CSR instead of the scipy
        train_matrix: -> pred_list [U, k] item ids, best first."""
        rank = -self.model.predict(None, seq, None, True)
        rank = rank.cpu().data.numpy().copy()
        U = rank.shape[0]
        rows = np.repeat(np.arange(U), np.diff(seen_indptr))
        rank[rows, seen_idx] = 1e24
        ind = np.argpartition(rank, k)[:, :k]
        arr = rank[np.arange(U)[:, None], ind]
        order = np.argsort(arr)[np.arange(U), ::]
        return ind[np.arange(U)[:, None], order]
