"""Full-catalog evaluation on B200: encoder forward -> K7 scoring with fused per-user top-K -> HR/NDCG/MRR.

Replaces evaluate_loader_full / get_full_sort_score (/root/reference/sasrec/utils.py:710-740, :686-708) and the
sampled-candidate ranker evaluate_loader (:395-428).  The score row [U, I+1] is never materialised: the scoring
kernel keeps a sorted top-K list per user on chip (include/adt_b200.h: adt_score_topk).

Item-sharded mode (one 8xB200 box): every rank holds the whole (small) model, scores the contiguous catalog slice
[lo, hi) of its rank, and the per-shard lists are all-gathered ([world, U, K] pairs) and merged on every rank.
"""
import ctypes
import math
from typing import NamedTuple, Optional

import numpy as np
import torch

from . import _lib as L
from .model import _as_ids


class Catalog(NamedTuple):
    """What full-catalog evaluation ranks: score(u, row r) = <feats[u], table[r]> (+ bias[r]), reported as global item id first_id + r."""
    table: torch.Tensor                 # [n_rows, hidden] fp32 rows (a view of the model's item table)
    bias: Optional[torch.Tensor]        # [n_rows] fp32 per-item term added to every score, or None
    first_id: int                       # global item id of table row 0
    hidden: int                         # feature width the encoder produces
    version: object = None              # identity of what a derived table was built from (STOSA rebuilds its rows in place, so the
                                        # table's own `_version` does not move); None for a view of a parameter


def catalog_of(model):
    """The one place that decides which rows of a model are ranked.  Models whose score is not a plain dot product with the whole
    item table (Bert4Rec: tied head rows 1..itemnum + mask_bias; STOSA: centred rows derived from both item tables + a bias, rebuilt
    by this call when stale) define `scoring_catalog()`; every other model ranks all rows of `item_emb.weight` from id 0, without a
    bias."""
    f = getattr(model, "scoring_catalog", None)
    if f is not None:
        return f()
    E = model.item_emb.weight
    return Catalog(E, None, 0, E.shape[1])


def shard_bounds(n_rows, world, rank):
    """contiguous, 4-row aligned slice of `rank` of the catalog rows 0..n_rows-1 (catalog_of(model).table)."""
    per = (n_rows + world - 1) // world
    per = (per + 3) // 4 * 4
    lo = min(n_rows, rank * per)
    return lo, min(n_rows, lo + per)


def merge_topk(scores, ids, K):
    """merge per-shard lists: scores/ids [S, U, K] -> [U, K], order (score desc, id asc); -1 ids are padding.
    Pure torch; runs on CPU (gloo tests) and CUDA alike."""
    S, U, k = scores.shape
    sc = scores.permute(1, 0, 2).reshape(U, S * k)
    idx = ids.permute(1, 0, 2).reshape(U, S * k)
    sc = torch.where(idx < 0, torch.full_like(sc, float("-inf")), sc)
    # lexicographic (score desc, id asc): stable sort by id asc first, then stable by score desc
    o1 = torch.argsort(idx, dim=1, stable=True)
    sc1, id1 = torch.gather(sc, 1, o1), torch.gather(idx, 1, o1)
    o2 = torch.argsort(sc1, dim=1, descending=True, stable=True)
    return torch.gather(sc1, 1, o2)[:, :K], torch.gather(id1, 1, o2)[:, :K]


class CatalogScorer:
    """Full-catalog top-K for a batch of users (replaces predict(full=True) + the host argpartition/sort, utils.py:718-731).

    Multi-GPU (one process per GPU): catalogs of at least `shard_min_items` rows are ITEM-SHARDED -- every rank scores the same
    users against its contiguous catalog slice, the per-shard lists are all-gathered and merged on the device
    (adt_topk_merge).  Smaller catalogs are not worth a collective: every rank scores ITS OWN users against the whole table
    (`sharded` False; the caller hands each rank a different user slice and all-reduces the metric sums at the end)."""

    def __init__(self, model, K=10, n_splits=None, process_group=None, use_tensor_cores=True, tc_min_items=32768,
                 shard_min_items=262144, shard=None):
        self.model, self.K = model, int(K)
        self.use_tc = use_tensor_cores
        self.tc_min_items = tc_min_items   # below this catalog size the exact fp32 kernel is already latency bound and cheaper
        self._tab = None           # (bf16 copy of this rank's catalog shard, max |e|^2 scalar, max |bias| scalar)
        self._tab_key = None       # identity/version of the fp32 table (and bias) the bf16 copy was made from
        self.lib = L.lib()
        self.pg = process_group
        self.world, self.rank = 1, 0
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
            self.rank = torch.distributed.get_rank(process_group)
        n_rows = self.catalog().table.shape[0]
        self.sharded = self.world > 1 and (bool(shard) if shard is not None else n_rows >= shard_min_items)
        self.n_splits = n_splits
        self._buf = {}
        self._fallback = None      # device counter: users re-run on the exact fp32 kernel because the bf16 bound was inconclusive

    # ------------------------------------------------------------------ helpers
    def catalog(self):
        return catalog_of(self.model)

    def bounds(self):
        """this rank's row range of the catalog (rows, not item ids: id = catalog().first_id + row)"""
        n_rows = self.catalog().table.shape[0]
        return shard_bounds(n_rows, self.world, self.rank) if self.sharded else (0, n_rows)

    @property
    def fallback_users(self):
        return 0 if self._fallback is None else int(self._fallback.item())

    def _stream(self, dev):
        return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def _table_key(self):
        c = self.catalog()
        E, b = c.table, c.bias
        return (E.data_ptr(), E._version, tuple(E.shape), getattr(self.model, "_adt_param_version", 0),
                None if b is None else (b.data_ptr(), b._version), c.version)

    def refresh_table(self):
        """(re)build the bf16 copy of the catalog shard and the bound scalars (max |e|^2, max |bias|) from the CURRENT table and bias
        (in place when the shape is unchanged, so a captured graph keeps reading the same buffers)."""
        c = self.catalog()
        E = c.table
        lo, hi = self.bounds()
        shard = E[lo:hi]
        if self._tab is not None and self._tab[0].shape == shard.shape and self._tab[0].device == E.device:
            tab, mx, mxb = self._tab
            mx.zero_()
        else:
            tab = torch.empty(shard.shape, dtype=torch.bfloat16, device=E.device)
            mx = torch.zeros(1, dtype=torch.float32, device=E.device)
            mxb = torch.zeros(1, dtype=torch.float32, device=E.device)
        L.check(self.lib.adt_to_bf16(L.ptr(shard), L.ptr(tab), ctypes.c_int64(shard.shape[0]), ctypes.c_int32(shard.shape[1]), L.ptr(mx),
                                     self._stream(E.device)), "adt_to_bf16")
        if c.bias is not None and hi > lo:
            torch.amax(c.bias[lo:hi].detach().abs(), dim=0, keepdim=True, out=mxb)
        self._tab, self._tab_key = (tab, mx, mxb), self._table_key()

    def ensure_table(self):
        """the bf16 candidates' error bound only holds for the table they were generated from: refresh whenever the fp32 table was
        replaced, modified in place (torch ops bump `_version`) or stepped by this package's optimisers (`_adt_param_version`).
        Not callable during graph capture -- GraphedScorer calls it before every replay."""
        if self._tab is None or self._tab_key != self._table_key():
            self.refresh_table()

    def ensure_current(self):
        """bring everything the kernels read up to date with the model: the catalog itself where the model derives it (catalog_of
        rebuilds STOSA's rows) and, on the tensor-core path, its bf16 copy.  Not callable during graph capture -- GraphedScorer calls
        it before every replay."""
        c = self.catalog()
        if self._uses_tc(c.hidden, *self.bounds()):
            self.ensure_table()

    def _uses_tc(self, H, lo, hi):
        return self.use_tc and H % 64 == 0 and H <= 512 and (hi - lo) >= self.tc_min_items

    # ------------------------------------------------------------------ public
    @torch.no_grad()
    def topk(self, log_seqs, seen_indptr=None, seen_idx=None, answers=None, metric_acc=None):
        """-> (scores [U,K] fp32, ids [U,K] int32), best first, seen items excluded (utils.py:725).
        answers [U] + metric_acc (float64 device tensor [6]): fused HIT/NDCG@5,10 + MRR sums (get_full_sort_score)."""
        m = self.model
        dev = self.catalog().table.device
        seq = _as_ids(log_seqs, dev)
        feats = m.final_feats(seq)
        return self.topk_from_feats(feats, seen_indptr, seen_idx, answers, metric_acc)

    @torch.no_grad()
    def topk_from_feats(self, feats, seen_indptr=None, seen_idx=None, answers=None, metric_acc=None):
        dev = feats.device
        ip = _as_ids(seen_indptr, dev) if seen_indptr is not None else None
        ix = _as_ids(seen_idx, dev) if seen_idx is not None else None
        ans = _as_ids(answers, dev) if answers is not None else None
        if self._uses_tc(feats.shape[1], *self.bounds()) and not torch.cuda.is_current_stream_capturing():
            self.ensure_table()
        return self._device_topk(feats, ip, ix, ans, metric_acc)

    @torch.no_grad()
    def _device_topk(self, feats, ip, ix, ans, metric_acc):
        """everything after the encoder, device side only (no host synchronisation: capturable)."""
        lo, hi = self.bounds()
        local_metrics = not self.sharded
        if self._uses_tc(feats.shape[1], lo, hi):
            os_, oi = self._topk_tc(feats, ip, ix, lo, hi, ans if local_metrics else None, metric_acc if local_metrics else None)
        else:
            os_, oi = self._topk_exact(feats, ip, ix, lo, hi, ans if local_metrics else None, metric_acc if local_metrics else None)
        if not self.sharded:
            return os_, oi
        return self._merge(os_, oi, ans, metric_acc)

    # ------------------------------------------------------------------ kernels
    @torch.no_grad()
    def _topk_tc(self, feats, ip, ix, lo, hi, ans, metric_acc):
        """tensor-core path: tcgen05 candidate generation + exact fp32 re-score; users whose bf16 bound was inconclusive are
        flagged on the device and re-run by the exact kernel in the same stream (masked launch: unflagged tiles exit at once)."""
        dev = feats.device
        U, H = feats.shape
        c = self.catalog()
        if self._tab is None:
            self.refresh_table()
        tab, mx, mxb = self._tab
        n_items = hi - lo
        K = self.K
        kc, ns = ctypes.c_int32(0), ctypes.c_int32(0)
        self.lib.adt_score_tc_plan(ctypes.c_int32(U), ctypes.c_int32(H), ctypes.c_int32(n_items), ctypes.c_int32(K), ctypes.byref(kc), ctypes.byref(ns))
        KC, S = kc.value, ns.value
        key = ("tc", U, S, KC)
        if key not in self._buf:
            pk = torch.empty(2, U, K, dtype=torch.int32, device=dev)        # [0] scores (float bits), [1] ids: one all-gather payload
            self._buf[key] = (torch.empty(S, U, KC, device=dev), torch.empty(S, U, KC, dtype=torch.int32, device=dev),
                              torch.empty(2 * S, U, device=dev), pk, torch.empty(U, dtype=torch.int32, device=dev),
                              torch.empty(U, H, dtype=torch.bfloat16, device=dev))
        ps, pi, pt, pk, flags, fb = self._buf[key]
        os_, oi = pk[0].view(torch.float32), pk[1]
        self._last_pk = pk
        if self._fallback is None:
            self._fallback = torch.zeros(1, dtype=torch.int64, device=dev)
        st = self._stream(dev)
        L.check(self.lib.adt_to_bf16(L.ptr(feats), L.ptr(fb), ctypes.c_int64(U), ctypes.c_int32(H), None, st), "adt_to_bf16")
        bias = c.bias[lo:hi] if c.bias is not None else None
        a = L.fill(L.adt_score_topk_tc_args(), feats=feats, feats_bf16=fb, U=U, H=H, item_emb=c.table[lo:hi], item_emb_bf16=tab, n_items=n_items,
                   item_offset=c.first_id + lo, max_normsq=mx, seen_indptr=ip, seen_idx=ix, K=K, KC=KC, n_splits=S, part_scores=ps, part_ids=pi,
                   part_thr=pt, out_scores=os_, out_ids=oi, flags=flags, answers=ans, metric_acc=metric_acc,
                   item_bias=bias, max_abs_bias=mxb if bias is not None else None)
        L.check(self.lib.adt_score_topk_tc(ctypes.byref(a), st), "adt_score_topk_tc")
        self._fallback += flags.sum()
        self._topk_exact(feats, ip, ix, lo, hi, ans, metric_acc, out=(os_, oi), user_mask=flags)
        return os_, oi

    @torch.no_grad()
    def _topk_exact(self, feats, ip, ix, lo, hi, ans=None, metric_acc=None, out=None, user_mask=None):
        c = self.catalog()
        dev = feats.device
        U, H = feats.shape
        n_items = hi - lo
        tiles = (U + 63) // 64
        S = self.n_splits or max(1, min(256, (2 * 148 + tiles - 1) // tiles, (n_items + 255) // 256))
        key = ("ex", U, S)
        if key not in self._buf:
            pk = torch.empty(2, U, self.K, dtype=torch.int32, device=dev)
            self._buf[key] = (torch.empty(S, U, self.K, device=dev), torch.empty(S, U, self.K, dtype=torch.int32, device=dev), pk)
        ps, pi, pk = self._buf[key]
        os_, oi = out if out is not None else (pk[0].view(torch.float32), pk[1])
        if out is None:
            self._last_pk = pk
        a = L.fill(L.adt_score_topk_args(), feats=feats, U=U, H=H, item_emb=c.table[lo:hi], n_items=n_items, item_offset=c.first_id + lo,
                   seen_indptr=ip, seen_idx=ix, K=self.K, n_splits=S, part_scores=ps, part_ids=pi, out_scores=os_, out_ids=oi,
                   answers=ans, metric_acc=metric_acc, user_mask=user_mask,
                   item_bias=c.bias[lo:hi] if c.bias is not None else None)
        L.check(self.lib.adt_score_topk(ctypes.byref(a), self._stream(dev)), "adt_score_topk")
        return os_, oi

    @torch.no_grad()
    def _merge(self, os_, oi, ans=None, metric_acc=None):
        """item-sharded mode: ONE all-gather of the packed (score bits, id) lists, merged on the device by adt_topk_merge."""
        U, K, dev = os_.shape[0], self.K, os_.device
        key = ("mg", U)
        if key not in self._buf:
            self._buf[key] = (torch.empty(self.world, 2, U, K, dtype=torch.int32, device=dev), torch.empty(2, U, K, dtype=torch.int32, device=dev),
                              torch.empty(2, U, K, dtype=torch.int32, device=dev))
        g, mine, res = self._buf[key]
        pk = getattr(self, "_last_pk", None)
        if pk is not None and pk.data_ptr() == os_.data_ptr() and pk[1].data_ptr() == oi.data_ptr():
            src = pk                                         # already packed (our own output buffers)
        else:
            mine[0].view(torch.float32).copy_(os_)
            mine[1].copy_(oi)
            src = mine
        torch.distributed.all_gather_into_tensor(g, src, group=self.pg)
        L.check(self.lib.adt_topk_merge(ctypes.c_void_p(g.data_ptr()), ctypes.c_void_p(g.data_ptr() + 4 * U * K), ctypes.c_int32(self.world),
                                        ctypes.c_int64(2 * U * K), ctypes.c_int32(U), ctypes.c_int32(K), L.ptr(res[0]), L.ptr(res[1]),
                                        L.ptr(ans), L.ptr(metric_acc), self._stream(dev)), "adt_topk_merge")
        return res[0].view(torch.float32), res[1]


class GraphedScorer:
    """Fixed-shape evaluation batch (U users x L positions, seen-set CSR of at most `max_seen` ids, one held-out answer per user)
    replayed as ONE CUDA graph: encoder forward + catalog scoring + fused top-K + the exact re-run of flagged users + (item-sharded)
    the all-gather and device-side merge + the HIT/NDCG/MRR sums.  Per batch the host copies the ids into the static buffers and
    replays; nothing is read back until the caller asks for the metrics."""

    def __init__(self, scorer, U, L_, max_seen, capture_collective=True):
        self.sc = scorer
        cat = scorer.catalog()
        dev = cat.table.device
        self.U, self.L = int(U), int(L_)
        self.seq = torch.zeros(U, L_, dtype=torch.int32, device=dev)
        self.ip = torch.zeros(U + 1, dtype=torch.int32, device=dev)
        self.ix = torch.zeros(max(1, int(max_seen)), dtype=torch.int32, device=dev)
        self.ans = torch.zeros(U, dtype=torch.int32, device=dev)
        self.metric_acc = torch.zeros(6, dtype=torch.float64, device=dev)
        self.tc = scorer._uses_tc(cat.hidden, *scorer.bounds())
        if self.tc:
            scorer.refresh_table()
        # the collective of the item-sharded path is captured with the rest when NCCL allows it, else issued between two graphs
        self.split = scorer.sharded and not capture_collective
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):          # warm-up outside capture (lazy allocations, cudaFuncSetAttribute, NCCL channels)
            for _ in range(2):
                self._device_part()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.metric_acc.zero_()
        if scorer._fallback is not None:
            scorer._fallback.zero_()
        self.graph = torch.cuda.CUDAGraph()
        if self.split:
            with torch.cuda.graph(self.graph):
                self.local = self._local_part()
            self.out = None
        else:
            with torch.cuda.graph(self.graph):
                self.out = self._device_part()

    @torch.no_grad()
    def _local_part(self):
        sc = self.sc
        self.feats = sc.model.final_feats(self.seq)
        lo, hi = sc.bounds()
        if self.tc:
            return sc._topk_tc(self.feats, self.ip, self.ix, lo, hi, None, None)
        return sc._topk_exact(self.feats, self.ip, self.ix, lo, hi, None, None)

    @torch.no_grad()
    def _device_part(self):
        self.feats = self.sc.model.final_feats(self.seq)
        return self.sc._device_topk(self.feats, self.ip, self.ix, self.ans, self.metric_acc)

    @torch.no_grad()
    def topk(self, log_seqs, seen_indptr, seen_idx, answers=None):
        """same contract as CatalogScorer.topk for a [U, L] batch; the returned tensors are overwritten by the next call.
        With `answers`, the metric sums accumulate in self.metric_acc (read them with metrics())."""
        def src(a):   # host numpy or torch tensor (any device) -> int32 tensor that copy_ can read
            return a.to(torch.int32) if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32))
        seq, ip, ix = src(log_seqs), src(seen_indptr), src(seen_idx)
        if tuple(seq.shape) != (self.U, self.L) or ip.numel() != self.U + 1 or ix.numel() > self.ix.numel():
            raise ValueError(f"GraphedScorer was built for [{self.U},{self.L}] batches with at most {self.ix.numel()} seen ids")
        self.sc.ensure_current()
        self.seq.copy_(seq, non_blocking=True)
        self.ip.copy_(ip, non_blocking=True)
        self.ix[:ix.numel()].copy_(ix, non_blocking=True)
        if answers is not None:
            self.ans.copy_(src(answers), non_blocking=True)
        else:
            self.ans.fill_(-1)
        self.graph.replay()
        if self.split:
            return self.sc._merge(*self.local, self.ans, self.metric_acc)
        return self.out

    def metrics(self, reset=True):
        """HIT@5/10, NDCG@5/10, MRR accumulated since the last reset (one device -> host read)."""
        res = metrics_from_acc(self.metric_acc)
        if reset:
            self.metric_acc.zero_()
        return res


def metrics_from_acc(acc):
    """accumulator of the fused metric epilogue -> the dict get_full_sort_score (utils.py:686-708) reports."""
    a = acc.tolist() if isinstance(acc, torch.Tensor) else list(acc)
    U = max(a[5], 1.0)
    return {"HIT@5": a[0] / U, "NDCG@5": a[1] / U, "HIT@10": a[2] / U, "NDCG@10": a[3] / U, "MRR": a[4] / U, "users": int(a[5])}


def hit_ndcg_mrr(answers, topk_ids, ks=(5, 10)):
    """get_full_sort_score (utils.py:686-708) for one held-out answer per user.  Host side, exact integers.
    returns dict HIT@k, NDCG@k, MRR (MRR over the returned list, 0 when absent: utils.py:546-569)."""
    ids = np.asarray(topk_ids.cpu() if isinstance(topk_ids, torch.Tensor) else topk_ids)
    ans = np.asarray(answers).reshape(-1, 1)
    hit = ids == ans
    U = ids.shape[0]
    has = hit.any(axis=1)
    first = np.where(has, hit.argmax(axis=1), ids.shape[1])
    res = {}
    for k in ks:
        inside = first < k
        res[f"HIT@{k}"] = float(inside.sum()) / U
        res[f"NDCG@{k}"] = float((1.0 / np.log2(first[inside] + 2.0)).sum()) / U
    res["MRR"] = float((1.0 / (first[has] + 1.0)).sum()) / U
    return res


@torch.no_grad()
def rank_of_first_candidate(model, user_ids, log_seqs, item_idx):
    """evaluate_loader's `(-predict).argsort().argsort()[:, 0]` (utils.py:407-410) without the two sorts:
    rank = #{j : s_j > s_0} (ties broken like a stable argsort: earlier columns first)."""
    return sampled_rank(model, log_seqs, item_idx)[0]


@torch.no_grad()
def sampled_rank(model, log_seqs, item_idx, metric_acc=None):
    """-> (rank [U] int32, scores [U,C]).  Encoder on the CUDA path, candidate gather-dot + rank count (+ optionally the
    HR/NDCG/AUC sums of utils.py:411-427 into metric_acc[7], float64 device tensor) in ONE library launch -- no [U,C,H]
    gather, no bmm, no sort."""
    from .model import score_candidates
    dev = model.item_emb.weight.device
    seq = _as_ids(log_seqs, dev)
    if hasattr(model, "final_feats"):
        final = model.final_feats(seq)
    else:        # supernet: no last LayerNorm, candidate blocks blended on the host side
        B, Lq = seq.shape
        from .blocks import DropCfg
        x, _, _ = model.log2feats(seq, DropCfg(0.0, 0, 0, False))
        final = x.view(B, Lq, model.hidden)[:, -1, :].contiguous()
    scores, rank = score_candidates(model.item_emb.weight, final, item_idx, False, want_rank=True, metric_acc=metric_acc)
    return rank, scores


def sampled_metrics_from_acc(acc):
    """device accumulator of adt_candidate_scores -> ((NDCG, HR) dicts for k = 5, 10), AUC, MRR) as evaluate_loader returns them."""
    a = acc.tolist() if isinstance(acc, torch.Tensor) else list(acc)
    U = max(a[5], 1.0)
    return ({5: a[1] / U, 10: a[3] / U}, {5: a[0] / U, 10: a[2] / U}), a[6] / U, a[4] / U


def sampled_metrics(rank, n_candidates, ks=(5, 10)):
    """HR/NDCG@k and the reference's AUC (with its C = 1 + n_candidates quirk, utils.py:424-427)."""
    rank = np.asarray(rank.cpu() if isinstance(rank, torch.Tensor) else rank).astype(np.int64)
    U = len(rank)
    ndcg = {k: float((1.0 / np.log2(rank[rank < k] + 2.0)).sum()) / U for k in ks}
    hr = {k: float((rank < k).sum()) / U for k in ks}
    C = 1 + n_candidates
    auc = float(np.mean((C - (rank + 1)) / (C - 1)))
    return (ndcg, hr), auc
