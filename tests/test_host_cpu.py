"""CPU tests: C-ABI library loads and exports every declared symbol, the host-side mirror of the reference interface
(parameter names/shapes, error behaviour), metric/merge host logic, and the N>1 paths on gloo (world_size 2)."""
import os
import types
import numpy as np
import pytest
import torch

from helpers import golden_names, load_golden, sd_from, GOLDEN


def test_header_parses_and_library_exports_every_symbol():
    import __graft_entry__ as g
    from adt_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        g.build()
    lib = _lib.lib()
    assert len(_lib.FUNCTIONS) >= 18
    for f in _lib.FUNCTIONS:
        assert hasattr(lib, f), f
    assert lib.adt_version() >= 100
    # struct layouts come from the header: spot-check one
    d = _lib.adt_dropout()
    assert [n for n, _ in d._fields_] == ["enabled", "p", "seed", "step", "site", "base", "step_dev"]


def test_ctypes_mirrors_match_the_c_struct_layouts(tmp_path):
    """the Python side generates its ctypes.Structure classes from include/adt_b200.h; compile the same header with gcc
    and compare sizeof / offsetof of EVERY field, so that a header edit can never silently shift the boundary."""
    import ctypes
    import subprocess
    from adt_b200 import _lib
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{_lib.HEADER}"', 'int main(void) {']
    for name, cls in _lib.STRUCTS.items():
        lines.append(f'  printf("{name} . %zu\\n", sizeof({name}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{name} {fname} %zu\\n", offsetof({name}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    seen = 0
    for ln in filter(None, out):
        name, fname, val = ln.split()
        cls = _lib.STRUCTS[name]
        mine = ctypes.sizeof(cls) if fname == "." else getattr(cls, fname).offset
        assert mine == int(val), (name, fname, mine, int(val))
        seen += 1
    assert seen == sum(len(c._fields_) + 1 for c in _lib.STRUCTS.values()) and seen > 300


@pytest.mark.parametrize("name", golden_names())
def test_state_dict_matches_reference_names_and_shapes(name):
    """drop-in contract: reference checkpoints load into our module and vice versa (SURVEY 8b)."""
    from adt_b200 import SASRecADT
    g = load_golden(name)
    d = g["dims"]
    args = types.SimpleNamespace(device="cpu", num_heads=d["nh"], maxlen=d["L"], num_layers=d["nl"], hidden_units=d["H"], dropout=0.5)
    m = SASRecADT(100, d["I"], args)
    ref = sd_from(g)
    ours = m.state_dict()
    assert list(ours.keys()) == list(ref.keys())
    for k in ref:
        assert tuple(ours[k].shape) == tuple(ref[k].shape), k
    m.load_state_dict(ref)  # strict
    assert [n for n, _ in m.named_parameters()] == [k for k in ref.keys()]


def test_no_cpu_fallback():
    from adt_b200 import SASRecADT
    from adt_b200._lib import AdtError
    args = types.SimpleNamespace(device="cpu", num_heads=2, maxlen=8, num_layers=1, hidden_units=16, dropout=0.0)
    m = SASRecADT(10, 20, args)
    ids = np.ones((2, 8), np.int64)
    with pytest.raises(AdtError):
        m(None, ids, ids, ids, ids)
    with pytest.raises(AdtError):
        m.predict(None, ids, ids)


def test_lambdas_tables_and_candidate_mapping():
    from adt_b200.lambdas import get_lambdas, get_weight, candidate_to_lambdas
    assert get_lambdas("ml-1m") == ([0.104292, 0.065892], [0.100833, 0.000607])   # sasrec/utils.py:856
    assert get_lambdas("beauty") == ([0.0124, 0.122], [0.0001, 0.0])
    assert get_lambdas("nope") is None
    choice = [0, 0.0001, 0.0005, 0.001, 0.005, 0.01]
    cand = [0.7053411308078107, 0.9542592593410837, 0.9296478828883573, 0.28425047269448145, 0.1600125621449342, 0.47495464861462977]
    rec, ind = candidate_to_lambdas(cand, choice, choice)
    txt = open(os.path.join(os.path.dirname(__file__), "golden", "candidates_to_lambdas.txt")).read().strip()
    assert f"{rec} {ind}" == txt
    assert get_weight(choice, 0.0) == 0


def test_merge_topk_and_shards():
    from adt_b200.evaluate import merge_topk, shard_bounds
    rng = np.random.default_rng(0)
    U, I, K, S = 7, 203, 5, 3
    scores = torch.from_numpy(rng.standard_normal((U, I)).astype(np.float32))
    scores[:, 17] = scores[:, 23]  # an exact tie: lower id first
    bounds = [shard_bounds(I, S, r) for r in range(S)]
    assert bounds[0][0] == 0 and bounds[-1][1] == I and all(bounds[i][1] == bounds[i + 1][0] for i in range(S - 1))
    ps, pi = [], []
    for lo, hi in bounds:
        s, i = torch.topk(scores[:, lo:hi], min(K, hi - lo), dim=1)
        pad = K - s.shape[1]
        ps.append(torch.cat([s, torch.full((U, pad), float("-inf"))], 1))
        pi.append(torch.cat([(i + lo).int(), torch.full((U, pad), -1, dtype=torch.int32)], 1))
    ms, mi = merge_topk(torch.stack(ps), torch.stack(pi), K)
    order = np.lexsort((np.tile(np.arange(I), (U, 1)), -scores.numpy()), axis=1)[:, :K]
    assert np.array_equal(mi.numpy(), order)


def test_metrics_match_oracle():
    from adt_b200.evaluate import hit_ndcg_mrr, sampled_metrics
    from oracle import sasrec_oracle as O
    rng = np.random.default_rng(1)
    U, K = 50, 40
    pred = np.stack([rng.permutation(200)[:K] for _ in range(U)])
    answers = np.where(rng.random(U) < 0.6, pred[np.arange(U), rng.integers(0, K, U)], 999)
    ours = hit_ndcg_mrr(answers, pred)
    ref = O.full_sort_metrics(answers.reshape(-1, 1), pred)
    for k in ref:
        assert abs(ours[k] - ref[k]) < 1e-12, k
    logits = rng.standard_normal((U, 101)).astype(np.float32)
    (ndcg_r, hr_r), auc_r, rank_r = O.rank_metrics(-logits)
    rank = (logits[:, 1:] > logits[:, :1]).sum(1)
    assert np.array_equal(rank, rank_r)
    (ndcg, hr), auc = sampled_metrics(rank, 101)
    assert hr == hr_r and abs(auc - auc_r) < 1e-12 and all(abs(ndcg[k] - ndcg_r[k]) < 1e-6 for k in ndcg)


def _gloo_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from adt_b200.evaluate import merge_topk, shard_bounds
    from oracle import sasrec_oracle as O
    from helpers import load_golden, sd_from, ids
    # (1) item-sharded evaluation: local top-K on this rank's catalog slice, all_gather, merge == single-process top-K
    g = torch.Generator().manual_seed(5)
    U, I, H, K = 9, 101, 8, 4
    feats, E = torch.randn(U, H, generator=g), torch.randn(I, H, generator=g)
    lo, hi = shard_bounds(I, world, rank)
    s, i = torch.topk(feats @ E[lo:hi].t(), K, dim=1)
    gs = [torch.empty_like(s) for _ in range(world)]
    gi = [torch.empty(U, K, dtype=torch.int32) for _ in range(world)]
    dist.all_gather(gs, s.contiguous())
    dist.all_gather(gi, (i + lo).int().contiguous())
    ms, mi = merge_topk(torch.stack(gs), torch.stack(gi), K)
    ref = torch.topk(feats @ E.t(), K, dim=1)[1]
    ok1 = bool(torch.equal(mi.long(), ref))
    # (2) data-parallel loss normalisation: BCE is a mean over the valid positions of the GLOBAL batch (main.py:151-153),
    #     MSE/NLL means over global rows: all-reduced accumulators reproduce the single-process loss
    gd = load_golden("tiny_p0")
    d = gd["dims"]
    cfg = O.Cfg(d["I"], d["L"], d["H"], d["nh"], d["nl"], 0.0)
    sd = sd_from(gd)
    seq, dec, pos, neg = ids(gd)
    l1, l2, wd = list(gd["lambdas1"]), list(gd["lambdas2"]), float(gd["wd"])
    B = seq.shape[0]
    sl = slice(rank * B // world, (rank + 1) * B // world)
    out = O.forward(sd, cfg, seq[sl], dec[sl], pos[sl], neg[sl])
    valid = pos[sl] != 0
    acc = torch.zeros(3 + 2 * d["nl"], dtype=torch.float64)
    acc[0] = torch.nn.functional.softplus(-out["pos_logits"][valid]).double().sum()
    acc[1] = torch.nn.functional.softplus(out["neg_logits"][valid]).double().sum()
    acc[2] = valid.sum()
    for j in range(d["nl"]):     # decoder layer j pairs with enc_inputs[nl-1-j]; dec_outputs is already reversed
        i_enc = d["nl"] - 1 - j
        acc[3 + j] = ((out["enc_inputs"][i_enc] - out["dec_outputs"][i_enc]) ** 2).double().sum()
    for l in range(d["nl"]):
        r = out["rec_true"][l]
        acc[3 + d["nl"] + l] = -torch.diagonal(r, dim1=-2, dim2=-1).double().sum()
    dist.all_reduce(acc)
    Mg, Hh, nh, nl = B * d["L"], d["H"], d["nh"], d["nl"]
    total = (acc[0] + acc[1]) / acc[2]
    for j in range(nl):
        total = total + l1[nl - 1 - j] * acc[3 + j] / (Mg * Hh)
    for l in range(nl):
        total = total + l2[nl - 1] * acc[3 + nl + l] / (Mg * nh)
    total = total + wd * torch.norm(sd["item_emb.weight"]).double()
    ok2 = abs(float(total) - float(gd["loss"])) / abs(float(gd["loss"])) < 1e-5
    # (3) evolution: one candidate per rank, gathered fitness identical on every rank and equal to the serial result
    from adt_b200.evolution import evaluate_population
    cands = [np.array([0.1 * c, 0.05 * c + 0.2]) for c in range(5)]
    fit = lambda c: (float(c.sum()), float(c[0] * 2), float(c[1] - 1))
    res = evaluate_population(cands, fit)
    ok3 = bool(np.allclose(res, np.array([fit(c) for c in cands])))
    # ... and with the local fitness tuples computed up front (PopulationEvaluator: several candidates in flight per rank)
    from adt_b200.evolution import assign
    res2 = evaluate_population(cands, None, local=[fit(cands[c]) for c in assign(len(cands), world, rank)])
    ok3 = ok3 and bool(np.allclose(res2, res))
    ret[rank] = (ok1, ok2, ok3)
    dist.destroy_process_group()


def test_world_size_2_gloo_sharded_eval_and_dp_loss():
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 29500 + os.getpid() % 2000
    mp.spawn(_gloo_worker, args=(2, port, ret), nprocs=2, join=True)
    assert dict(ret) == {0: (True, True, True), 1: (True, True, True)}


def test_stosa_surface_on_cpu():
    """reference parameter names/shapes (fixtures hold the reference's own state_dict) and the loud no-CPU-fallback error."""
    from adt_b200.stosa import DisenDistSAModel
    from adt_b200._lib import AdtError
    z = np.load(os.path.join(GOLDEN, "stosa_beauty_p3.npz"))
    B, L, H, nh, nl, I = [int(v) for v in z["cfg"]]
    args = types.SimpleNamespace(item_size=I + 2, num_users=B, maxlen=L, hidden_units=H, num_heads=nh, num_layers=nl, dropout=0.3,
                                 attention_dropout=0.3, initializer_range=0.02, pvn_weight=0.005)
    m = DisenDistSAModel(args)
    ref = {k[4:]: z[k].shape for k in z.files if k.startswith("sd0/")}
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == ref
    assert list(m.state_dict().keys()) == list(ref.keys())
    with pytest.raises(AdtError):
        m.finetune(z["seq"], z["dec"], np.arange(B))
    with pytest.raises(ValueError):      # stosa/modules.py:191-194
        DisenDistSAModel(types.SimpleNamespace(**{**vars(args), "num_heads": 5}))


_REFERENCE_STAND_IN = '''
"""stand-in for the reference's sasrec/model.py: its module interface and parameter names over the oracle restatement"""
import torch
from adt_b200.model import SASRecADT as _Named
from oracle import sasrec_oracle as O


class SASRecADT(_Named):
    def _cfg(self):
        return O.Cfg(self.item_num, self.maxlen, self.hidden, self.num_heads, self.num_layers)

    def forward(self, user_ids, log_seqs, dec_seqs, pos_seqs, neg_seqs):
        ids = [torch.as_tensor(a).long() for a in (log_seqs, dec_seqs, pos_seqs, neg_seqs)]
        out = O.forward(dict(self.named_parameters()), self._cfg(), *ids)
        return out["pos_logits"], out["neg_logits"], out["enc_inputs"], out["dec_outputs"], out["rec_ind"]

    def predict(self, user_ids, log_seqs, item_indices, full=False):
        return O.predict(dict(self.named_parameters()), self._cfg(), torch.as_tensor(log_seqs).long(), item_indices, full)
'''


def test_bench_reference_arm_contract(tmp_path):
    """`bench.py --impl reference` (the CPU arm beside ours): rank 0 prints ONE JSON line with the same keys and the same
    workload string as our arm; every other rank exits 0 without work.  The arm runs the reference itself where its sources
    are found (oracle/ref_runner.ref_dir); they are not part of this repository, so elsewhere it runs a stand-in with the
    reference's module interface."""
    import json
    import subprocess
    import sys
    from oracle import ref_runner
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "0"]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    try:
        ref_runner.ref_dir()
    except RuntimeError:
        (tmp_path / "sasrec").mkdir()
        (tmp_path / "sasrec" / "model.py").write_text(_REFERENCE_STAND_IN)
        env["ADT_REFERENCE_DIR"] = str(tmp_path)
    other = subprocess.run(cmd, env={**env, "RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, capture_output=True, text=True, timeout=300)
    assert other.returncode == 0 and other.stdout.strip() == ""
    r0 = subprocess.run(cmd, env={**env, "RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"}, capture_output=True, text=True, timeout=600)
    assert r0.returncode == 0, r0.stderr[-2000:]
    lines = [ln for ln in r0.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "impl", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "train_seqs_per_sec" and d["unit"] == "seqs/s" and d["n_gpus"] == 2
    assert d["steps"] == 2 and d["warmup"] == 0                      # the arm honours --steps / --warmup (VERDICT r1)
    assert d["cpu_baseline"]["kind"] == "reference"                   # the label bench.py gives this arm, whichever model ran
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    assert d["config"]["workload"].startswith("SASRec-ADT C2: train step (items=12101, maxlen=50, hidden=64")
    assert set(d["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"} and d["cpu_baseline"]["kind"] in ("port", "reference")
    assert d["e2e"] == {"value": d["value"], "unit": "seqs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
