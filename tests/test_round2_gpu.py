"""Round-2 GPU parity tests (all through the C ABI): the benched configuration against the live oracle, the tensor-core
scorer at 100k / 1M items, the library's own candidate scoring / ranking / fused metrics, per-parameter Adam semantics
of the supernet optimiser, dropout streams of the compat path."""
import ctypes
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _c2_model(cfg, seed=0):
    from adt_b200.model import SASRecADT
    torch.manual_seed(seed)
    args = types.SimpleNamespace(device="cuda", num_heads=cfg["nh"], maxlen=cfg["L"], num_layers=cfg["nl"], hidden_units=cfg["H"], dropout=cfg["p"])
    m = SASRecADT(1, cfg["items"], args)
    for _, prm in m.named_parameters():
        if prm.dim() >= 2:
            torch.nn.init.xavier_normal_(prm.data)
    g = torch.Generator().manual_seed(seed + 1)
    for _, prm in m.named_parameters():
        if prm.dim() == 1:
            prm.data.add_(0.05 * torch.randn(prm.shape, generator=g))
    return m.cuda()


@pytest.mark.parametrize("precision,use_graph", [("bf16", True), ("fp32", True)])
def test_benched_c2_configuration_against_live_oracle(precision, use_graph):
    """EXACTLY what bench.py times -- C2 shape, B = 256, CUDA-graph replay, bf16 (and fp32) GEMM cores -- against the oracle
    evaluated live on the host with the same Philox streams: loss within 2e-2 (bf16) / 1e-5 (fp32), embedding gather bit exact,
    global gradient norm, and every parameter's gradient direction (cosine)."""
    from adt_b200 import synth
    _against_live_oracle(synth.CONFIGS["C2"], precision, use_graph)


@pytest.mark.parametrize("H,nh,use_graph,Lq", [(128, 2, False, 40), (256, 2, True, 40), (192, 3, False, 40), (128, 2, False, 100), (256, 2, True, 200)])
def test_wide_model_tcgen05_block_path_against_live_oracle(H, nh, use_graph, Lq):
    """wide models (H >= 128) in the bf16 mode take the tcgen05 block path (block_tc.cuh: every linear layer one adt_gemm_tc launch,
    warp-per-row kernels in between, forward AND backward; sequences longer than 64 also run attention as strided-batch tcgen05 GEMMs
    + a softmax row kernel): the same check as the benched configuration -- loss, gradient norm, bit-exact embedding gather,
    per-parameter gradient cosine -- against the oracle evaluated live on the host."""
    from adt_b200 import synth
    cfg = dict(synth.CONFIGS["C2"], H=H, nh=nh, L=Lq, B=32, items=3000)
    if Lq > 64:
        cfg.update(geo=1.0 / 60, lo=8, add=6)      # longer histories, so that the long rows are not mostly padding
    _against_live_oracle(cfg, "bf16", use_graph)


def _against_live_oracle(cfg, precision, use_graph):
    from adt_b200 import synth
    from adt_b200.lambdas import get_lambdas
    from adt_b200.trainer import FusedTrainer
    from oracle import sasrec_oracle as O
    m = _c2_model(cfg).train()
    sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    l1, l2 = get_lambdas(cfg["dataset"])
    rng = np.random.default_rng(7)
    b0, b1 = synth.make_batch(rng, cfg), synth.make_batch(rng, cfg)
    tr = FusedTrainer(m, l1, l2, weight_decay=cfg["wd"], seed=1234, use_graph=use_graph, precision=precision)
    # the compared step is a REPLAY of the captured graph: step 0 (another batch) captures and runs, then the initial weights are
    # restored in place (the parameters are views of the flat buffer the graph has baked in)
    eng = m.engine
    tr.step(*b1)
    torch.cuda.synchronize()
    with torch.no_grad():
        cur = m.state_dict()
        for k, v in sd.items():
            cur[k].copy_(v.detach().cuda())
        eng.adam_m.zero_(); eng.adam_v.zero_()
    step_idx = tr.t
    w = tr.step(*b0)
    loss = tr.loss()
    gn = tr.grad_norm()
    ocfg = O.Cfg(cfg["items"], cfg["L"], cfg["H"], cfg["nh"], cfg["nl"], cfg["p"])
    batch = tuple(torch.from_numpy(a).long() for a in b0)
    loss_ref, _, gn_ref, _, out = O.train_step(sd, ocfg, batch, l1, l2, cfg["wd"], drop=O.Drop(cfg["p"], 1234, step_idx))
    tol = 2e-2 if precision == "bf16" else 1e-5
    assert abs(loss - float(loss_ref)) / abs(float(loss_ref)) < tol, (loss, float(loss_ref))
    assert abs(gn - float(gn_ref)) / float(gn_ref) < (2e-2 if precision == "bf16" else 1e-4), (gn, float(gn_ref))
    # embedding gather (+ scale, position, dropout, pad mask) is fp32 in both modes: bit exact against the oracle's first block input
    x0 = w["x"][0].cpu().numpy().reshape(cfg["B"], cfg["L"], cfg["H"])
    assert np.array_equal(x0, out["enc_inputs"][0].detach().numpy())
    worst = 1.0
    for k, _ in eng.order:
        if sd[k].grad is None:
            continue
        a = eng.grad_view(k).detach().cpu().numpy().ravel().astype(np.float64)     # holds the CLIPPED gradient after the step
        b = sd[k].grad.numpy().ravel().astype(np.float64)
        if np.linalg.norm(b) > 1e-7:
            worst = min(worst, float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30)))
    assert worst > (0.99 if precision == "bf16" else 0.9999), worst


def test_compat_forward_draws_fresh_dropout_masks_every_training_step():
    """ADVICE r1 (high): the reference loop calls model(u, seq, dec, pos, neg) once per step; every call must use a new dropout
    stream, and backward() must re-draw the masks of ITS forward."""
    from adt_b200 import testing as T
    g = T.load_golden("tiny_p5")
    m = T.model_from_golden(g).train()
    outs = [m(None, g["seq"], g["dec"], g["pos"], g["neg"]) for _ in range(2)]
    assert m.engine.drop_step == 2
    assert not torch.equal(outs[0][2][1], outs[1][2][1])          # second encoder block input differs: different masks
    # gradient of step k must equal the gradient computed right after forward k (no stale mask): forward, forward, backward(first) raises
    with pytest.raises(Exception):
        outs[0][0].sum().backward()
    m2 = T.model_from_golden(g).train()
    m2.engine.drop_step = 1
    o2 = m2(None, g["seq"], g["dec"], g["pos"], g["neg"])
    assert torch.equal(o2[0], outs[1][0])                         # same step index -> same masks -> identical logits
    m.eval()
    e1 = m(None, g["seq"], g["dec"], g["pos"], g["neg"])
    assert m.engine.drop_step == 2                                # eval forwards do not advance the stream


def test_predict_accepts_shared_candidate_list_and_checks_ids():
    """reference broadcasting: item_indices [B,C] or one 1-D list [C] (utils.evaluate / evaluate_valid); ids out of range raise
    instead of reading out of bounds; full=True equals the candidate scores of every id."""
    from adt_b200 import testing as T
    g = T.load_golden("tiny_p5")
    m = T.model_from_golden(g, prefix="sd1/").eval()      # the fixture's predictions were taken after its optimisation step
    B = g["seq"].shape[0]
    I = g["dims"]["I"]
    full = m.predict(None, g["seq"], None, True)
    assert full.shape == (B, I + 1)
    assert np.allclose(full.cpu().numpy(), g["pred_full"], rtol=1e-4, atol=2e-5)
    c2 = m.predict(None, g["seq"], g["cand"])
    assert np.allclose(c2.cpu().numpy(), g["pred_cand"], rtol=1e-4, atol=2e-5)
    shared = np.arange(1, 8)
    c1 = m.predict(None, g["seq"], shared)
    assert c1.shape == (B, 7)
    assert torch.allclose(c1, full[:, 1:8], rtol=1e-5, atol=1e-6)
    with pytest.raises(IndexError):
        m.predict(None, g["seq"], np.array([I + 5]))
    with pytest.raises(IndexError):
        bad = g["seq"].copy(); bad[0, -1] = I + 1
        m.predict(None, bad, shared)


def test_sampled_rank_and_fused_metrics_match_reference_protocol():
    """evaluate_loader (utils.py:395-428): rank of column 0 by double argsort, HR/NDCG@5,10, MRR, AUC with C+1 -- the library's
    gather-dot + rank-count + metric sums against the oracle's restatement on the same scores."""
    from adt_b200 import testing as T
    from adt_b200.evaluate import sampled_rank, sampled_metrics_from_acc
    from oracle import sasrec_oracle as O
    g = T.load_golden("c2mini_p5")
    m = T.model_from_golden(g).eval()
    rng = np.random.default_rng(3)
    U, C = g["seq"].shape[0], 101
    item_idx = np.stack([rng.permutation(g["dims"]["I"])[:C] + 1 for _ in range(U)])      # distinct candidates: no exact score ties
    acc = torch.zeros(7, dtype=torch.float64, device="cuda")
    rank, scores = sampled_rank(m, g["seq"], item_idx, metric_acc=acc)
    pred = -scores.cpu()
    ref_rank = pred.argsort(dim=1).argsort(dim=1)[:, 0].numpy()
    assert np.array_equal(rank.cpu().numpy(), ref_rank)
    (ndcg, hr), auc, mrr = sampled_metrics_from_acc(acc)
    (o_ndcg, o_hr), o_auc, o_rank = O.rank_metrics(pred)
    assert np.array_equal(o_rank, ref_rank)
    for k in (5, 10):
        assert abs(hr[k] - o_hr[k]) < 1e-12 and abs(ndcg[k] - o_ndcg[k]) < 1e-6
    assert abs(auc - o_auc) < 1e-12
    r = ref_rank.astype(np.float64)
    for k in (5, 10):
        assert abs(hr[k] - float((r < k).mean())) < 1e-12
        assert abs(ndcg[k] - float(np.where(r < k, 1.0 / np.log2(r + 2.0), 0.0).mean())) < 1e-9
    assert abs(auc - float(np.mean(((C + 1) - (r + 1)) / C))) < 1e-12
    assert abs(mrr - float(np.mean(1.0 / (r + 1)))) < 1e-12


@pytest.mark.parametrize("I,H", [(100_000, 64), (100_000, 256), (100_000, 192), (1_000_000, 64), (1_000_000, 256)])
def test_tensor_core_scorer_large_catalogs_match_full_sort(I, H):
    """adt_score_topk_tc at 100k / 1M items (n_splits > 1: cross-split threshold exchange, n_splits*KC up to 2048), U = 512:
    ids identical to the oracle's full_sort_topk on fp32 scores (up to rounding-level ties), seen items excluded, and the fused
    HIT/NDCG/MRR sums equal to the oracle's metrics of the same lists."""
    from adt_b200.evaluate import CatalogScorer, metrics_from_acc
    from oracle import sasrec_oracle as O
    U, K = 512, 10
    g = torch.Generator().manual_seed(I // 1000 + H)
    E = torch.randn(I + 1, H, generator=g) * 0.1
    feats = torch.randn(U, H, generator=g)
    rng = np.random.default_rng(5)
    seen = [np.unique(rng.integers(1, I + 1, size=rng.integers(0, 40))) for _ in range(U)]
    indptr = np.zeros(U + 1, np.int32)
    indptr[1:] = np.cumsum([len(s) for s in seen])
    idx = np.concatenate(seen).astype(np.int32)
    fake = types.SimpleNamespace(item_emb=types.SimpleNamespace(weight=E.cuda()), hidden=H)
    sc = CatalogScorer(fake, K=K, use_tensor_cores=True)
    assert sc._uses_tc(H, 0, I + 1)
    # reference ranking in chunks of users (the [U, I+1] fp32 score matrix of 1M x 512 is 2 GB)
    ref = np.zeros((U, K), np.int64)
    scores_at = []
    for u0 in range(0, U, 64):
        s = (feats[u0:u0 + 64] @ E.t()).numpy()
        ref[u0:u0 + 64] = O.full_sort_topk(s, seen[u0:u0 + 64], k=K)
        scores_at.append(s)
    answers = ref[np.arange(U), rng.integers(0, K, size=U)]
    answers[::3] = 1 + (np.arange(len(answers[::3])) % I)          # a third of the users: an arbitrary (mostly missed) answer
    acc = torch.zeros(6, dtype=torch.float64, device="cuda")
    s_, ids = sc.topk_from_feats(feats.cuda(), indptr, idx, answers=answers.astype(np.int32), metric_acc=acc)
    ids = ids.cpu().numpy()
    mism = 0
    for u in range(U):
        srow = scores_at[u // 64][u % 64]
        for r in range(K):
            if ids[u, r] != ref[u, r]:
                mism += 1
                assert abs(srow[ids[u, r]] - srow[ref[u, r]]) <= 2e-6 * np.abs(srow).max(), (u, r)
        assert not set(ids[u].tolist()) & set(seen[u].tolist())
    assert mism <= U * K // 200
    got = metrics_from_acc(acc)
    exp = O.full_sort_metrics(answers.reshape(-1, 1), ids)
    for key in ("HIT@5", "NDCG@5", "HIT@10", "NDCG@10", "MRR"):
        assert abs(got[key] - exp[key]) < 1e-9, (key, got[key], exp[key])
    first = np.array([np.where(ids[u] == answers[u])[0][0] if (ids[u] == answers[u]).any() else -1 for u in range(U)])
    assert got["users"] == U
    assert abs(got["HIT@10"] - float((first >= 0).mean())) < 1e-12
    assert abs(got["HIT@5"] - float(((first >= 0) & (first < 5)).mean())) < 1e-12
    assert abs(got["NDCG@10"] - float(np.where(first >= 0, 1.0 / np.log2(first + 2.0), 0.0).mean())) < 1e-9
    assert abs(got["MRR"] - float(np.where(first >= 0, 1.0 / (first + 1.0), 0.0).mean())) < 1e-9


def test_stale_bf16_table_is_refreshed_after_training_steps():
    """ADVICE r1 (medium): a CatalogScorer kept across training must not generate tensor-core candidates from an old table."""
    from adt_b200.evaluate import CatalogScorer
    H, I, U = 64, 40_000, 64
    g = torch.Generator().manual_seed(1)
    E = (torch.randn(I + 1, H, generator=g) * 0.1).cuda()
    fake = types.SimpleNamespace(item_emb=types.SimpleNamespace(weight=E), hidden=H)
    feats = torch.randn(U, H, generator=g).cuda()
    sc = CatalogScorer(fake, K=10)
    _, i0 = sc.topk_from_feats(feats)
    i0 = i0.clone()
    with torch.no_grad():
        E.copy_(torch.randn(I + 1, H, generator=g).cuda() * 0.1)     # in-place update (bumps the tensor version)
    _, i1 = sc.topk_from_feats(feats)
    ex = CatalogScorer(fake, K=10, use_tensor_cores=False)
    _, ie = ex.topk_from_feats(feats)
    assert torch.equal(i1, ie) and not torch.equal(i0, i1)
    # raw-pointer updates (this package's optimisers) announce themselves through _adt_param_version
    E.data.view(-1)[:].mul_(1.0)        # no semantic change; now emulate a raw update
    fake._adt_param_version = 1
    key0 = sc._tab_key
    sc.topk_from_feats(feats)
    assert sc._tab_key != key0


def test_segmented_adam_matches_torch_adam_when_active_parameters_change():
    """VERDICT r1 item 3: FlatOptimizer on a model whose active parameter set changes every step (supernet set_choice) must match
    torch.optim.Adam(weight_decay=...) + clip_grad_norm_ elementwise: untouched parameters are not decayed, keep their moments and
    their own step count."""
    from adt_b200.dp import FlatOptimizer
    torch.manual_seed(0)

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.blocks = torch.nn.ModuleList(torch.nn.Linear(16, 16) for _ in range(5))
            self.emb = torch.nn.Embedding(30, 16)

        def forward(self, ids, active):
            x = self.emb(ids)
            for i in active:
                x = torch.tanh(self.blocks[i](x))
            return x.pow(2).mean()

    a, b = Net().cuda(), Net().cuda()
    b.load_state_dict(a.state_dict())
    opt_a = FlatOptimizer(a, lr=1e-2, betas=(0.9, 0.999), weight_decay=1e-2, clip=0.05)
    opt_b = torch.optim.Adam(b.parameters(), lr=1e-2, betas=(0.9, 0.999), weight_decay=1e-2)
    ids = torch.randint(0, 30, (8, 5)).cuda()
    for active in ([0, 1], [1, 3], [0, 1, 2, 3, 4], [4], [1, 3]):
        opt_a.zero_grad()
        a(ids, active).backward()
        opt_a.step()
        opt_b.zero_grad(set_to_none=True)
        b(ids, active).backward()
        torch.nn.utils.clip_grad_norm_(b.parameters(), 0.05)
        opt_b.step()
        for (n, pa), (_, pb) in zip(a.named_parameters(), b.named_parameters()):
            assert torch.allclose(pa, pb, rtol=2e-5, atol=2e-7), (active, n, float((pa - pb).abs().max()))
    assert not opt_a.uniform


def test_workspace_bytes_reports_what_the_engine_allocates():
    from adt_b200 import _lib as L
    q = L.fill(L.adt_workspace_query(), B=256, L=50, H=64, nh=2, nl=2, K=10, n_splits=37)
    sz = L.adt_workspace_sizes()
    L.check(L.lib().adt_workspace_bytes(ctypes.byref(q), ctypes.byref(sz)))
    M = 256 * 50
    assert sz.sort_keys == 4 * 4 * M * 4
    assert sz.score_part == 37 * 256 * 10 * 8
    assert sz.saved > 0 and sz.scratch > 0 and sz.scatter_rows == 2 * ((4 * M + 31) // 32) * 64 * 4


def test_reference_staging_runs_on_this_box():
    """the staged reference sources (oracle/build_ref.py) must import and step without the reference checkout, because bench.py's
    reference arm and cpu_baseline leg run them.  The reference's sources are not part of this repository: skipped without them."""
    from oracle import ref_runner as R
    from adt_b200 import synth
    try:
        R.ref_dir()
    except RuntimeError as e:
        pytest.skip(str(e))
    cfg = dict(synth.CONFIGS["C2"], B=8)
    tr = R.RefTrainer(cfg, [0.0124, 0.122], [0.0001, 0.0], device="cpu")
    rng = np.random.default_rng(0)
    l0 = tr.step(*synth.make_batch(rng, cfg))
    assert np.isfinite(l0)


@pytest.mark.parametrize("nh,Lq", [(2, 50), (4, 64), (1, 33)])
def test_sequence_resident_block_kernels_match_row_tile_kernels(nh, Lq):
    """the one-CTA-per-sequence evaluation encoder (kernels_seq.cuh, ADT_SEQ_FUSED=1) against the 3-kernel row-tile forward it replaces
    (=0): both runs train with the row-tile kernels, so the three training steps agree; the evaluation pass then sees the same bf16
    operands and its top-10 ids and scores agree to bf16-flip level."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = []
    for fused in ("0", "1"):
        env = dict(os.environ, ADT_SEQ_FUSED=fused)
        r = subprocess.run([sys.executable, os.path.join(root, "tools", "seq_ab.py"), str(nh), str(Lq)], capture_output=True, text=True, env=env,
                           timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        res.append(json.loads(r.stdout.strip().splitlines()[-1]))
    a, b = res
    for k in range(3):
        assert abs(a["loss"][k] - b["loss"][k]) / abs(a["loss"][k]) < 2e-5, (k, a["loss"], b["loss"])
        assert abs(a["gnorm"][k] - b["gnorm"][k]) / a["gnorm"][k] < 1e-3, (k, a["gnorm"], b["gnorm"])
        assert abs(a["gsum"][k] - b["gsum"][k]) / a["gsum"][k] < 1e-3
    assert abs(a["psum"] - b["psum"]) / a["psum"] < 1e-4
    # three optimisation steps with fp32-atomic weight gradients later, near-ties of a 12k-item catalog may swap places
    same = np.mean(np.array(a["ids"]) == np.array(b["ids"]))
    assert same > 0.9, same
    assert np.abs(np.array(a["scores"]) - np.array(b["scores"])).max() < 1e-2


def _ab_wide(env_name, nh, Lq, Hd):
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = []
    for v in ("0", "1"):
        env = dict(os.environ, **{env_name: v})
        r = subprocess.run([sys.executable, os.path.join(root, "tools", "seq_ab.py"), str(nh), str(Lq), str(Hd)], capture_output=True, text=True,
                           env=env, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        res.append(json.loads(r.stdout.strip().splitlines()[-1]))
    return res


@pytest.mark.parametrize("nh,Lq,Hd", [(2, 50, 128), (2, 40, 256), (3, 33, 192)])
def test_hoisted_tcgen05_weight_gradients_match_in_kernel_ones(nh, Lq, Hd):
    """wide models in the bf16 mode: the backward row-tile kernels write bf16 copies of their dY / X tiles and each weight gradient is one
    split-K tcgen05 GEMM reading both MN-major (ADT_WGRAD_HOIST=1, the default) -- against the in-kernel mma.sync + atomics path (=0):
    same bf16 operand rounding, so every parameter's gradient norm, the losses and the updated parameters agree to accumulation order."""
    a, b = _ab_wide("ADT_WGRAD_HOIST", nh, Lq, Hd)
    for n, v in a["gnorms"].items():
        assert abs(v - b["gnorms"][n]) <= 2e-4 * max(v, 1e-6) + 1e-9, (n, v, b["gnorms"][n])
    for k in range(3):
        assert abs(a["loss"][k] - b["loss"][k]) / abs(a["loss"][k]) < 2e-5, (k, a["loss"], b["loss"])
        assert abs(a["gnorm"][k] - b["gnorm"][k]) / a["gnorm"][k] < 1e-3, (k, a["gnorm"], b["gnorm"])
    assert abs(a["psum"] - b["psum"]) / a["psum"] < 1e-4


@pytest.mark.parametrize("nh,Lq,Hd", [(2, 50, 128), (2, 40, 256), (3, 33, 192)])
def test_tcgen05_forward_path_matches_row_tile_kernels(nh, Lq, Hd):
    """wide models in the bf16 mode: forward of the encoder / decoder blocks as tcgen05 GEMMs + warp-per-row kernels (block_tc.cuh,
    ADT_FWD_TC=1, the default) against the row-tile kernels (=0): same bf16 operand rounding, same Philox dropout streams, same saved
    activations -> losses, gradient norms, updated parameters and the evaluation top-10 agree to bf16-flip level."""
    a, b = _ab_wide("ADT_FWD_TC", nh, Lq, Hd)
    for k in range(3):
        assert abs(a["loss"][k] - b["loss"][k]) / abs(a["loss"][k]) < 2e-4, (k, a["loss"], b["loss"])
        assert abs(a["gnorm"][k] - b["gnorm"][k]) / a["gnorm"][k] < 5e-3, (k, a["gnorm"], b["gnorm"])
    for n, v in a["gnorms"].items():
        assert abs(v - b["gnorms"][n]) <= 5e-3 * max(v, 1e-6) + 1e-8, (n, v, b["gnorms"][n])
    assert abs(a["psum"] - b["psum"]) / a["psum"] < 1e-4
    assert np.mean(np.array(a["ids"]) == np.array(b["ids"])) > 0.8      # near-ties of the 12k-item catalog swap after three bf16 steps
    assert np.abs(np.array(a["scores"]) - np.array(b["scores"])).max() < 2e-2


@pytest.mark.parametrize("nh,Lq,Hd", [(2, 50, 128), (2, 40, 256), (3, 33, 192)])
def test_tcgen05_backward_path_matches_row_tile_kernels(nh, Lq, Hd):
    """wide models in the bf16 mode: backward of the encoder / decoder blocks as tcgen05 dgrad / wgrad GEMMs + warp-per-row adjoint kernels
    (block_tc.cuh, ADT_BWD_TC=1, the default) against the row-tile kernels (=0, with hoisted weight gradients): per-parameter gradient
    norms, losses, global gradient norms and updated parameters agree to bf16-flip level."""
    a, b = _ab_wide("ADT_BWD_TC", nh, Lq, Hd)
    for n, v in a["gnorms"].items():
        assert abs(v - b["gnorms"][n]) <= 5e-3 * max(v, 1e-6) + 1e-8, (n, v, b["gnorms"][n])
    for k in range(3):
        assert abs(a["loss"][k] - b["loss"][k]) / abs(a["loss"][k]) < 2e-4, (k, a["loss"], b["loss"])
        assert abs(a["gnorm"][k] - b["gnorm"][k]) / a["gnorm"][k] < 5e-3, (k, a["gnorm"], b["gnorm"])
    assert abs(a["psum"] - b["psum"]) / a["psum"] < 1e-4


@pytest.mark.parametrize("nh,Lq,Hd", [(2, 100, 128), (2, 200, 256), (3, 70, 192)])
def test_tcgen05_batched_attention_matches_row_tile_attention(nh, Lq, Hd):
    """sequences longer than 64 on the tcgen05 block path: attention as strided-batch GEMMs over (sequence, head) with the scores in HBM
    (ADT_ATTN_TC=1, the default) against the generic row-tile attention kernels (=0): same masks, same Philox dropout stream."""
    a, b = _ab_wide("ADT_ATTN_TC", nh, Lq, Hd)
    for k in range(3):
        assert abs(a["loss"][k] - b["loss"][k]) / abs(a["loss"][k]) < 2e-4, (k, a["loss"], b["loss"])
        assert abs(a["gnorm"][k] - b["gnorm"][k]) / a["gnorm"][k] < 5e-3, (k, a["gnorm"], b["gnorm"])
    for n, v in a["gnorms"].items():
        assert abs(v - b["gnorms"][n]) <= 5e-3 * max(v, 1e-6) + 1e-8, (n, v, b["gnorms"][n])
    assert abs(a["psum"] - b["psum"]) / a["psum"] < 1e-4


@pytest.mark.parametrize("M,N,K,act", [(256, 256, 256, 0), (1000, 768, 256, 2), (333, 200, 1024, 1), (2048, 26844, 256, 0), (130, 64, 72, 3)])
def test_tcgen05_linear_matches_fp32_linear(M, N, K, act):
    """adt_gemm_tc (TMA + tcgen05.mma, bf16 operands, fp32 accumulate) behind ops.linear(precision=1): forward, input gradient,
    weight gradient and bias gradient against torch fp32 on the bf16-rounded operands (the rounding is the only difference)."""
    from adt_b200 import ops
    g = torch.Generator().manual_seed(M + N + K)
    x = (torch.randn(M, K, generator=g) * 0.5).cuda().requires_grad_(True)
    W = (torch.randn(N, K, generator=g) * 0.05).cuda().requires_grad_(True)
    b = (torch.randn(N, generator=g) * 0.1).cuda().requires_grad_(True)
    dy = torch.randn(M, N, generator=g).cuda()
    old = ops.TC_MIN_WORK
    ops.TC_MIN_WORK = 0
    try:
        y = ops.linear(x, W, b, act=act, scale=0.5, precision=1)
        gx, gW, gb = torch.autograd.grad(y, (x, W, b), dy)
    finally:
        ops.TC_MIN_WORK = old
    r = lambda t: t.detach().to(torch.bfloat16).float()
    xr, Wr = r(x).requires_grad_(True), r(W).requires_grad_(True)
    br = b.detach().clone().requires_grad_(True)
    pre = (xr @ Wr.t() + br) * 0.5
    fn = {0: lambda t: t, 1: torch.relu, 2: lambda t: torch.nn.functional.gelu(t), 3: torch.nn.functional.elu}[act]
    yr = fn(pre)
    assert torch.allclose(y, yr, rtol=2e-3, atol=2e-3), float((y - yr).abs().max())
    # backward products round dy / x / W to bf16 too: compare against the same rounding
    dpre = torch.autograd.grad(yr, pre, dy, retain_graph=True)[0]
    dq = r(dpre)
    gx_ref = (dq @ Wr.detach()) * 0.5
    gW_ref = (dq.t() @ xr.detach()) * 0.5
    gb_ref = dpre.sum(0) * 0.5
    for got, ref, name in ((gx, gx_ref, "dx"), (gW, gW_ref, "dW"), (gb, gb_ref, "db")):
        err = float((got - ref).abs().max() / (ref.abs().max() + 1e-12))
        assert err < 5e-3, (name, err)


@pytest.mark.parametrize("B,nh,Lq,hd", [(3, 2, 200, 128), (2, 4, 70, 64), (2, 3, 129, 32)])
def test_tcgen05_batched_gemm_over_heads_and_sequences(B, nh, Lq, hd):
    """adt_gemm_tc as a strided batch (4-D TMA maps: columns, rows, head, sequence): the two products of attention on head slices of
    [B, L, H] tensors -- S = Q K^T (both K-major) and ctx = P V (V read MN-major), plus dK = dS^T Q (both MN-major) -- against torch
    on the same bf16-rounded operands."""
    import ctypes
    from adt_b200 import _lib as L
    lib = L.lib()
    H = nh * hd
    g = torch.Generator().manual_seed(B * 1000 + Lq)
    r = lambda *s: (torch.randn(*s, generator=g) * 0.3).cuda()
    q, k, v = r(B, Lq, H), r(B, Lq, H), r(B, Lq, H)
    qb, kb, vb = q.bfloat16().contiguous(), k.bfloat16().contiguous(), v.bfloat16().contiguous()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    Lp = (Lq + 7) // 8 * 8
    S = torch.zeros(B, nh, Lq, Lp, device="cuda")
    a = L.fill(L.adt_gemm_tc_args(), a_bf16=qb, b_bf16=kb, lda=H, ldb=H, c=S, ldc=Lp, M=Lq, N=Lq, K=hd, scale=1.0, batch_inner=nh, batch_outer=B,
               a_so=Lq * H, a_si=hd, b_so=Lq * H, b_si=hd, c_so=nh * Lq * Lp, c_si=Lq * Lp)
    L.check(lib.adt_gemm_tc(ctypes.byref(a), st), "adt_gemm_tc")
    qh = qb.float().view(B, Lq, nh, hd).permute(0, 2, 1, 3)
    kh = kb.float().view(B, Lq, nh, hd).permute(0, 2, 1, 3)
    vh = vb.float().view(B, Lq, nh, hd).permute(0, 2, 1, 3)
    S_ref = qh @ kh.transpose(-1, -2)
    assert torch.allclose(S[..., :Lq], S_ref, rtol=1e-3, atol=1e-3), float((S[..., :Lq] - S_ref).abs().max())
    # ctx = P V with P [B, nh, L, Lp] bf16 (zero beyond L) and V read MN-major from its [B, L, H] home
    P = torch.zeros(B, nh, Lq, Lp, device="cuda", dtype=torch.bfloat16)
    P[..., :Lq] = torch.softmax(S_ref, -1).bfloat16()
    ctx = torch.zeros(B, Lq, H, device="cuda")
    a = L.fill(L.adt_gemm_tc_args(), a_bf16=P, b_bf16=vb, lda=Lp, ldb=H, c=ctx, ldc=H, M=Lq, N=hd, K=Lq, scale=1.0, b_mn=1, batch_inner=nh,
               batch_outer=B, a_so=nh * Lq * Lp, a_si=Lq * Lp, b_so=Lq * H, b_si=hd, c_so=Lq * H, c_si=hd)
    L.check(lib.adt_gemm_tc(ctypes.byref(a), st), "adt_gemm_tc")
    ctx_ref = (P[..., :Lq].float() @ vh).permute(0, 2, 1, 3).reshape(B, Lq, H)
    assert torch.allclose(ctx, ctx_ref, rtol=2e-3, atol=2e-3), float((ctx - ctx_ref).abs().max())
    # dK = dS^T Q: both operands MN-major (dS as [K = query][M = key], Q as [K = query][N = d])
    dk = torch.zeros(B, Lq, H, device="cuda")
    a = L.fill(L.adt_gemm_tc_args(), a_bf16=P, b_bf16=qb, lda=Lp, ldb=H, c=dk, ldc=H, M=Lq, N=hd, K=Lq, scale=1.0, a_mn=1, b_mn=1, batch_inner=nh,
               batch_outer=B, a_so=nh * Lq * Lp, a_si=Lq * Lp, b_so=Lq * H, b_si=hd, c_so=Lq * H, c_si=hd)
    L.check(lib.adt_gemm_tc(ctypes.byref(a), st), "adt_gemm_tc")
    dk_ref = (P[..., :Lq].float().transpose(-1, -2) @ qh).permute(0, 2, 1, 3).reshape(B, Lq, H)
    assert torch.allclose(dk, dk_ref, rtol=2e-3, atol=2e-3), float((dk - dk_ref).abs().max())
