"""Host-side contract of hidden sizes beyond 256 (SASRec-ADT / Bert4Rec-ADT up to H = 512): every shape no path serves is refused with
an error that names its limit, the workspace query reports the scratch of the tcgen05 block path at H 384 / 512, and the sizes of the
shapes accepted before are unchanged."""
import ctypes

import pytest


def _lib():
    from adt_b200 import _lib as L
    try:
        lib = L.lib()
    except L.AdtError:
        pytest.skip("libadt_b200.so not built")
    lib.adt_attention_scratch_bytes.restype = ctypes.c_int64
    return L, lib


def _ws(L, lib, B, Lq, H, nh):
    q = L.fill(L.adt_workspace_query(), B=B, L=Lq, H=H, nh=nh, nl=2, K=10, n_splits=1)
    sz = L.adt_workspace_sizes()
    L.check(lib.adt_workspace_bytes(ctypes.byref(q), ctypes.byref(sz)), "adt_workspace_bytes")
    return {k: int(getattr(sz, k)) for k, _ in sz._fields_}


E_SHAPE = -1      # ADT_E_SHAPE of include/adt_b200.h
BLOCK_ENTRIES = ("adt_enc_block_fwd", "adt_enc_block_bwd", "adt_dec_block_fwd", "adt_dec_block_bwd")


def _struct(L, f):
    return {"adt_enc_block_fwd": L.adt_enc_block_fwd_args, "adt_enc_block_bwd": L.adt_enc_block_bwd_args,
            "adt_dec_block_fwd": L.adt_dec_block_fwd_args, "adt_dec_block_bwd": L.adt_dec_block_bwd_args}[f]


@pytest.mark.parametrize("Lq,H,nh,precision,msg", [
    (40, 384, 4, 0, "H > 256 needs precision 1"),            # the fp32 parity mode stays at H <= 256
    (600, 512, 8, 0, "H > 256 needs precision 1"),
    (40, 576, 4, 1, "H > 512"),
    (40, 1024, 8, 1, "H > 512"),
    (40, 288, 4, 1, "H % 64 == 0"),                          # hd 72 would pass every other rule
    (40, 416, 4, 1, "H % 64 == 0"),
    (40, 384, 2, 1, "multiple of 32 and at most 128"),       # hd 192
    (40, 512, 2, 1, "multiple of 32 and at most 128"),       # hd 256
    (40, 384, 8, 1, "multiple of 32 and at most 128"),       # hd 48
    (300, 320, 10, 1, "nh<=8"),
])
def test_wide_refusals_name_the_limit(Lq, H, nh, precision, msg):
    L, lib = _lib()
    for f in BLOCK_ENTRIES:
        b = L.fill(_struct(L, f)(), B=2, L=Lq, H=H, nh=nh, precision=precision)
        rc = getattr(lib, f)(ctypes.byref(b), None)
        assert rc == E_SHAPE, (f, rc)
        with pytest.raises(L.AdtError, match=msg):
            L.check(rc, f)
    a = L.fill(L.adt_attention_args(), B=2, L=Lq, H=H, nh=nh, mask_mode=0, training=0, precision=precision)
    for f in ("adt_attention_fwd", "adt_attention_bwd"):
        with pytest.raises(L.AdtError, match=msg):
            L.check(getattr(lib, f)(ctypes.byref(a), None), f)
    if precision:     # the workspace query assumes the bf16 mode: it refuses every other limit
        with pytest.raises(L.AdtError, match=msg):
            _ws(L, lib, 2, Lq, H, nh)


def test_row_kernels_refuse_beyond_512():
    L, lib = _lib()
    f = L.fill(L.adt_final_fwd_args(), M=4, H=576)
    with pytest.raises(L.AdtError, match="final_fwd: H"):
        L.check(lib.adt_final_logits_loss_fwd(ctypes.byref(f), None), "final_fwd")
    fb = L.fill(L.adt_final_bwd_args(), M=4, H=576)
    with pytest.raises(L.AdtError, match="final_bwd: H"):
        L.check(lib.adt_final_logits_loss_bwd(ctypes.byref(fb), None), "final_bwd")
    d = L.fill(L.adt_drl_args(), M=4, H=576)
    for fn in ("adt_drop_res_ln_fwd", "adt_drop_res_ln_bwd"):
        with pytest.raises(L.AdtError, match="H <= 512"):
            L.check(getattr(lib, fn)(ctypes.byref(d), None), fn)
    e = L.fill(L.adt_embed_fwd_args(), B=2, L=4, H=576)
    with pytest.raises(L.AdtError, match="H > 512"):
        L.check(lib.adt_embed_fwd(ctypes.byref(e), None), "embed_fwd")


def test_catalog_scorers_refuse_beyond_512():
    L, lib = _lib()
    s = L.fill(L.adt_score_topk_args(), U=4, H=576, n_items=100, K=10, n_splits=1)
    assert lib.adt_score_topk(ctypes.byref(s), None) == E_SHAPE
    t = L.fill(L.adt_score_topk_tc_args(), U=4, H=576, n_items=100, K=10, KC=32, n_splits=1)
    assert lib.adt_score_topk_tc(ctypes.byref(t), None) == E_SHAPE
    t = L.fill(L.adt_score_topk_tc_args(), U=4, H=480, n_items=100, K=10, KC=32, n_splits=1)      # not a multiple of 64
    assert lib.adt_score_topk_tc(ctypes.byref(t), None) == E_SHAPE


def _tc_sizes(B, Lq, H, nh):
    """bytes the tcgen05 block path addresses: forward 9 operand slots, backward 12, of M*H bf16 each; 10 bf16 H x H weights; the
    batched attention's area (L 65..256: packed bf16 q|k|v (+ dctx), fp32 scores (+ dP), bf16 P (+ dS)) behind them"""
    M, Lp = B * Lq, (Lq + 7) // 8 * 8
    zll = M * nh * Lp if Lq <= 256 else 0
    fwd = 9 * M * H * 2 + 10 * H * H * 2 + 1024 + 3 * M * H * 2 + zll * 6
    bwd = 12 * M * H * 2 + 10 * H * H * 2 + 1024 + 4 * M * H * 2 + zll * 12
    return fwd, bwd


@pytest.mark.parametrize("H,nh", [(320, 5), (384, 3), (384, 4), (384, 6), (448, 7), (512, 4), (512, 8)])
@pytest.mark.parametrize("B,Lq", [(2, 40), (4, 200), (2, 512), (1, 2048)])
def test_wide_workspace_sizes(H, nh, B, Lq):
    L, lib = _lib()
    if (H // nh) % 32:
        pytest.skip("head size not a multiple of 32")
    ws = _ws(L, lib, B, Lq, H, nh)
    fwd, bwd = _tc_sizes(B, Lq, H, nh)
    assert ws["fwd_scratch"] == fwd
    assert ws["wgrad_scratch"] == bwd
    M = B * Lq
    if Lq > 256:   # flash attention: packed bf16 operands + bf16 dctx + row sums, no L^2 term
        assert ws["attn_scratch"] == 256 + M * 3 * H * 2 + M * H * 2 + M * nh * 4
        assert lib.adt_attention_scratch_bytes(B, Lq, H, nh, 1) == ws["attn_scratch"]
    else:
        assert ws["attn_scratch"] == 0
    nb = (4 * M + 31) // 32
    assert ws["scatter_rows"] == 2 * nb * H * 4
    f = 4
    MH, lse = M * H * f, B * nh * Lq * f
    assert ws["saved"] == 2 * (6 * MH + lse + M * nh * nh * f) + 2 * (12 * MH + 2 * lse) + 2 * 3 * MH + MH + 2 * M * f


@pytest.mark.parametrize("H,nh", [(64, 2), (128, 2), (192, 4), (256, 4), (256, 8)])
@pytest.mark.parametrize("B,Lq", [(8, 50), (8, 200), (2, 512)])
def test_sizes_up_to_256_unchanged(H, nh, B, Lq):
    L, lib = _lib()
    ws = _ws(L, lib, B, Lq, H, nh)
    fwd, bwd = _tc_sizes(B, Lq, H, nh)
    assert ws["fwd_scratch"] == (fwd if H >= 128 else 0)
    assert ws["wgrad_scratch"] == (bwd if H >= 128 else 0)


def test_wide_shapes_pass_the_checks_into_argument_validation():
    """accepted wide shapes get past the shape checks: with no scratch the block entry points stop at the tcgen05 path's buffer check"""
    L, lib = _lib()
    for H, nh in ((384, 3), (384, 6), (512, 4), (512, 8)):
        for f in BLOCK_ENTRIES:
            b = L.fill(_struct(L, f)(), B=2, L=40, H=H, nh=nh, precision=1)
            with pytest.raises(L.AdtError, match="tcgen05 block path only"):
                L.check(getattr(lib, f)(ctypes.byref(b), None), f)
