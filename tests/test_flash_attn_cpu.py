"""Host-side contract of sequences longer than 256 positions: scratch sizes of the fused flash attention are O(B L H) with no L^2
term (and unchanged for L <= 256), and every shape no path serves is refused with an error that names the limit."""
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


@pytest.mark.parametrize("H,nh", [(64, 2), (256, 2), (256, 4)])
def test_flash_scratch_is_linear_in_sequence_length(H, nh):
    L, lib = _lib()
    B = 4
    for Lq in (512, 1024, 2048):
        M = B * Lq
        fwd = lib.adt_attention_scratch_bytes(B, Lq, H, nh, 0)
        bwd = lib.adt_attention_scratch_bytes(B, Lq, H, nh, 1)
        assert fwd == 256 + M * 3 * H * 2                                  # bf16 [q | k | v]
        assert bwd == 256 + M * 3 * H * 2 + M * H * 2 + M * nh * 4         # + bf16 dctx + delta
        ws = _ws(L, lib, B, Lq, H, nh)
        assert ws["attn_scratch"] == bwd
        if H >= 128:   # the tcgen05 block path's operand areas carry no [B nh L L] score term beyond 256 positions
            hh = H * H * 2
            assert ws["wgrad_scratch"] == 12 * M * H * 2 + 10 * hh + 1024 + 4 * M * H * 2
            assert ws["fwd_scratch"] == 9 * M * H * 2 + 10 * hh + 1024 + 3 * M * H * 2


def test_short_sequences_keep_their_sizes():
    L, lib = _lib()
    for Lq in (50, 200, 256):
        ws = _ws(L, lib, 8, Lq, 256, 4)
        assert ws["attn_scratch"] == 0
        Lp, M = (Lq + 7) // 8 * 8, 8 * Lq
        zll = M * 4 * Lp
        assert ws["fwd_scratch"] == 9 * M * 256 * 2 + 10 * 256 * 256 * 2 + 1024 + 3 * M * 256 * 2 + zll * 6
        tc = lib.adt_attention_scratch_bytes(8, Lq, 256, 4, 1)
        assert tc == (1024 + 4 * M * 256 * 2 + zll * 12 if Lq > 64 else 0)


def _attn_args(L, Lq, H, nh, precision):
    return L.fill(L.adt_attention_args(), B=2, L=Lq, H=H, nh=nh, mask_mode=0, training=0, precision=precision)


@pytest.mark.parametrize("Lq,H,nh,precision,msg", [
    (512, 64, 2, 0, "precision 1"),          # fp32 cores stop at 256 positions
    (512, 48, 2, 1, "multiple of 16"),       # hd 24
    (512, 256, 1, 1, "at most 128"),         # hd 256
    (2049, 64, 2, 1, "2048"),
])
def test_refusals_name_the_limit(Lq, H, nh, precision, msg):
    L, lib = _lib()
    a = _attn_args(L, Lq, H, nh, precision)
    for f in ("adt_attention_fwd", "adt_attention_bwd", "adt_attention_flash_fwd"):
        with pytest.raises(L.AdtError, match=msg):
            L.check(getattr(lib, f)(ctypes.byref(a), None), f)
    for f, st in (("adt_enc_block_fwd", L.adt_enc_block_fwd_args), ("adt_dec_block_bwd", L.adt_dec_block_bwd_args)):
        b = L.fill(st(), B=2, L=Lq, H=H, nh=nh, precision=precision)
        with pytest.raises(L.AdtError, match=msg):
            L.check(getattr(lib, f)(ctypes.byref(b), None), f)
    if precision:     # the workspace query has no precision: it refuses the head sizes and lengths no bf16 path serves
        with pytest.raises(L.AdtError, match=msg):
            _ws(L, lib, 2, Lq, H, nh)
