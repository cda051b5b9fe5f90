"""The SASRec-ADT encoder and decoder blocks, forward and backward, through the block C ABI on every default route, against fp64.

Each case runs both blocks once (block_harness.run) and compares every saved activation, out, rec, lse, dx, dctx, dfeats, denc, every
parameter gradient, nll_acc and mse_acc with block_ref's fp64 restatement on the same inputs: in the bf16 mode with the BF16 product
hook (every product operand rounded to bf16, as the kernels feed their MMAs), in the fp32 mode with the plain one.  The error is
max |got - ref| / max |ref| per tensor, with a cosine floor; the bounds are about twice the worst value measured on a B200 (DESIGN.md
section 5).  In the bf16 mode the kernels must also be at least 4x closer to the BF16 reference than to the plain fp64 one on out
and dx: otherwise the rounding plan of block_ref.py misses a point where the kernels round.  The kernel names each call launches
pin the route, so a later dispatch change cannot move a case to another route unnoticed."""
import numpy as np
import pytest
import torch

import block_harness as BH
import block_ref as R

pytestmark = pytest.mark.gpu

# the kernels each call launches, exactly (route pinning: a dispatch change that moves a case shows up as a different set)
_SMALL = {"enc_fwd": {"pre_fwd", "attn_fwd", "enc_post_fwd"}, "enc_bwd": {"enc_post_bwd", "attn_bwd", "pre_bwd"},
          "dec_fwd": {"pre_fwd", "attn_fwd", "mid_fwd", "dec_post_fwd"}, "dec_bwd": {"dec_post_bwd", "attn_bwd", "mid_bwd", "pre_bwd"}}
_FUSED = {"enc_fwd": {"pre_attn_fwd", "enc_post_fwd"}, "enc_bwd": {"enc_post_bwd", "attn_pre_bwd"},
          "dec_fwd": {"pre_attn_fwd", "mid_attn_fwd", "dec_post_fwd"}, "dec_bwd": {"dec_post_bwd", "attn_bwd", "mid_bwd", "attn_pre_bwd"}}
_FUSED_FWD = dict(_FUSED, enc_bwd=_SMALL["enc_bwd"], dec_bwd=_SMALL["dec_bwd"])              # one head: the backward runs separately
_SMALL_FLASH = {k: (v - {"attn_fwd", "attn_bwd"}) | {"row_tc", "attn_flash_" + k[4:]} for k, v in _SMALL.items()}
_HOIST = dict(_SMALL, enc_bwd=_SMALL["enc_bwd"] | {"wgrad_tc"}, dec_bwd=_SMALL["dec_bwd"] | {"wgrad_tc"})
_TC = {"enc_fwd": {"linear_tc", "row_tc"}, "enc_bwd": {"dgrad_tc", "row_tc", "wgrad_tc"}, "dec_fwd": {"linear_tc", "row_tc"},
       "dec_bwd": {"dgrad_tc", "row_tc", "wgrad_tc"}}
_TC_ROWTILE_ATTN = {k: v | {"attn_" + k[4:]} for k, v in _TC.items()}                      # attn_fwd / attn_bwd
_TC_BATCHED = {k: v | {"attn_gemm_tc", "attn_row_tc"} for k, v in _TC.items()}
_TC_FLASH = {k: v | {"attn_flash_" + k[4:]} for k, v in _TC.items()}

# route -> (case, kernels each call launches)
ROUTES = {
    "h64_small": (BH.Case(6, 20, 64, 2, [0, 3, 20, 19, 7, 1]), _SMALL),
    "h64_fused_c2": (BH.Case(7, 50, 64, 2, [0, 1, 20, 49, 50, 3, 0], b0=3, sdev=4), _FUSED),
    "h64_fused_l64_mask1": (BH.Case(5, 64, 64, 4, [0, 63, 10, 64, 0], mask_mode=1), _FUSED),
    "h64_fused_nh1_p0": (BH.Case(3, 33, 64, 1, [0, 33, 7], p=0.0), _FUSED_FWD),
    "h64_generic_attn": (BH.Case(3, 200, 64, 2, [0, 150, 200]), _SMALL),
    "h64_flash": (BH.Case(2, 300, 64, 2, [300, 17]), _SMALL_FLASH),
    "rowtile_h32": (BH.Case(5, 40, 32, 2, [0, 40, 3, 39, 11]), _SMALL),
    "rowtile_h96": (BH.Case(4, 70, 96, 2, [70, 0, 5, 60]), _SMALL),
    "rowtile_hoist_h128": (BH.Case(8, 40, 128, 2, [0, 40, 1, 2, 3, 30, 39, 0]), _HOIST),
    "tc_h192": (BH.Case(9, 60, 192, 3, [0, 60, 5, 59, 1, 0, 30, 2, 7]), _TC_ROWTILE_ATTN),
    "tc_h256_batched": (BH.Case(3, 200, 256, 2, [0, 200, 37]), _TC_BATCHED),
    "tc_h256_flash": (BH.Case(2, 300, 256, 4, [300, 9]), _TC_FLASH),
    "wide_h320": (BH.Case(3, 40, 320, 5, [0, 40, 13]), _TC_ROWTILE_ATTN),
    "wide_h384_hd128": (BH.Case(4, 130, 384, 3, [0, 130, 64, 1]), _TC_BATCHED),
    "wide_h448": (BH.Case(2, 33, 448, 7, [33, 4]), _TC_ROWTILE_ATTN),
    "wide_h512_l512": (BH.Case(1, 512, 512, 8, [100]), _TC_FLASH),
    "wide_h512_mask1": (BH.Case(3, 200, 512, 4, [0, 200, 77], mask_mode=1), _TC_BATCHED),
    # fp32 mode (precision 0) against the plain fp64 reference
    "fp32_c2": (BH.Case(7, 50, 64, 2, [0, 1, 20, 49, 50, 3, 0], b0=3, sdev=4, precision=0), _SMALL),
    "fp32_h96": (BH.Case(4, 70, 96, 2, [70, 0, 5, 60], precision=0), _SMALL),
    "fp32_h128": (BH.Case(8, 40, 128, 2, [0, 40, 1, 2, 3, 30, 39, 0], precision=0), _SMALL),
    "fp32_h256_l200": (BH.Case(3, 200, 256, 2, [0, 200, 37], precision=0), _SMALL),
}
# bound on max |got - ref| / max |ref| per route (about 2x the worst tensor measured on the route); the cosine floor is 1 - bound^2 / 4
BOUNDS = {"h64_small": 7e-3, "h64_fused_c2": 5e-3, "h64_fused_l64_mask1": 7e-3, "h64_fused_nh1_p0": 4e-3, "h64_generic_attn": 5e-3,
          "h64_flash": 2e-2, "rowtile_h32": 3e-4, "rowtile_h96": 6e-3, "rowtile_hoist_h128": 5e-3, "tc_h192": 4e-3, "tc_h256_batched": 7e-3,
          "tc_h256_flash": 2e-2, "wide_h320": 1e-2, "wide_h384_hd128": 8e-3, "wide_h448": 2e-2, "wide_h512_l512": 2e-2,
          "wide_h512_mask1": 2e-2, "fp32_c2": 2e-6, "fp32_h96": 5e-6, "fp32_h128": 2e-6, "fp32_h256_l200": 3e-6}
# routes on which the kernels are at least RATIO times closer to the BF16 reference than to plain fp64 on out and dx (measured 4.1 to
# 1e4).  On the others the ratio is 1.2 - 3.8 at errors of one bf16 ulp or less: see DESIGN.md section 5
RATIO, RATIO_ROUTES = 4.0, ("h64_fused_c2", "h64_fused_nh1_p0", "h64_generic_attn", "rowtile_h32", "rowtile_h96")


def measure(route, run_kw=None):
    """run one route and compare it with the references -> (metrics {name: (err, cos, err_plain)}, kernel names, kernel results)"""
    c, _ = ROUTES[route]
    inp = BH.inputs(c)
    got = BH.run(c, inp, **(run_kw or {}))
    bf16 = c.precision == 1
    met = {}
    for blk, fn in (("enc", R.enc_block), ("dec", R.dec_block)):
        h1 = got[f"{blk}/h1"]
        ref = fn(inp[blk], bf16, kernel_h1=h1)
        plain = fn(inp[blk], False, kernel_h1=h1) if bf16 else ref
        for k, v in ref.items():
            g = torch.from_numpy(np.asarray(got[f"{blk}/{k}"], dtype=np.float64))
            e, cs = R.err(g, v)
            met[f"{blk}/{k}"] = (e, cs, R.err(g, plain[k])[0], float(v.abs().max()), bool(torch.isfinite(g).all()))
    return met, {k[6:]: v for k, v in got.items() if k.startswith("names/")}, got


def _report(route, met):
    for k, (e, cs, ep, mx, fin) in sorted(met.items()):
        print(f"{route:22s} {k:14s} err {e:.3e} cos {cs:.9f} plain {ep:.3e} ratio {ep / max(e, 1e-300):8.1f} max {mx:.3e} finite {fin}")


@pytest.mark.parametrize("route", list(ROUTES))
def test_block_against_fp64(route):
    c, want = ROUTES[route]
    met, names, _ = measure(route)
    _report(route, met)
    for call, need in want.items():
        assert set(names[call]) == need, (call, sorted(names[call]), sorted(need))
    bound = BOUNDS[route]
    for k, (e, cs, ep, mx, fin) in met.items():
        assert fin, (k, "non-finite values: a row was left unwritten")
        if mx == 0.0:           # a single head: rec and nll_acc are identically zero
            assert e == 0.0 or e <= 1e-6, (k, e)
            continue
        assert e <= bound and cs >= 1.0 - bound * bound / 4, (k, e, cs, bound)
    if route in RATIO_ROUTES:
        for k in ("enc/out", "enc/dx", "dec/out", "dec/dx"):
            e, _, ep, _, _ = met[k]
            assert ep >= RATIO * e, (k, "kernel not closer to the bf16-hook reference than to plain fp64", e, ep)


def _rows_equal(a, b, keys):
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=False), (k, float(np.nanmax(np.abs(a[k] - b[k]))))


def _grads_close(a, b):
    """weight gradients and the fp64 loss sums: equal up to the order of their atomic additions"""
    for k in a:
        if "/g_" in k or k.endswith("_acc"):
            x, y = a[k], b[k]
            assert np.abs(x - y).max() <= 1e-5 * np.abs(y).max() + 1e-12, (k, float(np.abs(x - y).max()))


_DEC_ROWS = ("dec/d", "dec/q1", "dec/k1", "dec/v1", "dec/ctx1", "dec/lse1", "dec/a", "dec/q2", "dec/k2", "dec/v2", "dec/ctx2", "dec/lse2",
             "dec/c", "dec/h1", "dec/out", "dec/dx", "dec/dfeats", "dec/dctx", "dec/dctx2", "dec/denc")


@pytest.mark.parametrize("route", ["h64_fused_c2", "tc_h256_batched", "wide_h512_l512"])
def test_decoder_phase_split(route):
    """decoder forward phase 1 + 2 == phase 0 and backward phase 2 + 1 == phase 0, as the training step's two streams run them: row
    outputs bit for bit, weight gradients up to the order of their atomic sums"""
    c, _ = ROUTES[route]
    inp = BH.inputs(c)
    whole = BH.run(c, inp)
    split = BH.run(c, inp, phases=(0, 12, 21))
    _rows_equal(split, whole, _DEC_ROWS)
    _grads_close(split, whole)


_ENC_ROWS = ("enc/q", "enc/k", "enc/v", "enc/ctx", "enc/lse", "enc/y", "enc/h1", "enc/out", "enc/rec", "enc/dx", "enc/dctx")


@pytest.mark.parametrize("route", ["h64_fused_c2", "rowtile_hoist_h128", "tc_h256_batched", "wide_h384_hd128"])
def test_weight_mirror_same_bits(route):
    """calls given an adt_wmirror holding the RN-bf16 weights compute what calls that convert the fp32 weights themselves compute"""
    c, _ = ROUTES[route]
    inp = BH.inputs(c)
    a = BH.run(c, inp, wm=True)
    b = BH.run(c, inp)
    _rows_equal(a, b, _ENC_ROWS + _DEC_ROWS)
    _grads_close(a, b)
