"""CPU tests of the fused vocabulary head's host planner (adt_linear_ce_plan): the vocabulary chunks tile [0, V) exactly, each chunk's
scratch fits what the caller declared, and too small a scratch is refused with ADT_E_SHAPE."""
import pytest

from adt_b200 import _lib as L
from adt_b200 import ops


def _layout_bytes(R, vc):
    """the planner's scratch layout for a chunk of vc columns (rounded up to 128): bf16 dS [R, vc], per-tile (max, sum exp) partials
    [vc / 128, R] float2, the running per-row state (float2) and z at the label (float), each area 256-byte aligned."""
    a = lambda b: (b + 255) // 256 * 256
    vc = (vc + 127) // 128 * 128
    return a(2 * R * vc) + a(8 * R * (vc // 128)) + a(8 * R) + a(4 * R)


@pytest.mark.parametrize("R,V,H", [(1, 1600, 64), (129, 26844, 128), (4099, 70001, 256), (10240, 1000100, 256), (7, 128, 64), (300, 129, 64)])
@pytest.mark.parametrize("frac", [0.0, 0.013, 0.3, 1.0, 4.0])
def test_plan_chunks_tile_the_vocabulary_within_the_scratch(R, V, H, frac):
    _, mn = ops.linear_ce_plan(R, V, H, 1 << 62)
    assert mn == _layout_bytes(R, 128)
    full = ops.linear_ce_scratch_bytes(R, V, H, budget=1 << 62)
    nbytes = int(mn + frac * (full - mn))
    vc, mn2 = ops.linear_ce_plan(R, V, H, nbytes)
    assert mn2 == mn
    assert 1 <= vc <= V
    assert vc == V or vc % 128 == 0                       # chunk starts stay 128-column (and 16-byte) aligned
    assert _layout_bytes(R, vc) <= nbytes                 # the chunk respects the declared scratch
    assert vc == V or _layout_bytes(R, vc + 128) > nbytes  # and is the widest that does
    edges = list(range(0, V, vc)) + [V]
    cover = [c for a, b in zip(edges, edges[1:]) for c in (a, b)]
    assert cover[0] == 0 and cover[-1] == V and all(cover[i] == cover[i + 1] for i in range(1, len(cover) - 1, 2))
    assert sum(b - a for a, b in zip(edges, edges[1:])) == V
    if frac >= 1.0:
        assert vc == V                                    # linear_ce_scratch_bytes' full size covers V in one chunk


def test_plan_refuses_too_small_a_scratch():
    R, V, H = 4099, 70001, 256
    _, mn = ops.linear_ce_plan(R, V, H, 1 << 62)
    with pytest.raises(L.AdtError, match="scratch"):
        ops.linear_ce_plan(R, V, H, mn - 1)
    vc, mn2 = ctypes_plan(R, V, H, mn - 1)
    assert vc == 0 and mn2 == mn
    assert ctypes_plan(R, V, H, mn)[0] == 128


def test_plan_refuses_bad_shapes():
    for R, V, H in [(0, 100, 64), (10, 0, 64), (10, 100, 0), (-1, 100, 64)]:
        with pytest.raises(L.AdtError, match="positive"):
            ops.linear_ce_plan(R, V, H, 1 << 30)


def test_scratch_budget_bounds_memory_at_one_million_items():
    """at R 10,240, V 1,000,100 the default budget keeps the head's scratch to a few hundred MB: O(R Vc), not the 41 GB of one fp32
    [R, V] tensor"""
    R, V, H = 10240, 1000100, 256
    nbytes = ops.linear_ce_scratch_bytes(R, V, H)
    vc, _ = ops.linear_ce_plan(R, V, H, nbytes)
    assert nbytes <= ops.LINEAR_CE_SCRATCH and 128 <= vc < V
    assert nbytes < 0.01 * R * V * 4


def ctypes_plan(R, V, H, nbytes):
    import ctypes
    vc, mn = ctypes.c_int32(-1), ctypes.c_int64(-1)
    rc = L.lib().adt_linear_ce_plan(ctypes.c_int32(R), ctypes.c_int32(V), ctypes.c_int32(H), ctypes.c_int64(nbytes), ctypes.byref(vc), ctypes.byref(mn))
    assert rc == (0 if vc.value > 0 else -1)
    return vc.value, mn.value
