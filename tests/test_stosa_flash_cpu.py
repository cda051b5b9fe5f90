"""Host-side contract of STOSA-ADT's Wasserstein attention beyond the resident kernels' shared memory: the flash kernels' scratch is
O(B L H) with no L^2 term, adt_wattention_resident_fits states the resident limits, and every shape the flash kernels do not serve is
refused with an error that names the limit (before anything touches a GPU)."""
import ctypes

import pytest


def _lib():
    from adt_b200 import _lib as L
    try:
        lib = L.lib()
    except L.AdtError:
        pytest.skip("libadt_b200.so not built")
    lib.adt_wattention_scratch_bytes.restype = ctypes.c_int64
    return L, lib


@pytest.mark.parametrize("H,nh", [(64, 1), (64, 4), (128, 2)])
def test_wflash_scratch_is_linear_in_sequence_length(H, nh):
    L, lib = _lib()
    B = 8
    for bwd in (0, 1):
        n = [lib.adt_wattention_scratch_bytes(B, Lq, H, nh, bwd) for Lq in (256, 512, 1024, 2048)]
        per_row = 12 * H + 8 * nh + (4 * H + 12 * nh if bwd else 0)      # bf16 packs, fp32 norms (+ bf16 dctx pair, delta, vm, vc)
        for Lq, v in zip((256, 512, 1024, 2048), n):
            assert v == B * Lq * per_row + 8 * B * H + 4 * B              # + value means, first valid key
    assert lib.adt_wattention_scratch_bytes(B, 4096, H, nh, 0) == -1


# the longest sequence each head size accepts in the resident kernels' 220 KB of shared memory (forward, backward)
RESIDENT_LIMITS = {16: (484, 208), 32: (304, 132), 64: (168, 72)}


@pytest.mark.parametrize("hd", sorted(RESIDENT_LIMITS))
def test_resident_fits_matches_the_limits(hd):
    L, lib = _lib()
    for bwd, lim in enumerate(RESIDENT_LIMITS[hd]):
        for H, nh in ((hd, 1), (2 * hd, 2)):
            assert lib.adt_wattention_resident_fits(lim, H, nh, bwd) == 1
            assert lib.adt_wattention_resident_fits(lim + 1, H, nh, bwd) == 0
    assert lib.adt_wattention_resident_fits(200, 128, 4, 0) == 1       # (L 200, hd 32): the forward fits, the backward does not
    assert lib.adt_wattention_resident_fits(200, 128, 4, 1) == 0
    assert lib.adt_wattention_resident_fits(100, 64, 3, 0) < 0         # H % nh != 0


def _refusal(Lb, lib, fwd=True, **kw):
    dims = dict(B=2, L=512, H=64, nh=2)
    dims.update({k: v for k, v in kw.items() if k in dims})
    a = Lb.fill(Lb.adt_wattention_args(), **dims)
    for k, v in kw.items():
        if k not in dims:
            setattr(a, k, v)
    f = lib.adt_wattention_flash_fwd if fwd else lib.adt_wattention_flash_bwd
    rc = f(ctypes.byref(a), None)
    return rc, lib.adt_last_error().decode()


def test_wflash_refusals_name_the_limit():
    Lb, lib = _lib()
    ok = dict(tc_scratch=16, key_ids=16, lse=16)      # non-NULL placeholders: every case below is refused before any launch
    cases = [
        (dict(H=48, nh=2, **ok), "multiple of 16"),                       # hd 24
        (dict(H=40, nh=1, **ok), "multiple of 16"),
        (dict(H=128, nh=1, **ok), "at most 64"),                          # hd 128
        (dict(L=2049, **ok), "L > 2048"),
        (dict(key_ids=16, lse=16), "tc_scratch is NULL"),
        (dict(H=64, nh=3, **ok), "dims"),
    ]
    for kw, msg in cases:
        rc, err = _refusal(Lb, lib, **kw)
        assert rc == -1 and msg in err, (kw, rc, err)
    rc, err = _refusal(Lb, lib, fwd=False, **ok)                           # the backward needs the forward's outputs
    assert rc == -1 and "mctx_in" in err, err
