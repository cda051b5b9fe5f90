"""The H = 64 backward row-tile kernels (pre_bwd, mid_bwd, post_bwd<enc|dec>: dgrad chain and weight gradients on separate warps)
against the generic bf16 row-tile kernels, at shapes the small-kernel cases of test_gpu_shapes.py leave out: one head (no
independence head) without dropout, four heads, and a batch with more CTAs than two per SM on 148 SMs."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# (B, L, nh, nl, dropout, sequence lengths), as test_gpu_shapes._SMALL_CASES
_CASES = [
    (5, 10, 1, 2, 0.0, [10, 9, 4, 2, 1]),                     # single head: no independence head; dropout off; 50 rows
    (4, 40, 4, 2, 0.3, [40, 39, 21, 1]),                      # four heads; 160 rows: partial last tile
    (400, 50, 2, 2, 0.5, [(50 - b) % 51 for b in range(400)]),  # 20000 rows = 313 CTAs (> 2 x 148), partial last tile, empty sequences
]
# elementwise tolerance, as a fraction of each tensor's max.  The two kernel sets round different intermediates to bf16, and over
# 20000 rows that difference reaches 2.1 % of the max of item_emb and of encoder layer 1's conv1 weight gradient (B200, both with
# the 128-thread backward kernels and with the two-role ones, which agree with each other to 5e-5 of every tensor's max).  A row
# tile that is skipped or misplaced moves a gradient by far more than that.
_TOL = [2e-2, 2e-2, 3e-2]


if __name__ == "__main__":      # helper process (the kernel switches are read once per process)
    from test_gpu_shapes import _bf16_step_grads
    res = _bf16_step_grads(_CASES[int(sys.argv[1])])["bf16"]
    np.savez(sys.argv[2], loss=res[0], gnorm=res[1], **{"g/" + k: v for k, v in res[2].items()})
    sys.exit(0)


@pytest.mark.parametrize("case", range(len(_CASES)))
def test_bf16_small_bwd_kernels_match_generic_bf16(case, tmp_path):
    """same check as test_gpu_shapes.test_bf16_small_kernels_match_generic_bf16: gradients agree elementwise to _TOL[case] of each
    tensor's max, loss to 1e-4, gradient norm to 5e-3."""
    here = os.path.abspath(__file__)
    files = []
    for tag, env in (("small", {}), ("generic", {"ADT_ROW_SMALL": "0", "ADT_ATTN_SMALL": "0"})):
        f = str(tmp_path / f"{tag}.npz")
        e = dict(os.environ, **env)
        e["PYTHONPATH"] = os.path.dirname(os.path.dirname(here)) + os.pathsep + os.path.dirname(here) + os.pathsep + e.get("PYTHONPATH", "")
        subprocess.run([sys.executable, here, str(case), f], check=True, env=e, timeout=600)
        files.append(np.load(f))
    a, b = files
    assert abs(float(a["loss"]) - float(b["loss"])) / abs(float(b["loss"])) < 1e-4
    assert abs(float(a["gnorm"]) - float(b["gnorm"])) / float(b["gnorm"]) < 5e-3
    for k in a.files:
        if not k.startswith("g/"):
            continue
        x, y = a[k], b[k]
        if np.abs(y).max() < 1e-9:
            continue
        assert np.abs(x - y).max() <= _TOL[case] * np.abs(y).max() + 1e-7, (k, float(np.abs(x - y).max()), float(np.abs(y).max()))
