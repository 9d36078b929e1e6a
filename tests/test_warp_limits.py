"""CPU: the C-ABI limits of the activation warp (dh_warp_gather_dense, dh_warp_gather_list) and of the dense source maps
(dh_dense_source_maps), and the argument checks of diffusionhandles_b200.warp.  Every call passes fake device pointers and
is one the library must reject before any CUDA call.  Levels that stay valid are fast-path levels, which launch nothing
until every level has been read, so no request here can reach a launch even if a check regressed."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

INVALID = -1
FAKE = 0x1000          # 16-byte aligned, never dereferenced


def _levels(N, n, channels=4, hw=64 * 64):
    arr = (N.dh_warp_level * max(n, 1))()
    for i, l in enumerate(arr):
        l.inp, l.out, l.src_map = FAKE + 0x300000 * i, FAKE + 0x300000 * i + 0x100000, FAKE + 0x300000 * i + 0x200000
        l.channels, l.hw = channels, hw
    return arr


def test_dense_warp_rejects_what_it_cannot_run():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    ok = _levels(N, 8)
    assert lib.dh_warp_gather_dense(ok, 0, 1, None) == INVALID            # no level
    assert lib.dh_warp_gather_dense(ok, -1, 1, None) == INVALID
    assert lib.dh_warp_gather_dense(_levels(N, 9), 9, 1, None) == INVALID # above the 8 levels of one launch
    assert lib.dh_warp_gather_dense(ok, 2, 0, None) == INVALID            # no edit
    assert lib.dh_warp_gather_dense(ok, 2, -3, None) == INVALID
    assert lib.dh_warp_gather_dense(None, 2, 1, None) == INVALID
    for pos in (0, 1, 7):                                                  # the first, a middle and the last level
        for field, val in (("inp", None), ("out", None), ("src_map", None), ("channels", 0), ("channels", -1), ("hw", 0),
                           ("hw", -4096), ("out", "inp")):
            arr = _levels(N, 8)
            setattr(arr[pos], field, getattr(arr[pos], val) if val == "inp" else val)
            assert lib.dh_warp_gather_dense(arr, 8, 2, None) == INVALID, (pos, field, val)


def test_list_warp_rejects_what_it_cannot_run():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    ok = dict(inp=FAKE, C=4, hw=960, idx=FAKE + 0x100000, n=100, out=FAKE + 0x200000)
    for bad in (dict(C=0), dict(C=-1), dict(hw=0), dict(hw=-1), dict(n=-1), dict(idx=None), dict(inp=None), dict(out=None)):
        a = {**ok, **bad}
        assert lib.dh_warp_gather_list(a["inp"], a["C"], a["hw"], a["idx"], a["n"], a["out"], None) == INVALID, bad


def test_dense_source_maps_rejects_what_it_cannot_run():
    from diffusionhandles_b200 import _native as N
    lib = N.load()

    def call(sides, img_res=96, stride=100, B=2, corr=FAKE, n_corr=FAKE + 0x100000, maps=FAKE + 0x200000, n_levels=None):
        arr = (N.c_int * max(len(sides), 1))(*sides)
        return lib.dh_dense_source_maps(corr, n_corr, stride, None, B, img_res, arr, len(sides) if n_levels is None else n_levels,
                                        maps, None)

    for sides in ([7], [96, 48, 7], [128], [96, 192], [0], [96, -1], [], [1] * 9):
        assert call(sides) == INVALID, sides
    assert call([96, 48], n_levels=0) == INVALID
    assert call([8] * 8, n_levels=9) == INVALID
    assert call([96], stride=0) == INVALID
    assert call([96], stride=-1) == INVALID
    assert call([96], B=0) == INVALID
    assert call([96], img_res=0) == INVALID
    for field in ("corr", "n_corr", "maps"):
        assert call([96], **{field: None}) == INVALID, field
    assert lib.dh_dense_source_maps(FAKE, FAKE, 100, None, 1, 96, None, 1, FAKE, None) == INVALID     # no side table


def test_python_warp_argument_checks():
    """Shape errors are found before any pointer is taken (so CPU tensors are enough here)."""
    from diffusionhandles_b200 import warp
    a = torch.zeros((2, 3, 8, 8))
    m = torch.zeros((2, 64), dtype=torch.int32)
    for levels, maps, out in (([a], [m, m], None),                                   # one map per level
                              ([a], [torch.zeros((2, 63), dtype=torch.int32)], None),
                              ([a], [torch.zeros((1, 64), dtype=torch.int32)], None),
                              ([a], [torch.zeros(128, dtype=torch.int32)], None),
                              ([a], [m], [torch.zeros((2, 3, 8, 7))]),                 # output shape
                              ([a], [m], [torch.zeros((2, 4, 8, 8))]),
                              ([torch.zeros((2, 3, 64))], [m], None)):                 # not (B,C,h,w)
        with pytest.raises(ValueError):
            warp.warp_stacks(levels, maps, out)
    corr, n = torch.zeros((1, 4, 4), dtype=torch.int64), torch.zeros(1, dtype=torch.int32)
    for sides in ([], [8] * 9):
        with pytest.raises(ValueError):
            warp.dense_source_maps(corr, n, 8, sides)
    with pytest.raises(ValueError):
        warp.gather_list(torch.zeros((3, 64)), [0], [0])
