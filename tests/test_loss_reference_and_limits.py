"""CPU: the fp64 loss oracle (oracle.dh_oracle.foreground_loss / background_loss) pinned against torch fp64 autograd of the
reference's losses.py formulas, at the edges the K4 kernels are tested at (repeated cells in every list, grids other than 64,
maps whose area is not a multiple of 4, patch sizes up to 31, empty lists); and the loss-plan limits of the C ABI, which are
checked before anything touches the GPU."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import dh_oracle as O

f64 = torch.float64


def _t_local(f1, f2, x1, y1, x2, y2, patch):
    """losses.py local_average_feat_l1_loss."""
    H, W = f1.shape[-2:]
    w1 = torch.zeros(1, H, W, dtype=f64)
    w2 = torch.zeros(1, H, W, dtype=f64)
    w1[:, y1, x1] = 1
    w2[:, y2, x2] = 1
    pool = torch.nn.AvgPool2d(patch, stride=1, padding=patch // 2)
    a1 = pool(f1 * w1) / (pool(w1) + 1e-10)
    a2 = pool(f2 * w2) / (pool(w2) + 1e-10)
    return (a1[:, y1, x1] - a2[:, y2, x2]).abs().mean(dim=-1).mean()


def _t_loss(cur, orig, pc, size, term, patch):
    """losses.py compute_foreground_loss / compute_background_loss in fp64; returns (value, d value / d cur)."""
    c = torch.from_numpy(cur).to(f64).requires_grad_(True)
    uc = F.interpolate(c[None], size=size, mode="bilinear")[0]
    uo = F.interpolate(torch.from_numpy(orig).to(f64)[None], size=size, mode="bilinear")[0]
    if term == "fg":
        v = _t_local(uo, uc, pc["original_x"], pc["original_y"], pc["transformed_x"], pc["transformed_y"], patch)
    elif term == "local_avg":
        v = _t_local(uo, uc, pc["background_x"], pc["background_y"], pc["background_x"], pc["background_y"], patch)
    else:
        v = (uo[..., pc["background_y_orig"], pc["background_x_orig"]].mean(dim=-1)
             - uc[..., pc["background_y_trans"], pc["background_x_trans"]].mean(dim=-1)).abs().mean()
    (g,) = torch.autograd.grad(v, c, allow_unused=True)
    return v.item(), (torch.zeros_like(c) if g is None else g).numpy()


def _o_loss(cur, orig, pc, size, term, patch):
    if term == "fg":
        return O.foreground_loss(cur, orig, pc, size=size, patch=patch)
    return O.background_loss(cur, orig, pc, size=size, loss_type=term, patch=patch)


def _lists(rng, grid, n_fg, n_bg):
    """Index lists drawn WITH replacement (every list repeats cells), plus one cell repeated many times in each list."""
    def draw(n, hot):
        y, x = rng.integers(0, grid, n), rng.integers(0, grid, n)
        return np.concatenate([y, np.full(37, hot[0])]), np.concatenate([x, np.full(37, hot[1])])
    hot = (grid // 3, grid - 1)
    pc = {}
    pc["original_y"], pc["original_x"] = draw(n_fg, hot)
    pc["transformed_y"], pc["transformed_x"] = draw(n_fg, (grid - 1, 0))
    pc["background_y"], pc["background_x"] = draw(n_bg, hot)
    pc["background_y_orig"], pc["background_x_orig"] = draw(n_bg, (0, grid // 2))
    pc["background_y_trans"], pc["background_x_trans"] = draw(n_bg, hot)
    return pc


# (grid, native map h x w, patch).  Resized maps use sizes whose bilinear scale n / grid is a dyadic fraction, so the
# oracle's fp32 taps and torch's fp64 taps are the same numbers and the two fp64 computations agree to rounding.
CASES = [
    (64, (64, 64), 1), (64, (9, 9), 1), (64, (25, 25), 2), (64, (32, 48), 3), (64, (13, 13), 31), (64, (16, 16), 5),
    (32, (32, 32), 1), (32, (13, 13), 3), (32, (31, 31), 31), (32, (8, 16), 2),
    (48, (48, 48), 1), (48, (24, 24), 3), (48, (48, 48), 2),
    (63, (63, 63), 1), (63, (63, 63), 3), (63, (63, 63), 31),
]


@pytest.mark.parametrize("grid,hw,patch", CASES)
def test_oracle_losses_match_torch_fp64_autograd(grid, hw, patch):
    rng = np.random.default_rng(grid * 1000 + hw[0] * 37 + hw[1] + patch)
    C = 3
    cur = rng.normal(size=(C,) + hw)
    orig = rng.normal(size=(C,) + hw)
    pc = _lists(rng, grid, n_fg=int(rng.integers(50, 3000)), n_bg=int(rng.integers(50, 3000)))
    for term in ("fg", "local_avg", "global_avg"):
        p = 1 if term == "global_avg" else patch
        ref_v, ref_g = _t_loss(cur, orig, pc, (grid, grid), term, p)
        v, g = _o_loss(cur, orig, pc, (grid, grid), term, p)
        assert abs(v - ref_v) <= 1e-12 * abs(ref_v), (term, v, ref_v)
        assert g.shape == ref_g.shape
        assert np.abs(g - ref_g).max() <= 1e-12 * np.abs(ref_g).max(), (term, np.abs(g - ref_g).max(), np.abs(ref_g).max())


def test_oracle_global_avg_gradient_accumulates_repeated_cells():
    """A cell listed three times in bg_trans receives three gradient quanta (autograd of the indexing accumulates)."""
    C = 1
    cur = np.zeros((C, 64, 64))
    orig = np.ones((C, 64, 64))
    pc = {"background_y_orig": np.array([1]), "background_x_orig": np.array([1]),
          "background_y_trans": np.array([5, 5, 5, 9]), "background_x_trans": np.array([7, 7, 7, 2])}
    v, g = O.background_loss(cur, orig, pc, loss_type="global_avg")
    ref_v, ref_g = _t_loss(cur, orig, pc, (64, 64), "global_avg", 1)
    assert v == ref_v == 1.0
    assert g[0, 5, 7] == ref_g[0, 5, 7] == -0.75 and g[0, 9, 2] == ref_g[0, 9, 2] == -0.25
    assert np.array_equal(g, ref_g)


@pytest.mark.parametrize("empty", ["fg", "bg", "bg_orig", "bg_trans", "all"])
def test_oracle_losses_with_empty_lists_match_torch(empty):
    """An empty list gives a NaN loss like torch's mean over nothing; the gradient is what autograd makes of it."""
    rng = np.random.default_rng(5)
    cur, orig = rng.normal(size=(2, 32, 32)), rng.normal(size=(2, 32, 32))
    pc = _lists(rng, 64, 200, 200)
    none = np.zeros(0, np.int64)
    keys = {"fg": ["original", "transformed"], "bg": ["background"], "bg_orig": ["background_orig"],
            "bg_trans": ["background_trans"]}
    for k in (sum(keys.values(), []) if empty == "all" else keys[empty]):
        base, _, suffix = k.partition("_")
        for ax in ("y", "x"):
            pc[f"{base}_{ax}" + (f"_{suffix}" if suffix else "")] = none
    for term in ("fg", "local_avg", "global_avg"):
        for patch in ((1,) if term == "global_avg" else (1, 3)):
            ref_v, ref_g = _t_loss(cur, orig, pc, (64, 64), term, patch)
            v, g = _o_loss(cur, orig, pc, (64, 64), term, patch)
            if np.isnan(ref_v):
                assert np.isnan(v), (term, v)
            else:
                assert abs(v - ref_v) <= 1e-12 * abs(ref_v), (term, v, ref_v)
            assert np.array_equal(np.isnan(g), np.isnan(ref_g)), term
            fin = ~np.isnan(ref_g)
            assert np.abs(g[fin] - ref_g[fin]).max(initial=0.0) <= 1e-12 * np.abs(ref_g[fin]).max(initial=0.0), term


# ---- C ABI limits of the loss plan (no GPU work: the checks run before any launch) ----

def _build(lib, n_fg, n_bo=0, n_bt=0, n_bc=0, grid=64):
    """dh_build_loss_plan with fake pointers and a 16-byte plan buffer: a request the limit checks accept stops at the size
    check (DH_ERR_WORKSPACE), so no call here can reach a launch even if a limit check regressed."""
    fake = ctypes.c_void_p(0x1000)
    plan_bytes = ws_bytes = 16
    return lib.dh_build_loss_plan(fake, fake, n_fg, fake, n_bo, fake, n_bt, fake, n_bc, grid, fake, plan_bytes, fake, ws_bytes, None)


def test_plan_builder_rejects_lists_that_overflow_16_bit_plan_fields():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    UNSUPPORTED, WORKSPACE = -2, -4
    # per-cell background counts are 16-bit
    for kw in (dict(n_bo=65536), dict(n_bt=65536), dict(n_bc=65536), dict(n_bo=1 << 20, n_bt=1 << 20)):
        assert _build(lib, 10, **kw) == UNSUPPORTED, kw
    # the row length in row_desc is 16-bit: a row holds at most min(n_fg, cells + n_fg / 255) entries
    for grid in (1, 8, 64):
        n_max = (65535 - grid * grid) * 255 + 254        # largest n_fg with cells + n_fg // 255 <= 65535
        assert _build(lib, n_max + 1, grid=grid) == UNSUPPORTED, grid
        # the largest accepted n_fg passes this check and stops at the (deliberately tiny) plan buffer instead
        assert _build(lib, n_max, grid=grid) == WORKSPACE, grid
    assert _build(lib, 15_667_199, grid=64) == WORKSPACE          # ~15.6 M correspondences still fit at 64 x 64
    # lists of the limit length are accepted (again stopping at the plan buffer)
    assert _build(lib, 10, n_bo=65535, n_bt=65535, n_bc=65535) == WORKSPACE


def test_plan_info_refuses_a_plan_flagged_unusable():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    hdr = np.zeros(16, np.int32)
    hdr[0], hdr[5] = 7, 64               # n_pairs, grid
    desc = N.dh_loss_plan_desc()
    for flags, rc in ((0, 0), (1, 0), (2, -2), (3, -2)):
        hdr[7] = flags                   # PlanHeader.reserved: bit 0 binary background lists, bit 1 ELL table did not fit
        assert lib.dh_loss_plan_info(hdr.tobytes(), ctypes.byref(desc)) == rc, flags
        if rc == 0:
            assert desc.n_pairs == 7 and desc.flags == (flags & 1)

