"""K4 at its limits: the loss plan (dh_build_loss_plan) decoded and compared field by field with a host model of the builder,
inside a canary-guarded buffer; every instantiation of the fused patch-1 kernel and the general patch kernel driven by an
input that selects it and compared with the fp64 oracle; the developer knobs that change the launch (shared-memory placement,
groups per CTA) giving bit-identical results; and the edges of the Python API (8 layers, NULL gradients, zero weights, one
channel, cached runners)."""
import ctypes
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.dirname(os.path.abspath(__file__))):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from oracle import dh_oracle as O          # noqa: E402

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


# ------------------------------------------------------------------------------------------------
# host model of dh_build_loss_plan (dh_loss.cu) and a copy of plan_layout (dh_loss_plan.cuh)
# ------------------------------------------------------------------------------------------------
def plan_layout(grid, cap):
    cells = grid * grid
    slices = (cells + 31) // 32
    n = cap if cap > 0 else 1
    r16 = lambda b: (b + 15) // 16 * 16              # noqa: E731
    ent_cap = n + 32 * (min(n, cells) + n // 255 + 1) + 96 * slices
    L, o = {}, 64
    for name, size in (("row", r16((cells + 1) * 4)), ("bg", cells * 8), ("pairs", r16(n * 8)), ("ell_off", r16((slices + 1) * 4)),
                       ("row_desc", slices * 32 * 4), ("ent", r16(ent_cap * 4)), ("usrc_cell", r16(cells * 2)), ("own_masks", 256 * 8)):
        L[name] = o
        o += size
    L["total"], L["ent_cap"] = o, ent_cap
    return L


def _row_entries(srcs):
    """The distinct sources of one destination cell with their multiplicities, in the builder's emission order: sources
    ascending in chunks of 32 consecutive cell ids (starting at the smallest source); a multiplicity above 255 is split into
    entries of 255 and a remainder, emitted round by round within the chunk."""
    u, c = np.unique(srcs, return_counts=True)
    if c.max() <= 255:
        return list(zip(u.tolist(), c.tolist()))
    out = []
    chunk = (u - u[0]) // 32
    for ch in np.unique(chunk):
        us, cs = u[chunk == ch], c[chunk == ch].copy()
        while (cs > 0).any():
            live = cs > 0
            m = np.minimum(cs, 255)
            out += list(zip(us[live].tolist(), m[live].tolist()))
            cs -= np.where(live, m, 0)
    return out


def ell_order(ucount, exact=True):
    """Rows (destination cells with pairs) in ELL order: descending length, ties in raster order.  exact=False is the order
    of the length classes min(len, 255) alone."""
    rows = np.flatnonzero(ucount)
    key = ucount[rows] if exact else np.minimum(ucount[rows], 255)
    return rows[np.lexsort((rows, -key))]


def ell_groups(ucount, order):
    pad = (ucount[order] + 3) & ~3
    return int(sum(pad[s:s + 32].max() for s in range(0, len(order), 32)))


def model_plan(src, dst, bo, bt, bc, grid):
    cells = grid * grid
    src, dst = np.asarray(src, np.int64), np.asarray(dst, np.int64)
    n_fg = len(src)
    rows = {}
    if n_fg:
        o = np.lexsort((src, dst))
        ss, ds = src[o], dst[o]
        bounds = np.flatnonzero(np.diff(ds)) + 1
        for seg, d in zip(np.split(ss, bounds), ds[np.r_[0, bounds]]):
            rows[int(d)] = _row_entries(seg)
    ucount = np.array([len(rows.get(d, ())) for d in range(cells)], np.int64)
    row_ptr = np.concatenate([[0], np.cumsum(ucount)]).astype(np.int32)
    pairs = np.array([(s | (d << 16), m) for d in range(cells) for s, m in rows.get(d, ())], np.uint32).reshape(-1, 2)
    usrc = np.unique(src).astype(np.uint16)
    slot = np.zeros(cells, np.int64)
    slot[usrc] = np.arange(len(usrc))
    is_src = np.zeros(cells, bool)
    is_src[usrc] = True
    active = is_src | (ucount > 0)
    ar = np.flatnonzero(active)
    box = (ar.min() // grid, ar.max() // grid, (ar % grid).min(), (ar % grid).max()) if len(ar) else (grid, -1, grid, -1)
    order = ell_order(ucount)
    n_rows, n_slices = len(order), (len(order) + 31) // 32
    widths = [int(((ucount[order[s:s + 32]] + 3) & ~3).max()) for s in range(0, n_rows, 32)]
    ell_off = np.concatenate([[0], np.cumsum(widths)]).astype(np.int32)
    n_groups = int(ell_off[-1])
    row_desc = np.zeros(n_slices * 32, np.uint32)
    ent = np.zeros(n_groups * 32, np.uint32)
    ent_written = np.zeros(n_groups * 32, bool)
    for r, d in enumerate(order):
        s, lane = divmod(r, 32)
        row_desc[r] = d | (ucount[d] << 16)
        words = [sv | (slot[sv] << 12) | (m << 24) for sv, m in rows[int(d)]]
        words += [words[0] & 0xFFFFFF] * (((len(words) + 3) & ~3) - len(words))
        idx = (ell_off[s] + np.arange(len(words))) * 32 + lane
        ent[idx] = words
        ent_written[idx] = True
    cnt = [np.bincount(np.asarray(l, np.int64), minlength=cells) for l in (bo, bt, bc)]
    bgcnt = np.stack(cnt + [is_src.astype(np.int64)], 1).astype(np.uint16)
    binary = all(c.max(initial=0) <= 1 for c in cnt)
    hdr = np.array([len(pairs), n_fg, len(bo), len(bt), len(bc), grid, n_fg, 1 if binary else 0, *box, n_rows, n_slices, n_groups,
                    len(usrc)], np.int32)
    own = np.zeros((256, 2), np.uint32)
    flags = [c > 0 for c in cnt] + [ucount > 0]
    for t in range(256):
        for k in range(4):
            for i in range(4):
                q, b = 4 * (t + 256 * k) + i, 4 * k + i
                if q < cells:
                    own[t, 0] |= (int(flags[0][q]) << b) | (int(flags[1][q]) << (16 + b))
                    own[t, 1] |= (int(flags[2][q]) << b) | (int(flags[3][q]) << (16 + b))
    return dict(hdr=hdr, row_ptr=row_ptr, pairs=pairs, bgcnt=bgcnt, ell_off=ell_off, row_desc=row_desc, ent=ent,
                ent_written=ent_written, usrc=usrc, own=own, ucount=ucount)


_CANARY = 0xA5


def build_plan_guarded(dev, src, dst, bo, bt, bc, grid):
    """dh_build_loss_plan into a buffer over-allocated by the largest sliced-ELL table either row order could need and filled
    with a canary byte; returns (plan bytes, canary intact)."""
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    n_fg = len(src)
    plan_bytes = int(lib.dh_loss_plan_bytes(grid, n_fg))
    assert plan_bytes == plan_layout(grid, n_fg)["total"]
    m = model_plan(src, dst, bo, bt, bc, grid)
    worst = max(ell_groups(m["ucount"], ell_order(m["ucount"], e)) for e in (True, False)) if n_fg else 0
    extra = 4 * 32 * worst + 4096
    buf = torch.full((plan_bytes + extra,), _CANARY, dtype=torch.uint8, device=dev)
    ws_bytes = int(lib.dh_loss_plan_workspace_bytes(grid, n_fg))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    t = [torch.as_tensor(np.asarray(a, np.int32), device=dev) for a in (src, dst, bo, bt, bc)]
    p = [x.data_ptr() if x.numel() else None for x in t]
    N.check(lib.dh_build_loss_plan(p[0], p[1], n_fg, p[2], len(bo), p[3], len(bt), p[4], len(bc), grid, buf.data_ptr(), plan_bytes,
                                   ws.data_ptr(), ws_bytes, torch.cuda.current_stream(dev).cuda_stream), "dh_build_loss_plan")
    host = buf.cpu().numpy()
    return host[:plan_bytes], bool((host[plan_bytes:] == _CANARY).all()), m


def decode_plan(raw, grid, n_fg):
    L = plan_layout(grid, n_fg)
    cells, slices = grid * grid, (grid * grid + 31) // 32
    hdr = np.frombuffer(raw, np.int32, 16, 0)
    n_pairs, n_slices, n_groups, n_usrc = hdr[0], hdr[13], hdr[14], hdr[15]
    assert n_slices <= slices and n_groups * 32 <= L["ent_cap"]
    return dict(hdr=hdr, row_ptr=np.frombuffer(raw, np.int32, cells + 1, L["row"]),
                bgcnt=np.frombuffer(raw, np.uint16, 4 * cells, L["bg"]).reshape(cells, 4),
                pairs=np.frombuffer(raw, np.uint32, 2 * n_pairs, L["pairs"]).reshape(-1, 2),
                ell_off=np.frombuffer(raw, np.int32, n_slices + 1, L["ell_off"]),
                row_desc=np.frombuffer(raw, np.uint32, n_slices * 32, L["row_desc"]),
                ent=np.frombuffer(raw, np.uint32, n_groups * 32, L["ent"]),
                usrc=np.frombuffer(raw, np.uint16, n_usrc, L["usrc_cell"]),
                own=np.frombuffer(raw, np.uint32, 512, L["own_masks"]).reshape(256, 2))


def _rand_pairs(rng, grid, n):
    return rng.integers(0, grid * grid, n), rng.integers(0, grid * grid, n)


def plan_cases():
    """name -> (src, dst, bg_orig, bg_trans, bg_common, grid).  Deterministic."""
    rng = np.random.default_rng(2024)
    cases = {}
    # two destination cells with every source cell, 62 with 255 distinct sources: n_fg = 24002.  In length-class order the two
    # long rows land in different slices and the table needs 262,144 entries (more than the class order's bound allows)
    src, dst = [], []
    for d in range(64):
        s = np.arange(4096) if d in (0, 32) else rng.choice(4096, 255, replace=False)
        src.append(s)
        dst.append(np.full(len(s), d))
    cases["two_full_rows"] = (np.concatenate(src), np.concatenate(dst), [], [], [], 64)
    # 70 rows of length class 255 with unequal lengths (more than two slices of them), scattered destination cells
    dcells = rng.choice(4096, 70, replace=False)
    src, dst = [], []
    for d in dcells:
        s = rng.choice(4096, int(rng.integers(255, 900)), replace=False)
        src.append(s)
        dst.append(np.full(len(s), d))
    cases["class255_rows"] = (np.concatenate(src), np.concatenate(dst), [], [], [], 64)
    # one pair repeated 1000 times (split 255 + 255 + 255 + 235), a neighbouring source 300 times (split rounds interleave)
    src = np.concatenate([np.full(1000, 5), np.full(300, 6), np.full(3, 40), np.arange(100, 140), rng.integers(0, 4096, 500)])
    dst = np.concatenate([np.full(1343, 77), rng.integers(0, 4096, 500)])
    bo = rng.integers(0, 4096, 900)
    cases["split_multiplicities"] = (src, dst, bo, rng.integers(0, 4096, 900), bo[:300], 64)
    cases["one_source_all_destinations"] = (np.full(4096, 1234), np.arange(4096), [], [], [], 64)
    cases["single_pair"] = (np.array([4095]), np.array([0]), [17], [17], [3], 64)
    cases["background_only"] = (np.zeros(0, np.int64), np.zeros(0, np.int64), rng.integers(0, 4096, 2000),
                                rng.integers(0, 4096, 700), np.concatenate([np.arange(64), np.arange(64)]), 64)
    cases["grid1"] = (np.zeros(600, np.int64), np.zeros(600, np.int64), [0, 0, 0], [0], [0, 0], 1)
    s, d = _rand_pairs(rng, 8, 3000)
    cases["grid8"] = (s, d, rng.integers(0, 64, 40), rng.integers(0, 64, 40), rng.integers(0, 64, 10), 8)
    s, d = _rand_pairs(rng, 48, 20000)
    cases["grid48"] = (s, d, np.nonzero(rng.random(2304) < 0.3)[0], np.nonzero(rng.random(2304) < 0.3)[0],
                       np.nonzero(rng.random(2304) < 0.5)[0], 48)
    s, d = _rand_pairs(rng, 64, 30000)
    cases["grid64"] = (s, d, rng.integers(0, 4096, 3000), rng.integers(0, 4096, 3000), rng.integers(0, 4096, 3000), 64)
    return cases


def test_shipped_plans_keep_their_ell_order(golden_pc):
    """Plans of rigid edits have rows far below 255 entries: ordering rows by their exact length gives the same table as
    ordering them by length class (host model on the golden cfg1 correspondences)."""
    _, gp = golden_pc
    pc = O.process_correspondences(gp["cfg1/corr"].astype(np.int64), 512, 0)
    src = pc["original_y"] * 64 + pc["original_x"]
    dst = pc["transformed_y"] * 64 + pc["transformed_x"]
    m = model_plan(src, dst, [], [], [], 64)
    assert 0 < m["ucount"].max() <= 64
    assert np.array_equal(ell_order(m["ucount"], True), ell_order(m["ucount"], False))


def test_class_order_overflows_the_plan_bound_on_two_full_rows():
    """The input of test_plan_matches_host_model[two_full_rows] is the one that breaks the length-class order."""
    src, dst, _, _, _, grid = plan_cases()["two_full_rows"]
    m = model_plan(src, dst, [], [], [], grid)
    cap = plan_layout(grid, len(src))["ent_cap"]
    assert len(src) == 24002
    assert 32 * ell_groups(m["ucount"], ell_order(m["ucount"], False)) == 262144 > cap
    assert 32 * ell_groups(m["ucount"], ell_order(m["ucount"], True)) <= cap


@gpu
@pytest.mark.parametrize("name", list(plan_cases()))
def test_plan_matches_host_model(dev, name):
    src, dst, bo, bt, bc, grid = plan_cases()[name]
    raw, canary_ok, m = build_plan_guarded(dev, src, dst, bo, bt, bc, grid)
    assert canary_ok, "the plan builder wrote past the end of the plan"
    got = decode_plan(raw, grid, len(src))
    assert np.array_equal(got["hdr"], m["hdr"]), (got["hdr"], m["hdr"])
    for k in ("row_ptr", "pairs", "bgcnt", "ell_off", "row_desc", "usrc", "own"):
        assert np.array_equal(got[k], m[k]), k
    w = m["ent_written"]
    assert np.array_equal(got["ent"][w], m["ent"][w])
    assert 32 * m["hdr"][14] <= plan_layout(grid, len(src))["ent_cap"]
    # the library accepts the plan
    from diffusionhandles_b200 import _native as N
    desc = N.dh_loss_plan_desc()
    assert N.load().dh_loss_plan_info(raw[:64].tobytes(), ctypes.byref(desc)) == 0
    assert (desc.n_pairs, desc.flags, desc.ell_slices, desc.ell_groups, desc.n_src_cells) == \
        (m["hdr"][0], m["hdr"][7], m["hdr"][13], m["hdr"][14], m["hdr"][15])


# ------------------------------------------------------------------------------------------------
# kernel variants against the fp64 oracle
# ------------------------------------------------------------------------------------------------
def _pc(src, dst, bo, bt, bc, grid):
    yx = lambda c: (np.asarray(c, np.int64) // grid, np.asarray(c, np.int64) % grid)      # noqa: E731
    pc = {}
    pc["original_y"], pc["original_x"] = yx(src)
    pc["transformed_y"], pc["transformed_x"] = yx(dst)
    pc["background_y_orig"], pc["background_x_orig"] = yx(bo)
    pc["background_y_trans"], pc["background_x_trans"] = yx(bt)
    pc["background_y"], pc["background_x"] = yx(bc)
    return pc


def _lists(rng, grid, binary, n_fg=300):
    """Foreground pairs with duplicates; background lists from a mask (every cell at most once: the bit-mask instantiations)
    or drawn with replacement (cells repeat: the count instantiations).  A few hundred pairs keep the sliced-ELL table small
    enough for the shared-memory placements."""
    cells = grid * grid
    src = rng.integers(0, cells, n_fg)
    dst = np.clip(src + rng.integers(-3 * grid, 3 * grid, n_fg), 0, cells - 1)
    if binary:
        bo, bt, bc = (np.flatnonzero(rng.random(cells) < f) for f in (0.4, 0.4, 0.6))
    else:
        bo, bt, bc = (rng.integers(0, cells, int(f * cells)) for f in (0.4, 0.4, 0.6))
    return src, dst, bo, bt, bc


# name -> (grid, layer shapes (C, h, w), background type, patch, kernel that must run, lists, groups per CTA of the default
# launch or None).  dh_guidance_loss drops groups that would idle (sms * (groups - 1) >= work items), so only cases with
# more than 2 x 148 work items (one per flat plane, one per pair of resized planes) run several groups per CTA on a B200.
_F = "loss_fused_kernel<{}, {}, {}, {}>"


def variant_cases():
    rng = np.random.default_rng(11)
    out = {}
    for binary in (True, False):
        b = "true" if binary else "false"
        tag = "bin" if binary else "cnt"
        out[f"flat64_{tag}"] = (64, [(6, 64, 64)], "global_avg", 1, _F.format(64, b, 1, 4), _lists(rng, 64, binary), None)
        out[f"one_resized_{tag}"] = (64, [(5, 32, 32)], "global_avg", 1, _F.format(64, b, 2, 3), _lists(rng, 64, binary), None)
        out[f"two_resized_{tag}"] = (64, [(4, 32, 32), (3, 16, 16), (2, 64, 64)], "global_avg", 1, _F.format(64, b, 1, 3),
                                     _lists(rng, 64, binary), None)
        s, d, _, _, _, _ = plan_cases()["two_full_rows"]
        _, _, bo, bt, bc = _lists(rng, 64, binary)
        out[f"large_plan_{tag}"] = (64, [(4, 64, 64)], "local_avg", 1, _F.format(64, b, 0, 3), (s, d, bo, bt, bc), None)
        out[f"grid32_{tag}"] = (32, [(5, 32, 32), (3, 16, 16)], "global_avg", 1, _F.format(0, b, 0, 3), _lists(rng, 32, binary), None)
        out[f"grid48_{tag}"] = (48, [(4, 48, 48), (3, 24, 24)], "global_avg", 1, _F.format(0, b, 0, 3), _lists(rng, 48, binary), None)
    # enough work items for several groups per CTA (count lists: the instantiations the shipped configs never run); their lists
    # come from a generator of their own, so the other cases keep their inputs
    rm = np.random.default_rng(12)
    out["flat64_many_cnt"] = (64, [(640, 64, 64)], "global_avg", 1, _F.format(64, "false", 1, 4), _lists(rm, 64, False), 4)
    out["one_resized_many_cnt"] = (64, [(640, 32, 32)], "global_avg", 1, _F.format(64, "false", 2, 3), _lists(rm, 64, False), 3)
    out["grid48_many_cnt"] = (48, [(320, 48, 48)], "global_avg", 1, _F.format(0, "false", 0, 3), _lists(rm, 48, False), 3)
    out["patch3_native"] = (64, [(4, 64, 64)], "local_avg", 3, "loss_patch_kernel", _lists(rng, 64, True), None)
    out["patch3_resized"] = (64, [(3, 32, 32), (2, 16, 16)], "local_avg", 3, "loss_patch_kernel", _lists(rng, 64, False), None)
    out["patch1_odd_area"] = (64, [(4, 9, 9), (3, 13, 13)], "global_avg", 1, "loss_patch_kernel", _lists(rng, 64, False), None)
    out["grid63_patch1"] = (63, [(3, 63, 63)], "local_avg", 1, "loss_patch_kernel", _lists(rng, 63, False), None)
    out["grid63_patch3"] = (63, [(3, 63, 63), (2, 21, 21)], "local_avg", 3, "loss_patch_kernel", _lists(rng, 63, True), None)
    return out


FUSED_VARIANTS = {_F.format(g, b, m, k) for g, b, m, k in
                  [(0, "false", 0, 3), (0, "true", 0, 3), (64, "false", 0, 3), (64, "true", 0, 3), (64, "false", 1, 3),
                   (64, "true", 1, 3), (64, "false", 2, 3), (64, "true", 2, 3), (64, "false", 1, 4), (64, "true", 1, 4)]}


def _inputs(name, shapes):
    gen = torch.Generator().manual_seed(sum(map(ord, name)))
    curs = [torch.randn(s, generator=gen) for s in shapes]
    origs = [torch.randn(s, generator=gen) for s in shapes]
    fgw = [0.5 + i for i in range(len(shapes))]
    bgw = [1.75 - 0.5 * i for i in range(len(shapes))]
    return curs, origs, fgw, bgw


def run_variant(dev, name, case):
    """One guidance_loss evaluation (value, per-term parts and autograd gradients, all as NumPy)."""
    from diffusionhandles_b200 import losses
    grid, shapes, lt, patch, _, lists, _ = case
    pc = _pc(*lists, grid)
    curs, origs, fgw, bgw = _inputs(name, shapes)
    dc = [c.to(dev).requires_grad_(True) for c in curs]
    total, parts = losses.guidance_loss(dc, [o.to(dev) for o in origs], pc, fgw, bgw, bg_loss_type=lt,
                                        activations_size=(grid, grid), patch_size=patch)
    grads = torch.autograd.grad(total, dc)
    return total.item(), parts.cpu().numpy(), [g.cpu().numpy() for g in grads]


def kernels_of(fn):
    """The K4 loss kernels that ran inside fn(), from the kernel records of a torch.profiler trace: a dict from the name,
    normalised to 'loss_fused_kernel<kG, kBinary, kMem, kGroups>' or 'loss_patch_kernel', to the set of groups of 256
    threads per CTA it was launched with (its block size / 256)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    found = {}
    for e in events:
        if e.get("cat") != "kernel":
            continue
        m = re.search(r"loss_fused_kernel<(\d+), ?(true|false|\(bool\)[01]), ?(\d+), ?(\d+)>", e["name"])
        if m:
            b = {"(bool)1": "true", "(bool)0": "false"}.get(m.group(2), m.group(2))
            key = _F.format(m.group(1), b, m.group(3), m.group(4))
        elif re.search(r"\bloss_patch_kernel\b", e["name"]):
            key = "loss_patch_kernel"
        else:
            continue
        block = e.get("args", {}).get("block")
        assert block, ("the trace gives no block size for", e["name"], e.get("args"))
        found.setdefault(key, set()).add(block[0] // 256)
    return found


def _check_against_oracle(name, case, total, parts, grads):
    grid, shapes, lt, patch, _, lists = case[:6]
    pc = _pc(*lists, grid)
    curs, origs, fgw, bgw = _inputs(name, shapes)
    ref_total = 0.0
    for l, (c, o) in enumerate(zip(curs, origs)):
        c, o = c.numpy(), o.numpy()
        vf, gf = O.foreground_loss(c, o, pc, size=(grid, grid), patch=patch)
        vb, gb = O.background_loss(c, o, pc, size=(grid, grid), loss_type=lt, patch=patch)
        assert abs(parts[2 * l] - vf) <= 1e-5 * abs(vf), (name, l, "fg", parts[2 * l], vf)
        assert abs(parts[2 * l + 1] - vb) <= 1e-5 * abs(vb), (name, l, "bg", parts[2 * l + 1], vb)
        ref_total += fgw[l] * vf + bgw[l] * vb
        ref_g = fgw[l] * gf + bgw[l] * gb
        amb = O.loss_sign_ambiguity(c, o, pc, size=(grid, grid), bg_loss_type=lt, patch=patch)
        assert amb.mean() < 1e-2, (name, l, amb.mean())
        err = np.where(amb, 0.0, np.abs(grads[l] - ref_g)).max()
        assert err <= 1e-5 * np.abs(ref_g).max(), (name, l, err, np.abs(ref_g).max())
    assert abs(total - ref_total) <= 1e-5 * abs(ref_total), (name, total, ref_total)


@gpu
@pytest.mark.parametrize("name", list(variant_cases()))
def test_variant_matches_oracle(dev, name):
    case = variant_cases()[name]
    res = {}
    ran = kernels_of(lambda: res.setdefault("r", run_variant(dev, name, case)))
    print(f"{name}: {ran}")
    assert set(ran) == {case[4]}, (name, ran)
    if case[6] is not None:
        assert ran[case[4]] == {case[6]}, (name, ran)
    _check_against_oracle(name, case, *res["r"])


def test_every_fused_instantiation_is_selected():
    """The case table names every instantiation (test_variant_matches_oracle checks that each case runs its kernel)."""
    cases = variant_cases()
    assert {c[4] for c in cases.values() if c[4] != "loss_patch_kernel"} == FUSED_VARIANTS


_CHILD_KNOBS = [{"DH_LOSS_MEM": "0"}, {"DH_LOSS_GROUPS": "1"}, {"DH_LOSS_GROUPS": "2"}, {"DH_LOSS_NO_FOUR_GROUPS": "1"}]


def _child_main(out_path):
    """Runs every fused-kernel case with the knobs of this process's environment and saves the results."""
    dev = torch.device("cuda:0")
    saved = {}
    for name, case in variant_cases().items():
        if case[4] == "loss_patch_kernel":
            continue
        res = {}
        ran = kernels_of(lambda: res.setdefault("r", run_variant(dev, name, case)))
        total, parts, grads = res["r"]
        saved[f"{name}/total"] = np.float64(total)
        saved[f"{name}/parts"] = parts
        for i, g in enumerate(grads):
            saved[f"{name}/grad{i}"] = g
        saved[f"{name}/kernels"] = np.array(sorted(ran))
        saved[f"{name}/groups"] = np.array(sorted(g for v in ran.values() for g in v))
    np.savez(out_path, **saved)


@gpu
@pytest.mark.parametrize("knobs", _CHILD_KNOBS, ids=lambda k: "-".join(f"{a}={b}" for a, b in k.items()))
def test_launch_knobs_give_bit_identical_results(dev, tmp_path, knobs):
    """The knobs are read once per process: the same cases run in a child process with the knob set.  Sign counts are
    integers and every sum has a fixed order, so the results must be bit-identical to the default launch.  The *_many_*
    cases have enough work items to run several groups per CTA: their group counts are checked for both launches."""
    out = tmp_path / "child.npz"
    env = dict(os.environ, **knobs)
    for k in ("DH_LOSS_MEM", "DH_LOSS_GROUPS", "DH_LOSS_NO_FOUR_GROUPS", "DH_LOSS_DEBUG_BUF"):
        if k not in knobs:
            env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", str(out)], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    child = np.load(out)
    for name, case in variant_cases().items():
        if case[4] == "loss_patch_kernel":
            continue
        res = {}
        ran = kernels_of(lambda: res.setdefault("r", run_variant(dev, name, case)))
        total, parts, grads = res["r"]
        assert child[f"{name}/total"] == total, (name, knobs)
        assert np.array_equal(child[f"{name}/parts"], parts), (name, knobs)
        for i, g in enumerate(grads):
            assert np.array_equal(child[f"{name}/grad{i}"], g), (name, knobs, i)
        ks = [str(k) for k in child[f"{name}/kernels"]]
        groups = child[f"{name}/groups"].tolist()
        print(f"{knobs} {name}: {ks} groups {groups}, default {ran}")
        assert len(ks) == 1 and ks[0].startswith("loss_fused_kernel<"), (name, ks)
        if case[6] is not None:
            assert ran == {case[4]: {case[6]}}, (name, ran)
            want = int(knobs["DH_LOSS_GROUPS"]) if "DH_LOSS_GROUPS" in knobs else min(case[6], 3)
            assert groups == [want], (name, knobs, groups)
        if knobs.get("DH_LOSS_MEM") == "0":
            assert ks[0].endswith(", 0, 3>"), (name, ks)
        if "DH_LOSS_NO_FOUR_GROUPS" in knobs:
            assert not ks[0].endswith(", 4>"), (name, ks)


# ------------------------------------------------------------------------------------------------
# API edges
# ------------------------------------------------------------------------------------------------
def _edge_pc(seed=3, grid=64, binary=True):
    return _pc(*_lists(np.random.default_rng(seed), grid, binary), grid)


@gpu
@pytest.mark.parametrize("layout", ["eight_flat", "seven_flat_one_resized", "mixed_resized"])
def test_eight_layers_in_one_launch(dev, layout):
    shapes = {"eight_flat": [(3, 64, 64)] * 8,
              "seven_flat_one_resized": [(3, 64, 64)] * 7 + [(4, 32, 32)],
              "mixed_resized": [(3, 64, 64), (4, 32, 32), (2, 16, 16), (3, 64, 64), (2, 48, 48), (5, 32, 32), (1, 64, 64), (2, 8, 8)]}[layout]
    lists = _lists(np.random.default_rng(5), 64, False)
    case = (64, shapes, "global_avg", 1, None, lists, None)
    _check_against_oracle(layout, case, *run_variant(dev, layout, case))


@gpu
def test_a_ninth_layer_is_a_clean_error(dev):
    from diffusionhandles_b200 import losses
    pc = _edge_pc()
    for shape, patch in (((2, 64, 64), 1), ((2, 64, 64), 3)):
        curs = [torch.randn(shape, device=dev, requires_grad=True) for _ in range(9)]
        origs = [torch.randn(shape, device=dev) for _ in range(9)]
        with pytest.raises(ValueError):
            losses.guidance_loss(curs, origs, pc, [1.0] * 9, [1.0] * 9, patch_size=patch)
    torch.cuda.synchronize()


@gpu
def test_layers_without_gradient_and_zero_weights(dev):
    from diffusionhandles_b200 import losses
    pc = _edge_pc()
    shapes = [(3, 64, 64), (4, 32, 32), (2, 64, 64), (3, 16, 16)]
    curs, origs, _, _ = _inputs("nograd", shapes)
    fgw, bgw = [1.5, 0.0, 2.0, 0.0], [0.0, 1.25, 0.75, 0.0]
    for lt in ("global_avg", "local_avg"):
        dc = [c.to(dev).requires_grad_(i % 2 == 0) for i, c in enumerate(curs)]
        total, parts = losses.guidance_loss(dc, [o.to(dev) for o in origs], pc, fgw, bgw, bg_loss_type=lt)
        grads = torch.autograd.grad(total, [dc[0], dc[2]])
        ref_total = 0.0
        for l, (c, o) in enumerate(zip(curs, origs)):
            vf, gf = O.foreground_loss(c.numpy(), o.numpy(), pc)
            vb, gb = O.background_loss(c.numpy(), o.numpy(), pc, loss_type=lt)
            # every per-term value is reported, whatever its weight
            assert abs(parts[2 * l].item() - vf) <= 1e-5 * abs(vf) and abs(parts[2 * l + 1].item() - vb) <= 1e-5 * abs(vb)
            ref_total += fgw[l] * vf + bgw[l] * vb
            if l % 2 == 0:
                ref_g = fgw[l] * gf + bgw[l] * gb
                amb = O.loss_sign_ambiguity(c.numpy(), o.numpy(), pc, bg_loss_type=lt)
                err = np.where(amb, 0.0, np.abs(grads[l // 2].cpu().numpy() - ref_g)).max()
                assert err <= 1e-5 * np.abs(ref_g).max(), (lt, l, err)
        assert abs(total.item() - ref_total) <= 1e-5 * abs(ref_total)
        # a layer whose both weights are zero gets a zero gradient
        dz = [c.to(dev).requires_grad_(True) for c in curs]
        tz, _ = losses.guidance_loss(dz, [o.to(dev) for o in origs], pc, fgw, bgw, bg_loss_type=lt)
        gz = torch.autograd.grad(tz, dz)
        assert not gz[3].any() and gz[0].any()


@gpu
def test_one_channel_single_work_item(dev):
    for grid, shape in ((64, (1, 64, 64)), (64, (1, 16, 16)), (32, (1, 32, 32))):
        lists = _lists(np.random.default_rng(grid + shape[1]), grid, False)
        name = f"c1_{grid}_{shape[1]}"
        case = (grid, [shape], "global_avg", 1, None, lists, None)
        _check_against_oracle(name, case, *run_variant(dev, name, case))


@gpu
def test_cached_runner_is_reusable_and_bit_identical(dev):
    """The launch re-arms its queue counters in the cached workspace: repeated evaluations on one plan, alternating with a
    second plan, give identical bits."""
    from diffusionhandles_b200 import losses
    plans = []
    for seed in (1, 2):
        s, d, bo, bt, bc = (torch.as_tensor(np.asarray(a, np.int32), device=dev) for a in _lists(np.random.default_rng(seed), 64, seed == 1))
        plans.append(losses.LossPlan(64, dev, s, d, bo, bt, bc))
    shapes = [(4, 64, 64), (3, 32, 32)]
    curs, origs, fgw, bgw = _inputs("runner", shapes)
    curs, origs = [c.to(dev) for c in curs], [o.to(dev) for o in origs]
    first = {}
    for it in range(4):
        for k, plan in enumerate(plans):
            for kind in (1, 2) if k == 0 else (1,):
                sel = [0, 1] if kind == 1 else [0]
                out, grads = losses._launch([curs[i] for i in sel], [origs[i] for i in sel], [True] * len(sel),
                                            [fgw[i] for i in sel], [bgw[i] for i in sel], plan, 1, kind)
                res = (out.cpu().numpy(), [g.cpu().numpy() for g in grads])
                if it == 0:
                    first[(k, kind)] = res
                else:
                    ref = first[(k, kind)]
                    assert np.array_equal(res[0], ref[0]) and all(np.array_equal(a, b) for a, b in zip(res[1], ref[1])), (it, k, kind)
    assert not np.array_equal(first[(0, 1)][0], first[(1, 1)][0])


if __name__ == "__main__" and len(sys.argv) == 3 and sys.argv[1] == "--child":
    _child_main(sys.argv[2])
