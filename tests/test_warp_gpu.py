"""GPU: K3 (the activation warp: dh_warp_gather_dense / dh_warp_gather_list) and the dense source maps it reads
(dh_dense_source_maps), bit for bit against plain CPU references.

The warp is a copy, so every comparison is on bit patterns (int32 views), never on float values: -0.0 must stay -0.0,
NaN payloads must survive, and a missing source must give +0.0.  Inputs carry those special patterns.  Every output is a
view in the middle of a sentinel-filled buffer, so a write outside it or a skipped write shows; inputs and maps are
compared with a copy taken before the call.  The fast TMA kernel is run at every compiled stage count and at several
segment lengths and CTA counts (DH_WARP_STAGES / DH_WARP_SEG_CHUNKS / DH_WARP_CTAS_PER_SM, read on every call)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import dh_oracle as O

pytestmark = pytest.mark.gpu

INVALID = -1
INT32_MAX, INT32_MIN = 2 ** 31 - 1, -2 ** 31
SENTINEL = 0x7FBADBAD            # a NaN pattern the kernels never produce
PAD = 4096                       # sentinel words on each side of a guarded view: one whole 16 KB stage
# -0.0, two NaN payloads, the smallest subnormal, +inf, -inf
SPECIAL_BITS = [0x80000000, 0x7FC00001, 0xFFFFFFFF, 0x00000001, 0x7F800000, 0xFF800000]
MAP_KINDS = ("none", "bcast", "ident", "rev", "rand", "oob")
TUNABLES = ("DH_WARP_STAGES", "DH_WARP_SEG_CHUNKS", "DH_WARP_CTAS_PER_SM")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib(dev):
    from diffusionhandles_b200 import _native as N
    return N.load()


@pytest.fixture(autouse=True)
def default_tunables(monkeypatch):
    for k in TUNABLES:
        monkeypatch.delenv(k, raising=False)


def _i32(bits):
    return bits - (1 << 32) if bits >= 1 << 31 else bits


def make_input(gen, shape):
    """Random normals with SPECIAL_BITS sprinkled over about one word in 16 (CPU fp32)."""
    a = torch.randn(shape, generator=gen, dtype=torch.float32)
    flat = a.view(-1).view(torch.int32)
    k = max(len(SPECIAL_BITS), flat.numel() // 16)
    pos = torch.randint(0, flat.numel(), (k,), generator=gen)
    vals = torch.tensor([_i32(b) for b in SPECIAL_BITS], dtype=torch.int32)
    flat[pos] = vals.repeat(k // len(SPECIAL_BITS) + 1)[:k]
    return a


def make_map(gen, kind, hw, e):
    if kind == "none":
        return torch.full((hw,), -1, dtype=torch.int32)
    if kind == "bcast":                               # every cell reads the same source
        return torch.full((hw,), (7919 * e + 3) % hw, dtype=torch.int32)
    if kind == "ident":
        return torch.arange(hw, dtype=torch.int32)
    if kind == "rev":
        return torch.arange(hw - 1, -1, -1, dtype=torch.int32)
    m = torch.randint(0, hw, (hw,), generator=gen, dtype=torch.int32)    # repeats included
    if kind == "rand":
        return m
    oob = torch.tensor([hw, INT32_MAX, INT32_MIN, -2, -1], dtype=torch.int32)
    pick = oob[torch.randint(0, len(oob), (hw,), generator=gen)]
    return torch.where(torch.rand(hw, generator=gen) < 0.5, pick, m)


def make_maps(gen, B, hw, k0=0):
    """(B, hw) int32, edit e gets map kind k0 + e (mod 6) and its own random draw."""
    return torch.stack([make_map(gen, MAP_KINDS[(k0 + e) % len(MAP_KINDS)], hw, e) for e in range(B)])


def place(t, dev, offset=0):
    """(buffer, view): a copy of CPU tensor t (4-byte elements) at word offset PAD + offset of a sentinel-filled int32
    device buffer.  The view is contiguous, with t's dtype and shape."""
    n = t.numel()
    buf = torch.full((PAD + offset + n + PAD,), SENTINEL, dtype=torch.int32)
    buf[PAD + offset:PAD + offset + n] = t.reshape(-1).view(torch.int32)
    buf = buf.to(dev)
    return buf, buf[PAD + offset:PAD + offset + n].view(t.dtype).view(t.shape)


def place_empty(shape, dev, offset=0, dtype=torch.float32):
    n = int(np.prod(shape))
    buf = torch.full((PAD + offset + n + PAD,), SENTINEL, dtype=torch.int32, device=dev)
    return buf, buf[PAD + offset:PAD + offset + n].view(dtype).view(shape)


def assert_bits(got, want, what):
    got, want = got.reshape(-1).view(torch.int32).cpu(), want.reshape(-1).view(torch.int32).cpu()
    assert got.shape == want.shape, what
    if not torch.equal(got, want):
        bad = (got != want).nonzero().flatten()
        i = int(bad[0])
        raise AssertionError(f"{what}: {bad.numel()} of {got.numel()} words differ, first at {i}: "
                             f"got {int(got[i]) & 0xFFFFFFFF:#010x}, want {int(want[i]) & 0xFFFFFFFF:#010x}")


def assert_guard(buf, offset, n, what):
    assert bool((buf[:PAD + offset] == SENTINEL).all()), f"{what}: write before the output"
    assert bool((buf[PAD + offset + n:] == SENTINEL).all()), f"{what}: write after the output"


def ref_dense(a, m):
    """out[e,c,q] = a[e,c,m[e,q]] if 0 <= m[e,q] < hw else +0.0, on bit patterns (int32)."""
    B, C_ = a.shape[:2]
    hw = m.shape[1]
    bits = a.reshape(B, C_, hw).view(torch.int32)
    ok = (m >= 0) & (m < hw)
    idx = torch.where(ok, m, 0).long()[:, None, :].expand(B, C_, hw)
    g = torch.gather(bits, 2, idx)
    return torch.where(ok[:, None, :], g, 0).reshape(a.shape)


def ref_list(a, idx):
    """out[c,i] = a[c, idx[i]] if 0 <= idx[i] < hw else +0.0 (a (C,hw) fp32), on bit patterns."""
    hw = a.shape[1]
    bits = a.view(torch.int32)
    ok = (idx >= 0) & (idx < hw)
    g = bits[:, torch.where(ok, idx, 0).long()]
    return torch.where(ok[None, :], g, 0)


def warp_checked(dev, levels, maps, in_off=0, out_off=0, map_off=0, reps=1):
    """warp_stacks on guarded copies of CPU levels / maps; checks outputs, guards and unchanged inputs.  With reps > 1
    the same outputs are cleared back to the sentinel and the call repeated."""
    from diffusionhandles_b200 import warp
    ins = [place(a, dev, in_off) for a in levels]
    ms = [place(m, dev, map_off) for m in maps]
    outs = [place_empty(tuple(a.shape), dev, out_off) for a in levels]
    before = [b.clone() for b, _ in ins + ms]
    refs = [ref_dense(a, m) for a, m in zip(levels, maps)]
    for r in range(reps):
        for b, _ in outs:
            b.fill_(SENTINEL)
        res = warp.warp_stacks([v for _, v in ins], [v for _, v in ms], [v for _, v in outs])
        assert all(x is v for x, (_, v) in zip(res, outs))
        torch.cuda.synchronize()
        for i, ((ob, ov), ref) in enumerate(zip(outs, refs)):
            shape = tuple(levels[i].shape)
            assert_bits(ov, ref, f"level {i} {shape} rep {r}")
            assert_guard(ob, out_off, ov.numel(), f"level {i} {shape}")
    for (b, _), c in zip(ins + ms, before):
        assert torch.equal(b, c), "an input or a map changed"


# ---- 1. fast-path shapes -------------------------------------------------------------------------------------------
FAST_PLANES = [(2, 2), (2, 4), (4, 4), (8, 16), (16, 16), (16, 32), (32, 32), (32, 64), (64, 64)]


def fast_channels(hw):
    """C*hw below one 16 KB chunk, exactly one, three chunks, three chunks and one plane (a partial last chunk)."""
    per = 4096 // hw
    return ([per - 1] if per > 1 else []) + [per, 3 * per, 3 * per + 1]


@pytest.mark.parametrize("B", [1, 3, 37])
@pytest.mark.parametrize("plane", FAST_PLANES, ids=lambda p: f"{p[0]}x{p[1]}")
def test_fast_path_shapes(dev, plane, B):
    h, w = plane
    gen = torch.Generator().manual_seed(1000 * h + w + B)
    starts = range(len(MAP_KINDS)) if B == 1 else ((0, 3) if B == 3 else (0,))
    for C_ in fast_channels(h * w):
        a = make_input(gen, (B, C_, h, w))
        for k0 in starts:
            warp_checked(dev, [a], [make_maps(gen, B, h * w, k0)])


# ---- 2. launch tunables ----------------------------------------------------------------------------------------------
STAGES = ["2", "3", "4", "6", "8", "5", "0"]            # 5 and 0 are not compiled: 4 stages
SEG_CHUNKS = ["1", "3", "10", "1000", "0", "-1"]        # 0 and -1: the default 10
CTAS = ["1", "2", "8", "0", "99"]                       # 0 and 99: the default 1


@pytest.fixture(scope="module")
def tunable_stack(dev):
    """One 4-level stack, B = 8: 64x64x320 (64 chunks per edit, 2560 one-chunk segments - many per CTA at every CTA
    count), 32x32x40 (10 chunks: not a multiple of 3-chunk segments), 16x16x161 (10 chunks and one partial) and
    8x8x1280 (20 chunks)."""
    B = 8
    gen = torch.Generator().manual_seed(7)
    shapes = [(320, 64, 64), (40, 32, 32), (161, 16, 16), (1280, 8, 8)]
    levels = [make_input(gen, (B, c, h, w)) for c, h, w in shapes]
    maps = [make_maps(gen, B, h * w, k0) for k0, (_, h, w) in enumerate(shapes)]
    ins = [place(a, dev)[1] for a in levels]
    ms = [place(m, dev)[1] for m in maps]
    outs = [place_empty(tuple(a.shape), dev) for a in levels]
    refs = [ref_dense(a, m) for a, m in zip(levels, maps)]
    return ins, ms, outs, refs


@pytest.mark.parametrize("stages", STAGES)
def test_launch_tunables(dev, tunable_stack, monkeypatch, stages):
    from diffusionhandles_b200 import warp
    ins, ms, outs, refs = tunable_stack
    configs = [(stages, s, CTAS[i % len(CTAS)]) for i, s in enumerate(SEG_CHUNKS)]
    configs += [(stages, SEG_CHUNKS[i % len(SEG_CHUNKS)], c) for i, c in enumerate(CTAS)]
    for st, seg, ctas in configs:
        monkeypatch.setenv("DH_WARP_STAGES", st)
        monkeypatch.setenv("DH_WARP_SEG_CHUNKS", seg)
        monkeypatch.setenv("DH_WARP_CTAS_PER_SM", ctas)
        for b, _ in outs:
            b.fill_(SENTINEL)
        warp.warp_stacks(ins, ms, [v for _, v in outs])
        torch.cuda.synchronize()
        for i, ((ob, ov), ref) in enumerate(zip(outs, refs)):
            what = f"stages={st} seg={seg} ctas={ctas} level {i}"
            assert_bits(ov, ref, what)
            assert_guard(ob, 0, ov.numel(), what)


# ---- 3. levels -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seg", [None, "1", "3"])
def test_eight_fast_levels(dev, monkeypatch, seg):
    if seg is not None:
        monkeypatch.setenv("DH_WARP_SEG_CHUNKS", seg)
    gen = torch.Generator().manual_seed(8)
    shapes = [(1025, 2, 2), (513, 2, 4), (300, 4, 4), (40, 8, 16), (17, 16, 16), (9, 16, 32), (3, 32, 64), (2, 64, 64)]
    B = 3
    levels = [make_input(gen, (B, c, h, w)) for c, h, w in shapes]
    warp_checked(dev, levels, [make_maps(gen, B, h * w, i) for i, (_, h, w) in enumerate(shapes)])


def test_fast_and_generic_levels_interleaved(dev):
    """Generic levels first, in the middle and last; the five fast ones share one launch."""
    gen = torch.Generator().manual_seed(9)
    shapes = [(7, 24, 24), (3, 64, 64), (1025, 2, 2), (9, 10, 6), (17, 16, 16), (8, 32, 32), (40, 8, 16), (1, 1, 7)]
    B = 3
    levels = [make_input(gen, (B, c, h, w)) for c, h, w in shapes]
    maps = [make_maps(gen, B, h * w, i) for i, (_, h, w) in enumerate(shapes)]
    warp_checked(dev, levels, maps, reps=2)


def test_nine_levels_are_rejected(dev):
    from diffusionhandles_b200 import warp
    gen = torch.Generator().manual_seed(10)
    shapes = [(4, 8, 8)] * 4 + [(3, 5, 5)] + [(2, 16, 16)] * 4
    levels = [place(make_input(gen, (2, c, h, w)), dev)[1] for c, h, w in shapes]
    maps = [place(make_maps(gen, 2, h * w, 4), dev)[1] for _, h, w in shapes]
    outs = [place_empty((2, c, h, w), dev) for c, h, w in shapes]
    with pytest.raises(ValueError):
        warp.warp_stacks(levels, maps, [v for _, v in outs])
    torch.cuda.synchronize()
    for b, v in outs:
        assert bool((b.cpu() == SENTINEL).all())


# ---- 4. generic path -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("plane", [(24, 24), (96, 96), (128, 128), (3, 5), (1, 1), (1, 7), (10, 6)],
                         ids=lambda p: f"{p[0]}x{p[1]}")
def test_generic_path_shapes(dev, plane):
    h, w = plane
    gen = torch.Generator().manual_seed(100 * h + w)
    for C_ in (1, 7, 8, 9):
        a = make_input(gen, (3, C_, h, w))
        for k0 in (0, 3):
            warp_checked(dev, [a], [make_maps(gen, 3, h * w, k0)])


# fast-eligible shapes; an offset of 1-3 words leaves a pointer off 16 bytes (the generic path), 4 keeps it aligned
MISALIGNED_SHAPES = [(3, 8, 32, 32), (2, 3, 64, 64), (3, 1025, 2, 2)]


@pytest.mark.parametrize("offset", [1, 2, 3, 4])
@pytest.mark.parametrize("which", ["in", "map"])
def test_warp_misaligned_in_and_map(dev, which, offset):
    gen = torch.Generator().manual_seed(11 + offset)
    for B, C_, h, w in MISALIGNED_SHAPES:
        a = make_input(gen, (B, C_, h, w))
        m = make_maps(gen, B, h * w, offset)
        warp_checked(dev, [a], [m], in_off=offset if which == "in" else 0, map_off=offset if which == "map" else 0)


@pytest.mark.parametrize("offset", [1, 2, 3, 4])
def test_warp_misaligned_out(dev, offset):
    gen = torch.Generator().manual_seed(21 + offset)
    for B, C_, h, w in MISALIGNED_SHAPES:
        a = make_input(gen, (B, C_, h, w))
        warp_checked(dev, [a], [make_maps(gen, B, h * w, offset)], out_off=offset)
    # all three at once, on a two-level stack
    levels = [make_input(gen, (2, 8, 32, 32)), make_input(gen, (2, 5, 3, 5))]
    maps = [make_maps(gen, 2, 1024, 1), make_maps(gen, 2, 15, 4)]
    warp_checked(dev, levels, maps, in_off=offset, out_off=offset, map_off=offset)


# ---- 5. validation before any launch -----------------------------------------------------------------------------------
@pytest.mark.parametrize("bad", ["null_map", "channels0", "in_is_out", "hw0"])
def test_dense_validates_every_level_before_launching(dev, lib, bad):
    """A valid generic level 0 followed by an invalid level 1: the call is rejected and level 0's output is untouched."""
    from diffusionhandles_b200 import _native as N
    gen = torch.Generator().manual_seed(12)
    a = make_input(gen, (1, 2, 3, 5))
    _, a_dev = place(a, dev)
    _, m_dev = place(make_maps(gen, 1, 15, 4), dev)
    ob, o_dev = place_empty((1, 2, 3, 5), dev)
    arr = (N.dh_warp_level * 2)()
    for l in arr:
        l.inp, l.out, l.src_map, l.channels, l.hw = a_dev.data_ptr(), o_dev.data_ptr(), m_dev.data_ptr(), 2, 15
    _, o2_dev = place_empty((1, 2, 3, 5), dev)
    arr[1].out = o2_dev.data_ptr()
    if bad == "null_map":
        arr[1].src_map = None
    elif bad == "channels0":
        arr[1].channels = 0
    elif bad == "hw0":
        arr[1].hw = 0
    else:
        arr[1].out = arr[1].inp
    assert lib.dh_warp_gather_dense(arr, 2, 1, N.stream_handle(dev)) == INVALID
    torch.cuda.synchronize()
    assert bool((ob.cpu() == SENTINEL).all()), "level 0 was written by a rejected call"


# ---- 6. streams and repeatability --------------------------------------------------------------------------------------
def test_warp_on_a_side_stream(dev):
    from diffusionhandles_b200 import warp
    gen = torch.Generator().manual_seed(13)
    shapes = [(320, 64, 64), (7, 24, 24), (1280, 8, 8)]
    B = 4
    levels = [make_input(gen, (B, c, h, w)) for c, h, w in shapes]
    maps = [make_maps(gen, B, h * w, i) for i, (_, h, w) in enumerate(shapes)]
    src = [a.to(dev) for a in levels]
    msrc = [m.to(dev) for m in maps]
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        ins = [torch.empty_like(a) for a in src]
        ms = [torch.empty_like(m) for m in msrc]
        for d, x in zip(ins + ms, src + msrc):
            d.copy_(x)                                   # the inputs are produced on the side stream
        outs = warp.warp_stacks(ins, ms)
        outs2 = warp.warp_stacks(ins, ms)
    s.synchronize()
    for i, (a, m, o, o2) in enumerate(zip(levels, maps, outs, outs2)):
        ref = ref_dense(a, m)
        assert_bits(o, ref, f"side stream level {i}")
        assert_bits(o2, o, f"second call level {i}")


# ---- 7. gather_list ------------------------------------------------------------------------------------------------------
def _list_idx(gen, n, hw):
    idx = torch.randint(0, hw, (n,), generator=gen, dtype=torch.int32)
    oob = torch.tensor([hw, INT32_MAX, INT32_MIN, -2, -1], dtype=torch.int32)
    pick = oob[torch.randint(0, len(oob), (n,), generator=gen)]
    return torch.where(torch.rand(n, generator=gen) < 0.25, pick, idx)


def gather_list_checked(dev, lib, a, idx, out_off=0):
    from diffusionhandles_b200 import _native as N
    C_, hw = a.shape
    n = idx.numel()
    ab, a_dev = place(a, dev)
    ib, i_dev = place(idx, dev) if n else place(torch.zeros(1, dtype=torch.int32), dev)
    ob, o_dev = place_empty((C_, n), dev, out_off)
    before = [ab.clone(), ib.clone()]
    out_ptr = ob.data_ptr() + 4 * (PAD + out_off)        # (an empty view has no data pointer; the call still needs one)
    rc = lib.dh_warp_gather_list(a_dev.data_ptr(), C_, hw, i_dev.data_ptr(), n, out_ptr, N.stream_handle(dev))
    assert rc == 0
    torch.cuda.synchronize()
    assert_bits(o_dev, ref_list(a, idx), f"gather_list C={C_} n={n} offset {out_off}")
    assert_guard(ob, out_off, C_ * n, f"gather_list C={C_} n={n}")
    assert torch.equal(ab, before[0]) and torch.equal(ib, before[1])


@pytest.mark.parametrize("C_", [1, 7, 8, 9, 1281])
def test_gather_list(dev, lib, C_):
    from diffusionhandles_b200 import warp
    h, w = 24, 40
    gen = torch.Generator().manual_seed(14 + C_)
    a = make_input(gen, (C_, h * w))
    for n in (0, 1, 2, 3, 5, 4099):
        gather_list_checked(dev, lib, a, _list_idx(gen, n, h * w))
        # the Python entry: W[c, n] = A[c, y[n], x[n]]
        y = torch.randint(0, h, (n,), generator=gen)
        x = torch.randint(0, w, (n,), generator=gen)
        W = warp.gather_list(a.view(C_, h, w).to(dev), y.numpy(), x)
        assert tuple(W.shape) == (C_, n)
        assert_bits(W, a.view(C_, h, w)[:, y, x].contiguous(), f"gather_list python C={C_} n={n}")


@pytest.mark.parametrize("offset", [1, 2, 3])
def test_gather_list_misaligned_out(dev, lib, offset):
    gen = torch.Generator().manual_seed(15 + offset)
    for C_ in (1, 9):
        a = make_input(gen, (C_, 960))
        for n in (4, 8, 4096):
            gather_list_checked(dev, lib, a, _list_idx(gen, n, 960), out_off=offset)


# ---- 8. dense source maps -----------------------------------------------------------------------------------------------
def ref_source_maps(corr, n_corr, img_res, sides, winner_src=None):
    """O.dense_source_map per edit, on the first min(n_corr, cap) rows whose four coordinates lie in [0, img_res)."""
    cap = corr.shape[1]
    out = []
    for s in sides:
        per = []
        for e in range(corr.shape[0]):
            rows = corr[e, :min(max(int(n_corr[e]), 0), cap)]
            rows = rows[((rows >= 0) & (rows < img_res)).all(axis=1)]
            per.append(O.dense_source_map(rows, img_res, s, None if winner_src is None else winner_src[e]))
        out.append(np.stack(per))
    return out


def make_corr(rng, B, cap, img_res, hot_cells=None):
    """(B, cap, 4) int64 rows [x_src, y_src, x_dst, y_dst]; with hot_cells, destinations crowd into a few places so many
    rows share a cell at every level.  About one row in 16 has one coordinate outside the image."""
    corr = rng.integers(0, img_res, size=(B, cap, 4), dtype=np.int64)
    if hot_cells:
        spots = rng.integers(0, img_res, size=(hot_cells, 2))
        pick = spots[rng.integers(0, hot_cells, size=(B, cap))]
        corr[:, :, 2:] = np.minimum(pick + rng.integers(0, 3, size=(B, cap, 2)), img_res - 1)
    bad = rng.random((B, cap)) < 1 / 16
    col = rng.integers(0, 4, size=(B, cap))
    vals = np.array([-1, -img_res, img_res, img_res + 5, 2 ** 40, -2 ** 40], dtype=np.int64)
    corr[bad, col[bad]] = vals[rng.integers(0, len(vals), size=int(bad.sum()))]
    return corr


def maps_checked(dev, corr, n_corr, img_res, sides, winner_src=None):
    from diffusionhandles_b200 import warp
    c_dev = torch.from_numpy(corr).to(dev)
    n_dev = torch.from_numpy(np.asarray(n_corr, dtype=np.int32)).to(dev)
    w_dev = None if winner_src is None else torch.from_numpy(winner_src.astype(np.int32)).to(dev)
    before = [c_dev.clone(), n_dev.clone()] + ([w_dev.clone()] if w_dev is not None else [])
    ref = ref_source_maps(corr, n_corr, img_res, sides, winner_src)
    first = None
    for rep in range(2):
        maps = warp.dense_source_maps(c_dev, n_dev, img_res, sides, w_dev)
        got = [m.cpu() for m in maps]
        for s, g, r in zip(sides, got, ref):
            assert g.shape == (corr.shape[0], s * s)
            assert_bits(g, torch.from_numpy(r), f"side {s}")
        if first is None:
            first = got
        else:
            for a, b in zip(first, got):
                assert torch.equal(a, b)
    for a, b in zip(before, [c_dev, n_dev] + ([w_dev] if w_dev is not None else [])):
        assert torch.equal(a, b)


def _winner_src_96(rng, B):
    """(B, 96*96) winner source pixels, -1 = no winner: a single winner at the last pixel of the image, a sparse and a
    dense random field, no winner at all, and winners only on the last pixel of some 8x8 cells (edit e gets field e % 5)."""
    S = 96
    ws = np.full((B, S * S), -1, dtype=np.int64)
    for e in range(B):
        if e % 5 == 0:
            ws[e, S * S - 1] = 1234
        elif e % 5 == 1:
            sparse = rng.random(S * S) < 0.05
            ws[e, sparse] = rng.integers(0, S * S, size=int(sparse.sum()))
        elif e % 5 == 2:
            ws[e] = rng.integers(0, S * S, size=S * S)
        elif e % 5 == 4:
            for cy, cx in ((0, 0), (3, 7), (11, 11), (5, 0)):
                ws[e, (cy * 8 + 7) * S + cx * 8 + 7] = rng.integers(0, S * S)
    return ws


def test_dense_maps_eight_levels_odd_sides(dev):
    rng = np.random.default_rng(16)
    B, cap, S = 5, 300, 96
    sides = [96, 48, 32, 24, 12, 8, 3, 1]
    corr = make_corr(rng, B, cap, S, hot_cells=6)
    n_corr = [0, 1, 150, 299, 300]
    ws = _winner_src_96(rng, B)
    maps_checked(dev, corr, n_corr, S, sides)
    maps_checked(dev, corr, n_corr, S, sides, ws)
    # many rows in one cell: the lowest n wins at every level
    one = np.tile(np.array([[10, 20, 50, 60]], dtype=np.int64), (1, cap, 1))
    one[0, :, 0] = np.arange(cap) % S
    maps_checked(dev, one, [cap], S, sides)


def test_dense_maps_sd2_levels(dev):
    rng = np.random.default_rng(17)
    B, cap, S = 2, 5000, 512
    corr = make_corr(rng, B, cap, S, hot_cells=40)
    ws = rng.integers(-1, S * S, size=(B, S * S), dtype=np.int64)
    ws[1, rng.random(S * S) < 0.9] = -1
    maps_checked(dev, corr, [4000, 5000], S, [64, 32, 16, 8])
    maps_checked(dev, corr, [4000, 5000], S, [64, 32, 16, 8], ws)


def test_dense_maps_count_above_capacity(dev):
    """n_corr above the rows of an edit counts as the capacity: the next edit's rows (or, after the last edit, whatever
    follows the buffer) are never read.  The rows of edit e+1 sit in cells edit e leaves empty, so reading them shows."""
    rng = np.random.default_rng(18)
    B, cap, S = 3, 50, 96
    corr = np.empty((B, cap, 4), dtype=np.int64)
    for e in range(B):                                   # edit e: destinations in column band e of the image
        corr[e, :, 0:2] = rng.integers(0, S, size=(cap, 2))
        corr[e, :, 2] = rng.integers(32 * e, 32 * e + 32, size=cap)
        corr[e, :, 3] = rng.integers(0, S, size=cap)
    sides = [96, 12, 1]
    maps_checked(dev, corr, [cap + 20, 10, cap + 7], S, sides)
    maps_checked(dev, corr, [2 * cap, cap, INT32_MAX], S, sides, _winner_src_96(rng, B))


# ---- Python argument checks that need device tensors ------------------------------------------------------------------------
def test_warp_stacks_rejects_wrong_dtypes_and_layouts(dev):
    from diffusionhandles_b200 import warp
    a = torch.zeros((2, 3, 8, 8), device=dev)
    m = torch.zeros((2, 64), dtype=torch.int32, device=dev)
    with pytest.raises(TypeError):
        warp.warp_stacks([a.double()], [m])
    with pytest.raises(TypeError):
        warp.warp_stacks([a], [m.long()])
    with pytest.raises(TypeError):
        warp.warp_stacks([a], [m], [torch.zeros_like(a, dtype=torch.float64)])
    with pytest.raises(ValueError):
        warp.warp_stacks([torch.zeros((2, 3, 8, 8), device=dev).transpose(2, 3)], [m])
    with pytest.raises(ValueError):
        warp.warp_stacks([a], [torch.zeros((64, 2), dtype=torch.int32, device=dev).t()])
    with pytest.raises(ValueError):
        warp.warp_stacks([a], [m], [torch.zeros((2, 3, 8, 8), device=dev).transpose(2, 3)])
    with pytest.raises(ValueError):                      # levels with different batch sizes
        warp.warp_stacks([a, torch.zeros((3, 3, 8, 8), device=dev)], [m, torch.zeros((3, 64), dtype=torch.int32, device=dev)])
    with pytest.raises(TypeError):
        warp.dense_source_maps(torch.zeros((1, 4, 4), dtype=torch.int32, device=dev),
                               torch.zeros(1, dtype=torch.int32, device=dev), 8, [8])
    with pytest.raises(TypeError):
        warp.gather_list(a[0].double(), [0], [0])
