"""CPU: the limits of the multi-scene edit path - the C ABI of dh_edit_mesh_scenes and its workspace query (fake device pointers,
every call rejected before any CUDA call; the rejected calls pass a workspace of 0 unless the workspace is what they test), and
the argument errors of the Python scene calls, raised before any device work."""
import ctypes
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

OK, INVALID, UNSUPPORTED, WORKSPACE = 0, -1, -2, -4
FAKE = 0x1000          # 256-byte aligned, never dereferenced
H = W = 16
V_BG, F_BG = H * W, 2 * (H - 1) * (W - 1)
# three scenes: a large foreground, none at all, a small one
SCENE_V_FG, SCENE_F_FG = (30, 0, 12), (40, 0, 10)


def _i32(values):
    return (ctypes.c_int32 * max(len(values), 1))(*values)


def _host(n):
    return (ctypes.c_float * max(n, 1))(*([0.5] * max(n, 1)))


def _counts(n_scenes=3, V_bg=None, F_bg=None, V_fg=None, F_fg=None):
    return (V_bg or [V_BG] * n_scenes, F_bg or [F_BG] * n_scenes, V_fg or list(SCENE_V_FG[:n_scenes]),
            F_fg or list(SCENE_F_FG[:n_scenes]))


def _call(lib, ws_bytes=0, **kw):
    a = dict(n_scenes=3, bg_verts=FAKE, bg_faces=FAKE, fg_verts=FAKE, fg_colors=FAKE, fg_faces=FAKE, scene_index=[2, 0, 0, 1], B=None,
             angles=None, axes=None, shifts=None, R=_host(9), T=_host(3), sx=1.0, sy=1.0, blur=1e-5, target_z=FAKE, corr=FAKE,
             n_corr=FAKE, pix_to_face=None, ws=FAKE, H=H, W=W, counts=None)
    a.update(kw)
    V_bg, F_bg, V_fg, F_fg = a["counts"] if a["counts"] is not None else _counts(max(min(a["n_scenes"], 3), 1))
    index = a["scene_index"]
    B = len(index) if a["B"] is None else a["B"]
    nb = max(len(index) if isinstance(index, list) else B, 1)
    cnt = [_i32(c) if isinstance(c, list) else c for c in (V_bg, F_bg, V_fg, F_fg)]
    idx = _i32(index) if isinstance(index, list) else index
    angles = _host(nb) if a["angles"] is None else a["angles"]
    axes = _host(3 * nb) if a["axes"] is None else a["axes"]
    shifts = _host(3 * nb) if a["shifts"] is None else a["shifts"]
    return lib.dh_edit_mesh_scenes(a["n_scenes"], a["bg_verts"], a["bg_faces"], cnt[0], cnt[1], a["fg_verts"], a["fg_colors"],
                                   a["fg_faces"], cnt[2], cnt[3], B, idx, angles, axes, shifts, a["H"], a["W"], a["R"], a["T"], a["sx"],
                                   a["sy"], a["blur"], 1, 1, 1, a["target_z"], a["corr"], a["n_corr"], a["pix_to_face"], a["ws"], ws_bytes,
                                   None)


def _query(lib, n_scenes=3, counts=None, scene_index=(2, 0, 0, 1), B=None, h=H, w=W):
    V_bg, F_bg, V_fg, F_fg = counts if counts is not None else _counts(max(min(n_scenes, 3), 1))
    B = len(scene_index) if B is None else B
    return int(lib.dh_edit_mesh_scenes_workspace_bytes(n_scenes, _i32(V_bg), _i32(F_bg), _i32(V_fg), _i32(F_fg), B, _i32(list(scene_index)),
                                                       h, w))


def test_mesh_scenes_rejects_what_it_cannot_run():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    null_f = ctypes.POINTER(ctypes.c_float)()
    null_i = ctypes.POINTER(ctypes.c_int32)()
    # NULL required pointers: device arrays, host transform arrays, camera, count arrays, scene index
    for name in ("bg_verts", "target_z", "corr", "n_corr", "ws"):
        assert _call(lib, **{name: None}) == INVALID, name
    for name in ("angles", "axes", "shifts", "R", "T"):
        assert _call(lib, **{name: null_f}) == INVALID, name
    assert _call(lib, scene_index=null_i, B=4) == INVALID
    for k in range(4):
        counts = list(_counts())
        counts[k] = null_i
        assert _call(lib, counts=tuple(counts)) == INVALID, k
    # ... and the mesh arrays whenever the totals say they are read
    assert _call(lib, bg_faces=None) == INVALID
    assert _call(lib, fg_verts=None) == INVALID
    assert _call(lib, fg_colors=None) == INVALID
    assert _call(lib, fg_faces=None) == INVALID
    # no scenes, no edits, an index outside the table
    for n in (0, -1):
        assert _call(lib, n_scenes=n) == INVALID, n
    for b in (0, -1):
        assert _call(lib, B=b) == INVALID, b
    for bad in ([0, 3], [-1], [2, 0, 1 << 20]):
        assert _call(lib, scene_index=bad) == INVALID, bad
    # no background vertices, negative counts, foreground faces without vertices, negative sizes
    assert _call(lib, counts=_counts(V_bg=[V_BG, 0, V_BG])) == INVALID
    for k in range(4):
        counts = [list(c) for c in _counts()]
        counts[k][1] = -1
        assert _call(lib, counts=tuple(counts)) == INVALID, k
    assert _call(lib, counts=_counts(V_fg=[30, 0, 12], F_fg=[40, 5, 10])) == INVALID
    for name in ("H", "W"):
        assert _call(lib, **{name: -1}) == INVALID, name
    # negative or NaN blur radius, a corr that is not 32-byte aligned
    assert _call(lib, blur=-1e-5) == INVALID
    assert _call(lib, blur=float("nan")) == INVALID
    assert _call(lib, corr=FAKE + 8) == INVALID
    # sizes beyond the kernels: B or n_scenes above the grid-y limit, images above 2^29 pixels, totals beyond 31 bits
    assert _call(lib, scene_index=[0] * 65536) == UNSUPPORTED
    big = 65536
    assert _call(lib, n_scenes=big, counts=([V_BG] * big, [F_BG] * big, [0] * big, [0] * big)) == UNSUPPORTED
    assert _call(lib, H=1 << 15, W=1 << 15) == UNSUPPORTED
    assert _call(lib, counts=_counts(F_bg=[(1 << 31) - 1, 1, 1], F_fg=[1, 0, 0])) == UNSUPPORTED      # joined face index of scene 0
    assert _call(lib, counts=_counts(F_bg=[(1 << 30), (1 << 30), 1])) == UNSUPPORTED                # face total
    assert _call(lib, counts=_counts(V_bg=[(1 << 30), (1 << 30), 1])) == UNSUPPORTED                # vertex total
    # the moved vertices: sum over edits of V_fg, projected as one flat array
    assert _call(lib, counts=_counts(V_fg=[1 << 29, 0, 12], F_fg=[0, 0, 10]), scene_index=[0, 0, 0, 0]) == UNSUPPORTED
    # a workspace one byte short, also for a batch of scenes without any foreground
    need = _query(lib)
    assert need > 0
    assert _call(lib, ws_bytes=need - 1) == WORKSPACE
    assert _call(lib, counts=_counts(V_fg=[0, 0, 0], F_fg=[0, 0, 0]), fg_verts=None, fg_colors=None, fg_faces=None) == WORKSPACE


def test_mesh_scenes_workspace_query():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    # zero for every size the call rejects
    assert _query(lib, n_scenes=0) == 0
    assert _query(lib, scene_index=()) == 0
    assert _query(lib, scene_index=(0, 3)) == 0
    assert _query(lib, scene_index=(-1,)) == 0
    assert _query(lib, counts=_counts(V_bg=[V_BG, 0, V_BG])) == 0
    assert _query(lib, counts=_counts(V_fg=[30, -1, 12])) == 0
    assert _query(lib, counts=_counts(V_fg=[30, 0, 12], F_fg=[40, 5, 10])) == 0
    assert _query(lib, h=0) == 0 and _query(lib, w=0) == 0
    assert _query(lib, scene_index=[0] * 65536) == 0
    assert _query(lib, h=1 << 15, w=1 << 15) == 0
    assert _query(lib, counts=_counts(F_bg=[(1 << 31) - 1, 1, 1], F_fg=[1, 0, 0])) == 0
    # it grows with the edits and with the foreground the edits move
    sizes = [_query(lib, scene_index=[0] * b) for b in (1, 2, 4, 8, 16)]
    assert all(s > 0 for s in sizes) and all(b > a for a, b in zip(sizes, sizes[1:]))
    assert _query(lib, scene_index=(1, 1)) < _query(lib, scene_index=(0, 0))
    assert _query(lib, scene_index=[0] * 65535) > 0


def _scene_tensors(S=3, n=8, device="cpu"):
    g = torch.Generator().manual_seed(0)
    depths = 1.0 + torch.rand((S, 1, n, n), generator=g)
    masks = torch.zeros((S, 1, n, n))
    masks[:, :, 2:6, 2:6] = 1.0
    return depths.to(device), (depths + 0.5).to(device), masks.to(device)


EDIT = (10.0, torch.tensor([0.0, 1.0, 0.0]), torch.tensor([0.1, 0.0, 0.0]))


@pytest.mark.parametrize("mode", ["pc", "mesh"])
def test_scene_call_argument_errors(mode):
    from diffusionhandles_b200 import depth_transform as dt
    call = dt.transform_depth_pc_scenes if mode == "pc" else dt.transform_depth_mesh_scenes
    K = torch.eye(3)
    d, b, m = _scene_tensors()
    one = ([EDIT[0]], [EDIT[1]], [EDIT[2]])
    # mismatched lengths of the per-edit arguments and of scene_index
    with pytest.raises(ValueError):
        call(d, b, m, K, [0, 1], [10.0, 20.0], [EDIT[1]], [EDIT[2], EDIT[2]])
    with pytest.raises(ValueError):
        call(d, b, m, K, [0, 1], *one)
    with pytest.raises(ValueError):
        call(d, b, m, K, [], [], [], [])
    # mismatched scene counts or shapes, scenes of different sizes, a depth that is not (S,1,H,W)
    with pytest.raises(ValueError):
        call(d, b[:2], m, K, [0], *one)
    with pytest.raises(ValueError):
        call(d, b, m[..., :4], K, [0], *one)
    with pytest.raises(ValueError):
        call([d[:1], d[1:2, :, :4, :4]], [b[:1], b[1:2]], [m[:1], m[1:2]], K, [0], *one)
    with pytest.raises(ValueError):
        call(d[:, 0], b, m, K, [0], *one)
    # a batch of more than one image in one scene entry
    with pytest.raises(ValueError):
        call([d[:2]], [b[:2]], [m[:2]], K, [0], *one)
    # scene indices outside the table
    for bad in (3, -1, 100):
        with pytest.raises(IndexError):
            call(d, b, m, K, [bad], *one)


def test_pc_scenes_non_square_and_cpu_tensors():
    from diffusionhandles_b200 import _native as N
    from diffusionhandles_b200 import depth_transform as dt
    K = torch.eye(3)
    d, b, m = _scene_tensors()
    one = ([EDIT[0]], [EDIT[1]], [EDIT[2]])
    # the 'pc' transform needs a square mask (as transform_depth_pc)
    with pytest.raises(RuntimeError, match="square"):
        dt.transform_depth_pc_scenes(d[..., :6], b[..., :6], m[..., :6], K, [0], *one)
    # tensors on the CPU: there is no CPU path
    for call in (dt.transform_depth_pc_scenes, dt.transform_depth_mesh_scenes):
        with pytest.raises(N.NativeLibraryError):
            call(d, b, m, K, [2, 0], [10.0, 5.0], [EDIT[1]] * 2, [EDIT[2]] * 2)
    # an edit of a scene without foreground is the empty-mask result, as the single call gives it (no device needed)
    empty = torch.zeros_like(m)
    for call in (dt.transform_depth_pc_scenes, dt.transform_depth_mesh_scenes):
        disp, corrs = call(d, b, empty, K, [1, 1, 0], [10.0] * 3, [EDIT[1]] * 3, [EDIT[2]] * 3)
        assert disp.shape == (3, 1, 8, 8) and all(c.shape == (0, 4) and c.dtype == torch.int64 for c in corrs)
        for e, s in enumerate((1, 1, 0)):
            ref, _ = dt._empty_mask_result(d[s:s + 1], False)
            assert torch.equal(disp[e:e + 1], ref)
