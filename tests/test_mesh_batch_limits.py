"""CPU: the C-ABI limits of dh_edit_mesh_batch (mesh mode for B transforms of one scene).  Every call passes fake device
pointers and must be rejected before any CUDA call; the rejected calls also pass a workspace size of 0 unless the workspace is
what they test, so a regressed check still stops at the workspace test instead of reaching a launch."""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

OK, INVALID, UNSUPPORTED, WORKSPACE = 0, -1, -2, -4
FAKE = 0x1000          # 256-byte aligned, never dereferenced
H = W = 16
V_BG, F_BG, V_FG, F_FG = H * W, 2 * (H - 1) * (W - 1), 30, 40


def _host(n):
    return (ctypes.c_float * max(n, 1))(*([0.5] * max(n, 1)))


def _call(lib, ws_bytes=0, **kw):
    a = dict(bg_verts=FAKE, V_bg=V_BG, bg_faces=FAKE, F_bg=F_BG, fg_verts=FAKE, fg_colors=FAKE, V_fg=V_FG, fg_faces=FAKE,
             F_fg=F_FG, B=2, angles=None, axes=None, shifts=None, H=H, W=W, R=_host(9), T=_host(3), sx=1.0, sy=1.0, blur=1e-5,
             target_z=FAKE, corr=FAKE, n_corr=FAKE, pix_to_face=None, ws=FAKE)
    a.update(kw)
    nb = max(a["B"], 1) if a["B"] < (1 << 16) else 4
    angles = _host(nb) if a["angles"] is None else a["angles"]
    axes = _host(3 * nb) if a["axes"] is None else a["axes"]
    shifts = _host(3 * nb) if a["shifts"] is None else a["shifts"]
    return lib.dh_edit_mesh_batch(a["bg_verts"], a["V_bg"], a["bg_faces"], a["F_bg"], a["fg_verts"], a["fg_colors"], a["V_fg"],
                                  a["fg_faces"], a["F_fg"], a["B"], angles, axes, shifts, a["H"], a["W"], a["R"], a["T"], a["sx"],
                                  a["sy"], a["blur"], 1, 1, 1, a["target_z"], a["corr"], a["n_corr"], a["pix_to_face"], a["ws"],
                                  ws_bytes, None)


def test_mesh_batch_rejects_what_it_cannot_run():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    null = ctypes.POINTER(ctypes.c_float)()
    # NULL required pointers (device arrays, host transform arrays, camera)
    for name in ("bg_verts", "target_z", "corr", "n_corr", "ws"):
        assert _call(lib, **{name: None}) == INVALID, name
    for name in ("angles", "axes", "shifts", "R", "T"):
        assert _call(lib, **{name: null}) == INVALID, name
    # ... and the mesh arrays whenever their counts say they are read
    assert _call(lib, bg_faces=None) == INVALID
    assert _call(lib, fg_verts=None) == INVALID
    assert _call(lib, fg_colors=None) == INVALID
    assert _call(lib, fg_faces=None) == INVALID
    # no edits, no background vertices, negative counts, foreground faces without vertices
    for b in (0, -1):
        assert _call(lib, B=b) == INVALID, b
    assert _call(lib, V_bg=0) == INVALID
    for name in ("V_bg", "F_bg", "V_fg", "F_fg", "H", "W"):
        assert _call(lib, **{name: -1}) == INVALID, name
    assert _call(lib, V_fg=0, fg_verts=None, fg_colors=None) == INVALID        # F_fg = 40 faces over no vertices
    # negative or NaN blur radius
    assert _call(lib, blur=-1e-5) == INVALID
    assert _call(lib, blur=float("nan")) == INVALID
    # the rows are written as 32-byte vectors
    assert _call(lib, corr=FAKE + 8) == INVALID
    # sizes beyond the kernels: B above the grid-y limit, images above 2^29 pixels, face indices beyond 31 bits
    assert _call(lib, B=65536) == UNSUPPORTED
    assert _call(lib, B=1 << 20) == UNSUPPORTED
    assert _call(lib, H=1 << 15, W=1 << 15) == UNSUPPORTED
    assert _call(lib, F_bg=(1 << 31) - 1, F_fg=1) == UNSUPPORTED
    # a workspace one byte short
    need = int(lib.dh_edit_mesh_batch_workspace_bytes(2, V_BG, V_FG, H, W))
    assert need > 0
    assert _call(lib, ws_bytes=need - 1) == WORKSPACE
    assert _call(lib, ws_bytes=0, V_fg=0, F_fg=0, fg_verts=None, fg_colors=None, fg_faces=None) == WORKSPACE


def test_mesh_batch_workspace_query():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    q = lib.dh_edit_mesh_batch_workspace_bytes
    # zero for every size the call rejects
    for args in ((0, V_BG, V_FG, H, W), (-1, V_BG, V_FG, H, W), (2, 0, V_FG, H, W), (2, V_BG, -1, H, W), (2, V_BG, V_FG, 0, W),
                 (2, V_BG, V_FG, H, 0), (65536, V_BG, V_FG, H, W), (2, V_BG, V_FG, 1 << 15, 1 << 15)):
        assert q(*args) == 0, args
    # it grows with the edits and the foreground, and a foreground-free batch is valid
    sizes = [int(q(b, V_BG, V_FG, H, W)) for b in (1, 2, 4, 8, 16)]
    assert all(s > 0 for s in sizes) and all(b > a for a, b in zip(sizes, sizes[1:]))
    assert 0 < int(q(2, V_BG, 0, H, W)) < int(q(2, V_BG, V_FG, H, W))
    assert int(q(65535, V_BG, V_FG, H, W)) > 0
