"""CPU: the C-ABI limits of dh_guidance_loss_patch_batch.  Every call passes fake device pointers and a 16-byte plan buffer and
is one the library must reject before any CUDA call, so no request here can reach a launch even if a check regressed."""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

INVALID, UNSUPPORTED, WORKSPACE = -1, -2, -4
FAKE = 0x1000          # 16-byte aligned, never dereferenced


def _edits(N, n, n_layers=1, channels=4, hw=(64, 64), **kw):
    layers = (N.dh_loss_layer * n_layers)()
    for l in layers:
        l.cur = l.orig = l.grad = FAKE
        l.channels, (l.h, l.w) = channels, hw
        l.fg_weight = l.bg_weight = 1.0
    edits = (N.dh_loss_batch_edit * max(n, 1))()
    plan = ctypes.create_string_buffer(16)
    for e in edits:
        e.layers = ctypes.cast(layers, ctypes.POINTER(N.dh_loss_layer))
        e.n_layers = n_layers
        e.plan = ctypes.addressof(plan)
        e.n_fg, e.n_bg_orig, e.n_bg_trans, e.n_bg_common = 10, 10, 10, 10
        e.loss_out = FAKE
        for k, v in kw.items():
            setattr(e, k, v)
    return edits, (layers, plan)


def test_patch_batch_entry_rejects_what_it_cannot_run():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    ws_one = int(lib.dh_guidance_loss_patch_batch_workspace_bytes(1, 1, 4))
    assert ws_one == int(lib.dh_guidance_loss_patch_workspace_bytes(1, 4)) > 0

    def call(edits, n, ws_bytes=None, ws=FAKE, grid=64, patch=3, fg_kind=1, bg_kind=2):
        return lib.dh_guidance_loss_patch_batch(edits, n, grid, patch, fg_kind, bg_kind, ws,
                                                ws_one * max(n, 1) if ws_bytes is None else ws_bytes, None)

    edits, keep = _edits(N, 16)
    assert call(edits, 0) == INVALID                      # no edit
    assert call(edits, -1) == INVALID
    assert call(None, 3) == INVALID                       # NULL edit array
    assert call(edits, 3, ws=None) == INVALID             # NULL workspace
    big, keep_big = _edits(N, 200)
    assert call(big, 17) == UNSUPPORTED                   # above the 16 edits of one launch
    assert call(big, 200) == UNSUPPORTED
    # launch-wide arguments, checked for every edit: kinds, patch size, grid
    for kw in (dict(fg_kind=2), dict(fg_kind=-1), dict(bg_kind=3), dict(bg_kind=-1), dict(patch=0), dict(patch=32), dict(grid=0),
               dict(grid=65)):
        assert call(edits, 2, **kw) == INVALID, kw
    # layer shapes beyond the grid or the 64 x 64 native limit, an empty layer, 9 layers
    for hw in ((65, 64), (64, 65), (0, 64), (64, 0)):
        bad, keep_bad = _edits(N, 2, hw=hw)
        assert call(bad, 2) == INVALID, hw
    small, keep_small = _edits(N, 2, hw=(48, 48))
    assert call(small, 2, grid=32) == INVALID              # 48 x 48 maps on a 32 x 32 grid
    nine, keep9 = _edits(N, 2, n_layers=9)
    assert call(nine, 2) == INVALID
    no_ch, keep_ch = _edits(N, 2, channels=0)
    assert call(no_ch, 2) == INVALID
    # NULL per-edit pointers, negative list lengths
    for field in ("plan", "loss_out", "layers"):
        nul, keep_nul = _edits(N, 3)
        setattr(nul[1], field, None)
        assert call(nul, 3) == INVALID, field
    neg, keep_neg = _edits(N, 2, n_bg_trans=-1)
    assert call(neg, 2) == INVALID
    # an undersized workspace: every edit gets ws_bytes / n_edits rounded down to 8, so one byte short leaves each edit 8 short
    assert call(edits, 3, ws_bytes=3 * ws_one - 1) == WORKSPACE
    assert call(edits, 3, ws_bytes=ws_one) == WORKSPACE
    assert call(edits, 1, ws_bytes=ws_one - 1) == WORKSPACE    # a batch of one is checked like the single-edit call
    # one bad edit among good ones rejects the batch with that edit's code
    mixed, keep_mixed = _edits(N, 3)
    mixed[2].n_layers = 9
    assert call(mixed, 3) == INVALID
    mixed[2].n_layers, mixed[1].n_fg = 1, -5
    assert call(mixed, 3) == INVALID


def test_patch_batch_workspace_grows_with_the_edits():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    sizes = [int(lib.dh_guidance_loss_patch_batch_workspace_bytes(n, 3, 1280)) for n in range(1, 17)]
    one = int(lib.dh_guidance_loss_patch_workspace_bytes(3, 1280))
    assert sizes == [n * one for n in range(1, 17)]
    for args in ((0, 3, 1280), (17, 3, 1280), (-1, 3, 1280), (4, 0, 1280), (4, 9, 1280), (4, 3, 0)):
        assert lib.dh_guidance_loss_patch_batch_workspace_bytes(*args) == 0, args
