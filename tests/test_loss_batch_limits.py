"""CPU: the C-ABI limits of dh_guidance_loss_batch.  Every call passes fake device pointers and a 16-byte plan buffer and
is one the library must reject before any CUDA call, so no request here can reach a launch even if a check regressed."""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

INVALID, UNSUPPORTED, WORKSPACE = -1, -2, -4
FAKE = 0x1000          # 16-byte aligned, never dereferenced


def _edits(N, n, n_layers=1, channels=4, **kw):
    layers = (N.dh_loss_layer * n_layers)()
    for l in layers:
        l.cur = l.orig = l.grad = FAKE
        l.channels, l.h, l.w = channels, 64, 64
        l.fg_weight = l.bg_weight = 1.0
    edits = (N.dh_loss_batch_edit * max(n, 1))()
    plan = ctypes.create_string_buffer(16)
    for e in edits:
        e.layers = ctypes.cast(layers, ctypes.POINTER(N.dh_loss_layer))
        e.n_layers = n_layers
        e.plan = ctypes.addressof(plan)
        e.desc.ell_slices, e.desc.ell_groups, e.desc.n_src_cells, e.desc.flags = 1, 1, 1, 1
        e.n_fg, e.n_bg_orig, e.n_bg_trans, e.n_bg_common = 10, 10, 10, 10
        e.loss_out = FAKE
        for k, v in kw.items():
            setattr(e, k, v)
    return edits, (layers, plan)


def test_batch_entry_rejects_what_it_cannot_run():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    ws_one = int(lib.dh_guidance_loss_batch_workspace_bytes(1, 1, 4))

    def call(edits, n, ws_bytes=None, ws=FAKE):
        return lib.dh_guidance_loss_batch(edits, n, 64, 1, 1, ws, ws_one * max(n, 1) if ws_bytes is None else ws_bytes, None)

    edits, keep = _edits(N, 16)
    assert call(edits, 0) == INVALID                      # no edit
    assert call(None, 3) == INVALID                       # NULL edit array
    assert call(edits, 3, ws=None) == INVALID             # NULL workspace
    big, keep_big = _edits(N, 200)
    assert call(big, 17) == UNSUPPORTED                   # above the 16 edits of one launch
    assert call(big, 200) == UNSUPPORTED                  # above the SM count of any GPU (and the 16 edits)
    nine, keep9 = _edits(N, 2, n_layers=9)
    assert call(nine, 2) == INVALID                       # an edit with 9 layers, as dh_guidance_loss
    # an undersized workspace: every edit gets ws_bytes / n_edits, one byte short of what it needs
    assert call(edits, 3, ws_bytes=3 * ws_one - 1) == WORKSPACE
    assert call(edits, 3, ws_bytes=ws_one) == WORKSPACE
    # list lengths that do not fit a plan: negative (invalid) or beyond the 24-bit sign counts (unsupported)
    neg, keep_neg = _edits(N, 2, n_bg_trans=-1)
    assert call(neg, 2) == INVALID
    huge, keep_huge = _edits(N, 2, n_fg=1 << 24)
    assert call(huge, 2) == UNSUPPORTED
    # one bad edit among good ones rejects the batch with that edit's code
    mixed, keep_mixed = _edits(N, 3)
    mixed[2].n_layers = 9
    assert call(mixed, 3) == INVALID
    mixed[2].n_layers, mixed[1].n_fg = 1, 1 << 24
    assert call(mixed, 3) == UNSUPPORTED
    # a plan with pairs whose descriptor gives no sliced-ELL size (a batch cannot size its shared-memory copy)
    for field in ("ell_slices", "ell_groups"):
        no_ell, keep_ell = _edits(N, 2)
        setattr(no_ell[1].desc, field, 0)
        assert call(no_ell, 2) == INVALID, field
    # ... which is fine without foreground pairs: the empty edit passes, the next one stops the call with its own code
    empty, keep_empty = _edits(N, 2, n_fg=0)
    empty[0].desc.ell_slices = empty[0].desc.ell_groups = 0
    empty[1].n_fg = 1 << 24
    assert call(empty, 2) == UNSUPPORTED
    # grid and kinds are launch-wide and checked for every edit
    assert lib.dh_guidance_loss_batch(edits, 2, 65, 1, 1, FAKE, 2 * ws_one, None) == INVALID
    assert lib.dh_guidance_loss_batch(edits, 2, 64, 1, 3, FAKE, 2 * ws_one, None) == INVALID


def test_batch_workspace_grows_with_the_edits():
    from diffusionhandles_b200 import _native as N
    lib = N.load()
    sizes = [int(lib.dh_guidance_loss_batch_workspace_bytes(n, 3, 1280)) for n in range(1, 17)]
    one = int(lib.dh_guidance_loss_workspace_bytes(3, 1280))
    assert sizes == [n * one for n in range(1, 17)]
    assert all(b > a for a, b in zip(sizes, sizes[1:]))
    assert lib.dh_guidance_loss_batch_workspace_bytes(0, 3, 1280) == 0
    assert lib.dh_guidance_loss_batch_workspace_bytes(17, 3, 1280) == 0
