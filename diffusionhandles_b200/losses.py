"""Drop-in mirror of the reference's ``diffhandles/losses.py`` (same call signatures, 0-d fp32 results that are
differentiable w.r.t. ``activations``) backed by the fused K4 kernel, plus the fused multi-layer entry point
``guidance_loss`` that ``guided_inference`` (guided_stable_diffuser.py:417-434) evaluates every step.

Each call is ONE kernel pass that produces the loss value AND the gradient (stashed for autograd's backward);
backward only rescales the stash by the incoming gradient - and exits on the device when that is 1.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as N
from .guided_stable_diffuser import ProcessedCorrespondences

_FG, _BG_GLOBAL, _BG_LOCAL = 1, 1, 2


def _to_cells(y, x, grid: int, device) -> torch.Tensor:
    """Cell ids y*grid + x on the device.  Host-side index arrays are range checked here (the reference's tensor indexing
    raises IndexError for them; the kernels trust their lists); device tensors come from process_correspondences_device."""
    for name, v in (("y", y), ("x", x)):
        if not (isinstance(v, torch.Tensor) and v.is_cuda):
            a = np.asarray(v.cpu() if isinstance(v, torch.Tensor) else v)
            if a.size and (a.min() < 0 or a.max() >= grid):
                raise IndexError(f"{name} index out of range for a {grid} x {grid} loss grid: [{a.min()}, {a.max()}]")
    yy = torch.as_tensor(np.asarray(y) if not isinstance(y, torch.Tensor) else y).to(device=device, dtype=torch.int64)
    xx = torch.as_tensor(np.asarray(x) if not isinstance(x, torch.Tensor) else x).to(device=device, dtype=torch.int64)
    dev_checked = [(n, v) for n, v in (("y", y), ("x", x)) if isinstance(v, torch.Tensor) and v.is_cuda and v.numel()]
    if dev_checked:      # index tensors that live on the device: one small read-back (these entry points build a plan, which syncs anyway)
        ext = torch.stack([torch.stack([v.min(), v.max()]) for _, v in dev_checked]).cpu()
        for (n, _), (lo, hi) in zip(dev_checked, ext.tolist()):
            if lo < 0 or hi >= grid:
                raise IndexError(f"{n} index out of range for a {grid} x {grid} loss grid: [{int(lo)}, {int(hi)}]")
    return (yy.reshape(-1) * grid + xx.reshape(-1)).to(torch.int32).contiguous()


def _lists(pc, grid: int, device) -> Dict[str, torch.Tensor]:
    """Device-side int32 cell lists for a processed-correspondences dict."""
    if isinstance(pc, ProcessedCorrespondences) and pc.grid == grid and pc.device_lists["fg_src"].device == device:
        return pc.device_lists
    return {
        "fg_src": _to_cells(pc['original_y'], pc['original_x'], grid, device),
        "fg_dst": _to_cells(pc['transformed_y'], pc['transformed_x'], grid, device),
        "bg": _to_cells(pc['background_y'], pc['background_x'], grid, device),
        "bg_orig": _to_cells(pc['background_y_orig'], pc['background_x_orig'], grid, device),
        "bg_trans": _to_cells(pc['background_y_trans'], pc['background_x_trans'], grid, device),
    }


class LossPlan:
    """Device-side loss plan (dh_build_loss_plan): CSR of distinct (src,dst) cell pairs per destination cell with
    multiplicities + per-cell multiplicities of the background lists.  Built once per edit, reused every step."""

    def __init__(self, grid: int, device, fg_src=None, fg_dst=None, bg_orig=None, bg_trans=None, bg_common=None):
        lib = N.load()
        self.grid = grid
        self.n = [int(t.numel()) if t is not None else 0 for t in (fg_src, bg_orig, bg_trans, bg_common)]
        n_fg = self.n[0]
        # the kernels index shared / global memory with these cell ids: range-check them on the device (the reference's tensor
        # indexing raises IndexError); the single read-back rides on the synchronisation the header read below needs anyway
        lists = [t for t in (fg_src, fg_dst, bg_orig, bg_trans, bg_common) if t is not None and t.numel()]
        if lists:
            ext = torch.stack([torch.stack([t.min(), t.max()]) for t in lists]).cpu()
            if int(ext[:, 0].min()) < 0 or int(ext[:, 1].max()) >= grid * grid:
                raise IndexError(f"index out of range for a {grid} x {grid} loss grid (cell ids span [{int(ext[:, 0].min())}, {int(ext[:, 1].max())}])")
        plan_bytes = int(lib.dh_loss_plan_bytes(grid, n_fg))
        ws_bytes = int(lib.dh_loss_plan_workspace_bytes(grid, n_fg))
        if plan_bytes == 0:
            raise NotImplementedError(f"loss grids larger than 64 x 64 are not implemented (got {grid})")
        self.buf = torch.empty(plan_bytes, dtype=torch.uint8, device=device)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=device)

        def p(t):
            return N.ptr(t, torch.int32) if t is not None and t.numel() else None
        N.check(lib.dh_build_loss_plan(p(fg_src), p(fg_dst), n_fg, p(bg_orig), self.n[1], p(bg_trans), self.n[2], p(bg_common),
                                       self.n[3], grid, N.ptr(self.buf), plan_bytes, N.ptr(ws), ws_bytes,
                                       N.stream_handle(torch.device(device))), "dh_build_loss_plan")
        # one small read-back per edit: the plan header tells how big the box-local buffers of the kernel must be
        hdr = self.buf[:64].cpu().numpy().tobytes()
        self.desc = N.dh_loss_plan_desc()
        N.check(lib.dh_loss_plan_info(hdr, C.byref(self.desc)), "dh_loss_plan_info")
        self.n_pairs, self.box_cells, self.flags = self.desc.n_pairs, self.desc.box_cells, self.desc.flags
        self._tables = {}
        self._runners = {}

    def resize_tables(self, h: int, w: int, fg_kind: int, bg_kind: int) -> torch.Tensor:
        """Tables of a layer smaller than the loss grid (cached per shape and loss kind)."""
        key = (h, w, fg_kind, bg_kind)
        if key not in self._tables:
            lib = N.load()
            t = torch.empty(int(lib.dh_loss_resize_tables_bytes()), dtype=torch.uint8, device=self.buf.device)
            N.check(lib.dh_build_loss_resize_tables(N.ptr(self.buf), self.n[0], self.grid, h, w, fg_kind, bg_kind, N.ptr(t),
                                                    N.stream_handle(self.buf.device)), "dh_build_loss_resize_tables")
            self._tables[key] = t
        return self._tables[key]


def _plan_for(pc, grid: int, device, keys=("fg_src", "fg_dst", "bg_orig", "bg_trans", "bg")) -> LossPlan:
    """The (cached) plan of a processed-correspondences dict."""
    cache = getattr(pc, "_loss_plans", None) if isinstance(pc, ProcessedCorrespondences) else None
    key = (grid, str(device))
    if cache is not None and key in cache:
        return cache[key]
    ls = _lists(pc, grid, device)
    plan = LossPlan(grid, device, ls["fg_src"], ls["fg_dst"], ls["bg_orig"], ls["bg_trans"], ls["bg"])
    if isinstance(pc, ProcessedCorrespondences):
        if cache is None:
            pc._loss_plans = {}
        pc._loss_plans[key] = plan
    return plan


def _as_f32(t: torch.Tensor, dev) -> torch.Tensor:
    if t.dtype is torch.float32 and t.device == dev and t.is_contiguous():
        return t            # (only its data pointer is used: no detach needed)
    return t.detach().to(device=dev, dtype=torch.float32).contiguous()


def _needs_general(shapes, grid: int, patch: int, bg_kind: int) -> bool:
    """Whether layers of these (C,h,w) shapes go to the general patch kernel (dh_guidance_loss_patch) instead of K4."""
    # maps smaller than grid/8 (e.g. 4x4) exceed the tap window of the specialised patch-1 kernels: the general kernel takes them
    # 'local_avg' on a layer smaller than the grid needs the whole up-sampled map: the general kernel takes it (no shipped config does)
    # the patch-1 kernels move whole 16-byte groups of a plane: maps whose area is not a multiple of 4 (e.g. 9x9, 63x63) go to the
    # general kernel too
    return (patch != 1 or any(2 * -(-grid // min(sh[1], sh[2])) > 16 for sh in shapes)
            or any((sh[1] * sh[2]) % 4 for sh in shapes)
            or (bg_kind == _BG_LOCAL and any((sh[1], sh[2]) != (grid, grid) for sh in shapes)))


def _layers(plan: LossPlan, shapes, fg_kind: int, bg_kind: int, general: bool):
    """The ctypes ``dh_loss_layer`` array of one plan for layers of these (C,h,w) shapes, with the resize tables of the layers
    smaller than the loss grid (the general patch kernel takes none).  Returns (layers, tables); the caller keeps both alive."""
    layers = (N.dh_loss_layer * len(shapes))()
    tabs = []
    for i, sh in enumerate(shapes):
        if sh[1] > plan.grid or sh[2] > plan.grid:
            raise NotImplementedError(f"activation maps larger than the loss grid ({sh[1]}x{sh[2]} > {plan.grid}) are not implemented")
        layers[i].channels, layers[i].h, layers[i].w = sh
        t = plan.resize_tables(sh[1], sh[2], fg_kind, bg_kind) if not general and (sh[1], sh[2]) != (plan.grid, plan.grid) else None
        tabs.append(t)
        layers[i].resize_tables = N.ptr(t) if t is not None else None
    return layers, tabs


def _launch(curs: Sequence[torch.Tensor], origs: Sequence[torch.Tensor], want_grad: Sequence[bool],
            fgw: Sequence[float], bgw: Sequence[float], plan: LossPlan, fg_kind: int,
            bg_kind: int, patch: int = 1) -> Tuple[torch.Tensor, List[Optional[torch.Tensor]]]:
    lib = N.load()
    dev = curs[0].device
    if dev.type != "cuda":
        raise N.NativeLibraryError("guidance losses run on CUDA only; there is no CPU fallback")
    L = len(curs)
    shapes = tuple(tuple(c.shape) for c in curs)
    general = _needs_general(shapes, plan.grid, patch, bg_kind)
    key = (shapes, fg_kind, bg_kind, patch, general)
    runner = plan._runners.get(key)
    if runner is None:
        # per (plan, shapes): the ctypes layer array, the workspace and the resize tables are created once
        for c, o in zip(curs, origs):
            if c.dim() != 3 or tuple(c.shape) != tuple(o.shape):
                raise ValueError("activations must be (C,h,w) with matching recorded activations")
        layers, tabs = _layers(plan, shapes, fg_kind, bg_kind, general)
        ws_fn = lib.dh_guidance_loss_patch_workspace_bytes if general else lib.dh_guidance_loss_workspace_bytes
        ws_bytes = int(ws_fn(L, max(sh[0] for sh in shapes)))
        runner = (layers, torch.zeros(ws_bytes, dtype=torch.uint8, device=dev), ws_bytes, tabs)   # zero once: the kernel re-arms its queue counters
        plan._runners[key] = runner
    layers, ws, ws_bytes, _ = runner
    grads: List[Optional[torch.Tensor]] = []
    keep = []
    for i in range(L):
        if tuple(origs[i].shape) != shapes[i]:
            raise ValueError("activations must be (C,h,w) with matching recorded activations")
        c32, o32 = _as_f32(curs[i], dev), _as_f32(origs[i], dev)
        g = torch.empty_like(c32) if want_grad[i] else None
        keep.append((c32, o32))
        grads.append(g)
        layers[i].cur, layers[i].orig = c32.data_ptr(), o32.data_ptr()
        layers[i].grad = g.data_ptr() if g is not None else None
        layers[i].fg_weight, layers[i].bg_weight = float(fgw[i]), float(bgw[i])
    out = torch.empty(1 + 2 * L, dtype=torch.float32, device=dev)
    n_fg, n_bo, n_bt, n_bc = plan.n
    st = N.stream_handle(dev)
    if not general:
        N.check(lib.dh_guidance_loss(layers, L, plan.grid, plan.buf.data_ptr(), C.byref(plan.desc), n_fg, n_bo, n_bt, n_bc, fg_kind, bg_kind, out.data_ptr(), ws.data_ptr(), ws_bytes, st), "dh_guidance_loss")
    else:
        N.check(lib.dh_guidance_loss_patch(layers, L, plan.grid, patch, plan.buf.data_ptr(), n_fg, n_bo, n_bt, n_bc, fg_kind, bg_kind,
                                           out.data_ptr(), ws.data_ptr(), ws_bytes, st), "dh_guidance_loss_patch")
    return out, grads


class _FusedLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, spec, *acts):
        L = spec["L"]
        curs, origs = acts[:L], acts[L:]
        want = [ctx.needs_input_grad[1 + i] for i in range(L)]
        out, grads = _launch(curs, origs, want, spec["fgw"], spec["bgw"], spec["plan"], spec["fg_kind"], spec["bg_kind"],
                             spec.get("patch", 1))
        ctx.grads = grads
        ctx.n_inputs = len(acts)
        total, parts = out[0], out[1:]          # views of a buffer that is private to this call
        ctx.mark_non_differentiable(parts)
        return total, parts

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_total, _g_parts):
        lib = N.load()
        res = [None] * (1 + ctx.n_inputs)
        if ctx.grads is None:       # the gradient was produced by the forward pass and handed out (scaled in place) by the first backward
            raise RuntimeError("Trying to backward through the fused guidance loss a second time: its gradient buffers have already been "
                               "handed out. Re-evaluate the loss instead (retain_graph is not supported for this node).")
        live = [(i, g) for i, g in enumerate(ctx.grads) if g is not None]
        ctx.grads = None
        if live:
            dev = live[0][1].device
            scale = _as_f32(g_total, dev).reshape(1)
            ptrs = (C.c_void_p * len(live))(*[g.data_ptr() for _, g in live])
            sizes = (C.c_size_t * len(live))(*[g.numel() for _, g in live])
            # one launch for every layer; exits on the device when the incoming gradient is 1
            N.check(lib.dh_scale_inplace_many(ptrs, sizes, len(live), scale.data_ptr(), N.stream_handle(dev)), "dh_scale_inplace_many")
            for i, g in live:
                res[1 + i] = g
        return tuple(res)


_MAX_PATCH = 31


def _patch_of(patch_size) -> int:
    """patch_size of the local-average losses (losses.py:64: AvgPool2d(patch_size, stride=1, padding=patch_size//2))."""
    p = int(patch_size)
    if p < 1 or p != patch_size:
        raise ValueError(f"patch_size must be a positive integer, got {patch_size!r}")
    if p > _MAX_PATCH:
        raise NotImplementedError(f"patch_size > {_MAX_PATCH} is not implemented (every shipped config uses 1)")
    return p


def _grid_of(activations_size) -> int:
    hs, ws = int(activations_size[0]), int(activations_size[1])
    if hs != ws:
        raise NotImplementedError("only square loss grids are implemented (the reference always uses (64, 64))")
    return hs


def guidance_loss(activations: Sequence[torch.Tensor], activations_orig: Sequence[torch.Tensor], processed_correspondences,
                  fg_weights: Sequence[float], bg_weights: Sequence[float], bg_loss_type: str = 'global_avg',
                  activations_size=(64, 64), patch_size: int = 1, bg_patch_size: Optional[int] = None):
    """sum_l fgw[l]*compute_foreground_loss(l) + bgw[l]*compute_background_loss(l) in ONE fused launch
    (guided_stable_diffuser.py:417-428).  Returns (total 0-d tensor, per-term values (2L,) tensor: fg_0, bg_0, fg_1, ...).
    ``patch_size`` is the foreground patch (fg_patch_size), ``bg_patch_size`` the background one (defaults to the same);
    when the two differ the foreground and the background terms take one launch each."""
    if bg_loss_type not in ('global_avg', 'local_avg'):
        raise ValueError(f'Unknown background loss type: {bg_loss_type}')
    grid = _grid_of(activations_size)
    dev = activations[0].device
    fg_patch = _patch_of(patch_size)
    bg_patch = _patch_of(patch_size if bg_patch_size is None else bg_patch_size) if bg_loss_type == 'local_avg' else fg_patch
    plan = _plan_for(processed_correspondences, grid, dev)
    bg_kind = _BG_GLOBAL if bg_loss_type == 'global_avg' else _BG_LOCAL
    L = len(activations)
    if fg_patch == bg_patch:
        spec = dict(L=L, fgw=list(fg_weights), bgw=list(bg_weights), plan=plan, fg_kind=_FG, bg_kind=bg_kind, patch=fg_patch)
        return _FusedLoss.apply(spec, *activations, *activations_orig)
    zeros = [0.0] * L
    fg_total, fg_parts = _FusedLoss.apply(dict(L=L, fgw=list(fg_weights), bgw=zeros, plan=plan, fg_kind=_FG, bg_kind=0, patch=fg_patch),
                                          *activations, *activations_orig)
    bg_total, bg_parts = _FusedLoss.apply(dict(L=L, fgw=zeros, bgw=list(bg_weights), plan=plan, fg_kind=0, bg_kind=bg_kind, patch=bg_patch),
                                          *activations, *activations_orig)
    return fg_total + bg_total, fg_parts + bg_parts


def guidance_loss_and_grad(activations: Sequence[torch.Tensor], activations_orig: Sequence[torch.Tensor], processed_correspondences,
                           fg_weights: Sequence[float], bg_weights: Sequence[float], bg_loss_type: str = 'global_avg',
                           activations_size=(64, 64), patch_size: int = 1):
    """The same value as ``guidance_loss`` together with d(total)/d(activations[l]) for every layer, WITHOUT going through
    autograd: one fused launch, no graph node, no backward pass.  ``guided_denoise`` uses it and feeds the gradients to the
    U-Net's backward as ``grad_outputs`` (the chain rule the reference's ``autograd.grad(loss, latents)`` applies,
    guided_stable_diffuser.py:430-434).  Returns (total 0-d tensor, per-term values (2L,), [grad_l (C_l,h_l,w_l)])."""
    if bg_loss_type not in ('global_avg', 'local_avg'):
        raise ValueError(f'Unknown background loss type: {bg_loss_type}')
    grid = _grid_of(activations_size)
    plan = _plan_for(processed_correspondences, grid, activations[0].device)
    L = len(activations)
    out, grads = _launch(activations, activations_orig, [True] * L, fg_weights, bg_weights, plan, _FG,
                         _BG_GLOBAL if bg_loss_type == 'global_avg' else _BG_LOCAL, _patch_of(patch_size))
    return out[0], out[1:], grads


MAX_BATCH_EDITS = 16        # edits per batched K4 launch; larger batches run in chunks of this size


def _batch_runner(plans: Sequence[LossPlan], shapes, bg_kind: int, general: bool):
    """The ctypes edit and layer arrays, the workspace and the resize tables of one chunk of edits, created once per (plans,
    shapes, kernel) and cached on the first plan (the entry keeps the plans alive, so their ids stay unique).  ``general``:
    the chunk goes to the general patch kernel (dh_guidance_loss_patch_batch), which takes no resize tables."""
    key = ("batch", tuple(id(p) for p in plans), shapes, bg_kind, general)
    runner = plans[0]._runners.get(key)
    if runner is None:
        lib = N.load()
        n, L = len(plans), len(shapes)
        edits = (N.dh_loss_batch_edit * n)()
        layer_arrays, tabs = [], []
        for e, plan in enumerate(plans):
            layers, t = _layers(plan, shapes, _FG, bg_kind, general)
            layer_arrays.append(layers)
            tabs += t
            edits[e].layers = C.cast(layers, C.POINTER(N.dh_loss_layer))
            edits[e].n_layers = L
            edits[e].plan = plan.buf.data_ptr()
            edits[e].desc = plan.desc
            edits[e].n_fg, edits[e].n_bg_orig, edits[e].n_bg_trans, edits[e].n_bg_common = plan.n
        ws_fn = lib.dh_guidance_loss_patch_batch_workspace_bytes if general else lib.dh_guidance_loss_batch_workspace_bytes
        ws_bytes = int(ws_fn(n, L, max(sh[0] for sh in shapes)))
        # zeroed once: the patch-1 launch re-arms every edit's queue counters
        runner = (tuple(plans), edits, layer_arrays, torch.zeros(ws_bytes, dtype=torch.uint8, device=plans[0].buf.device), ws_bytes, tabs)
        plans[0]._runners[key] = runner
    return runner


def guidance_loss_and_grad_batch(activations: Sequence[torch.Tensor], activations_orig: Sequence[torch.Tensor],
                                 processed_correspondences: Sequence, fg_weights: Sequence[float], bg_weights: Sequence[float],
                                 bg_loss_type: str = 'global_avg', activations_size=(64, 64), patch_size: int = 1):
    """``guidance_loss_and_grad`` for B edits at once: ONE K4 launch per 16 edits (dh_guidance_loss_batch, or
    dh_guidance_loss_patch_batch for the inputs that the single-edit call sends to the general patch kernel: patch_size > 1,
    map areas that are not a multiple of 4 or below grid/8, 'local_avg' on resized layers).

    ``activations[l]`` is (B,C_l,h_l,w_l), what a U-Net run at batch B returns; ``activations_orig[l]`` is (C_l,h_l,w_l), shared
    by every edit (variants of one image), (B,C_l,h_l,w_l), or a sequence of B (C_l,h_l,w_l) tensors - one identity per edit,
    read in place (edits may share a tensor); ``processed_correspondences`` holds B dicts.  The weights are
    the same for every edit.  Returns (totals (B,), parts (B,2L), [grad_l (B,C_l,h_l,w_l)]): row / slice e is bit-identical to
    what ``guidance_loss_and_grad`` returns for edit e alone.  A chunk of one edit runs the single-edit kernels (the library picks
    them)."""
    if bg_loss_type not in ('global_avg', 'local_avg'):
        raise ValueError(f'Unknown background loss type: {bg_loss_type}')
    grid = _grid_of(activations_size)
    patch = _patch_of(patch_size)
    bg_kind = _BG_GLOBAL if bg_loss_type == 'global_avg' else _BG_LOCAL
    pcs = list(processed_correspondences)
    B, L = len(pcs), len(activations)
    if B < 1 or L < 1 or len(activations_orig) != L:
        raise ValueError("guidance_loss_and_grad_batch needs at least one edit and one layer, and one recorded activation per layer")
    for a, o in zip(activations, activations_orig):
        if a.dim() != 4 or a.shape[0] != B:
            raise ValueError(f"activations must be (B,C,h,w) with B = {B} edits, got {tuple(a.shape)}")
        if isinstance(o, torch.Tensor):
            if tuple(o.shape) not in (tuple(a.shape[1:]), tuple(a.shape)):
                raise ValueError(f"recorded activations must be (C,h,w) or (B,C,h,w) of the activations' shape, got {tuple(o.shape)}")
        elif len(o) != B or any(tuple(t.shape) != tuple(a.shape[1:]) for t in o):
            raise ValueError(f"a per-edit list of recorded activations must hold B = {B} tensors of shape {tuple(a.shape[1:])}")
    dev = activations[0].device
    if dev.type != "cuda":
        raise N.NativeLibraryError("guidance losses run on CUDA only; there is no CPU fallback")
    # the recorded activations of every (layer, edit): views, no copy
    orig_rows = [[o if isinstance(o, torch.Tensor) and o.dim() == 3 else o[e] for e in range(B)] for o in activations_orig]
    plans = [_plan_for(pc, grid, dev) for pc in pcs]
    shapes = tuple(tuple(a.shape[1:]) for a in activations)
    out = torch.empty(B, 1 + 2 * L, dtype=torch.float32, device=dev)
    general = _needs_general(shapes, grid, patch, bg_kind)
    lib = N.load()
    curs = [_as_f32(a, dev) for a in activations]
    converted = {}                     # one conversion per distinct tensor (a shared identity is converted once)
    for rows in orig_rows:
        for t in rows:
            if id(t) not in converted:
                converted[id(t)] = _as_f32(t, dev)
    origs = [[converted[id(t)] for t in rows] for rows in orig_rows]        # kept alive until the launches are enqueued
    grads = [torch.empty_like(c) for c in curs]
    plane = [4 * sh[0] * sh[1] * sh[2] for sh in shapes]        # bytes of one edit's slice of layer l
    cur_p, grad_p = [c.data_ptr() for c in curs], [g.data_ptr() for g in grads]
    org_p = [[t.data_ptr() for t in rows] for rows in origs]
    st = N.stream_handle(dev)
    for b0 in range(0, B, MAX_BATCH_EDITS):
        chunk = plans[b0:b0 + MAX_BATCH_EDITS]
        _, edits, layer_arrays, ws, ws_bytes, _ = _batch_runner(chunk, shapes, bg_kind, general)
        for j, layers in enumerate(layer_arrays):
            e = b0 + j
            for l in range(L):
                layers[l].cur, layers[l].grad = cur_p[l] + e * plane[l], grad_p[l] + e * plane[l]
                layers[l].orig = org_p[l][e]
                layers[l].fg_weight, layers[l].bg_weight = float(fg_weights[l]), float(bg_weights[l])
            edits[j].loss_out = out.data_ptr() + 4 * e * (1 + 2 * L)
        if general:
            N.check(lib.dh_guidance_loss_patch_batch(edits, len(chunk), grid, patch, _FG, bg_kind, ws.data_ptr(), ws_bytes, st),
                    "dh_guidance_loss_patch_batch")
        else:
            N.check(lib.dh_guidance_loss_batch(edits, len(chunk), grid, _FG, bg_kind, ws.data_ptr(), ws_bytes, st), "dh_guidance_loss_batch")
    return out[:, 0], out[:, 1:], grads


def compute_foreground_loss(activations, activations_orig, processed_correspondences, patch_size, activations_size):
    """losses.py:4-17."""
    grid = _grid_of(activations_size)
    spec = dict(L=1, fgw=[1.0], bgw=[0.0], plan=_plan_for(processed_correspondences, grid, activations.device), fg_kind=_FG, bg_kind=0,
                patch=_patch_of(patch_size))
    return _FusedLoss.apply(spec, activations, activations_orig)[0]


def compute_background_loss(activations, activations_orig, processed_correspondences, patch_size, activations_size,
                            loss_type='global_avg'):
    """losses.py:19-40."""
    if loss_type not in ('global_avg', 'local_avg'):
        raise ValueError(f'Unknown background loss type: {loss_type}')
    grid = _grid_of(activations_size)
    spec = dict(L=1, fgw=[0.0], bgw=[1.0], plan=_plan_for(processed_correspondences, grid, activations.device),
                fg_kind=0, bg_kind=_BG_GLOBAL if loss_type == 'global_avg' else _BG_LOCAL,
                patch=_patch_of(patch_size) if loss_type == 'local_avg' else 1)       # 'global_avg' ignores the patch
    return _FusedLoss.apply(spec, activations, activations_orig)[0]


def _two_sided(spec_fwd, spec_swapped, feat_map_1, feat_map_2):
    """Loss that is differentiable w.r.t. both maps: |a-b| is symmetric, so the gradient w.r.t. feat_map_1 is
    the same kernel with the roles of the two maps (and of their index lists) swapped."""
    loss = _FusedLoss.apply(spec_fwd, feat_map_2, feat_map_1.detach())[0]
    if feat_map_1.requires_grad:
        other = _FusedLoss.apply(spec_swapped, feat_map_1, feat_map_2.detach())[0]
        loss = loss + (other - other.detach())      # value counted once, gradient flows to feat_map_1
    return loss


def average_feat_l1_loss(feat_map_1, feat_map_2, x1, y1, x2, y2):
    """losses.py:42-49: |mean_n f1[:,y1,x1] - mean_n f2[:,y2,x2]|.mean()."""
    grid = _grid_of(feat_map_1.shape[-2:])
    dev = feat_map_2.device
    a, b = _to_cells(y1, x1, grid, dev), _to_cells(y2, x2, grid, dev)
    fwd = dict(L=1, fgw=[0.0], bgw=[1.0], plan=LossPlan(grid, dev, bg_orig=a, bg_trans=b), fg_kind=0, bg_kind=_BG_GLOBAL)
    swp = dict(L=1, fgw=[0.0], bgw=[1.0], plan=LossPlan(grid, dev, bg_orig=b, bg_trans=a), fg_kind=0, bg_kind=_BG_GLOBAL)
    return _two_sided(fwd, swp, feat_map_1, feat_map_2)


def local_average_feat_l1_loss(feat_map_1, feat_map_2, x1, y1, x2, y2, patch_size=1):
    """losses.py:51-84: mean_c mean_n |avg_p(f1)[c,y1,x1] - avg_p(f2)[c,y2,x2]| (avg_1 is the identity)."""
    patch = _patch_of(patch_size)
    grid = _grid_of(feat_map_1.shape[-2:])
    dev = feat_map_2.device
    a, b = _to_cells(y1, x1, grid, dev), _to_cells(y2, x2, grid, dev)
    fwd = dict(L=1, fgw=[1.0], bgw=[0.0], plan=LossPlan(grid, dev, fg_src=a, fg_dst=b), fg_kind=_FG, bg_kind=0, patch=patch)
    swp = dict(L=1, fgw=[1.0], bgw=[0.0], plan=LossPlan(grid, dev, fg_src=b, fg_dst=a), fg_kind=_FG, bg_kind=0, patch=patch)
    return _two_sided(fwd, swp, feat_map_1, feat_map_2)
