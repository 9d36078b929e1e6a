"""Drop-in mirror of the reference's ``diffhandles/depth_transform.py`` (same names, argument meaning and
error behaviour) backed by libdiffhandles_b200 (sm_100a CUDA kernels, C ABI in include/dh_b200.h).

There is no CPU implementation here: tensors must live on a CUDA device, otherwise the call raises
``NativeLibraryError``.  Reference lines are cited per function.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import numpy as np
import torch

from . import _native as N
from .engine import get_engine, make_rigid, pixel_grid
from .utils import pack_correspondences  # noqa: F401  (re-exported: the reference's depth_transform imports it too)


def normalize_depth(depth, bounds=None, return_bounds=False):
    """depth_transform.py:15-28: maps each batch element linearly onto [0, 255]; ``bounds`` = (min, max) tensors reuse another
    image's range (use_input_depth_normalization).  Elementwise torch ops in the reference's operation order
    (255 * (x - min), then the division), on whatever device ``depth`` lives."""
    if depth.dim() != 4:
        raise RuntimeError(f"normalize_depth expects a (B,1,H,W) tensor, got {depth.dim()} dimensions")
    if bounds is not None:
        lo, hi = bounds
    else:
        lo, hi = torch.aminmax(depth.flatten(start_dim=1), dim=1)
        lo, hi = lo.reshape(-1, 1, 1, 1), hi.reshape(-1, 1, 1, 1)
    scaled = (depth - lo) * 255 / (hi - lo)
    return (scaled, (lo, hi)) if return_bounds else scaled


def depth_to_mesh(depth: torch.Tensor, intrinsics: torch.Tensor, extrinsics_R: torch.Tensor = None,
                  extrinsics_t: torch.Tensor = None, mask: torch.Tensor = None):
    """depth_transform.py:30-71: a depth map as a triangle mesh.  One vertex per pixel inside ``mask`` (all pixels without
    one), unprojected on the device; every 2x2 block of pixels whose corners are all vertices gives two counter-clockwise
    triangles (bottom-left, top-right, top-left) and (bottom-left, bottom-right, top-right), blocks in raster order; the
    per-vertex ``color`` attribute is (x/(W-1), y/(H-1), 1 if a mask was given else 0), which the renderer carries to the
    target image as the source coordinate of each rendered pixel."""
    from .mesh import Mesh
    H, W = depth.shape[-2], depth.shape[-1]
    dev = depth.device
    inside = torch.ones((H, W), dtype=torch.bool, device=dev) if mask is None else mask.reshape(H, W).to(dev).bool()
    rows, cols = torch.nonzero(inside, as_tuple=True)                       # raster order = vertex order
    world = depth_to_world_coords(depth, intrinsics=intrinsics, extrinsics_R=extrinsics_R, extrinsics_t=extrinsics_t)
    verts = world[rows, cols].contiguous()
    # vertex number of every pixel (-1 outside the mask), then the four corners of every 2x2 block
    number = torch.full((H, W), -1, dtype=torch.int64, device=dev)
    number[rows, cols] = torch.arange(rows.numel(), dtype=torch.int64, device=dev)
    tl, tr, bl, br = number[:-1, :-1], number[:-1, 1:], number[1:, :-1], number[1:, 1:]
    quads = torch.stack([torch.stack([bl, tr, tl], dim=-1), torch.stack([bl, br, tr], dim=-1)], dim=-2)   # (H-1, W-1, 2, 3)
    faces = quads.reshape(-1, 3)
    faces = faces[(faces >= 0).all(dim=-1)].contiguous()
    mesh = Mesh(verts=verts, faces=faces)
    xs, ys = torch.linspace(0, 1, W, device=dev), torch.linspace(0, 1, H, device=dev)
    flag = torch.full((rows.numel(),), 0.0 if mask is None else 1.0, dtype=xs.dtype, device=dev)
    mesh.add_vert_attribute("color", torch.stack([xs[cols], ys[rows], flag], dim=-1))
    return mesh


def _require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise N.NativeLibraryError(
            f"{name} is on {t.device}; diffusionhandles_b200 runs on CUDA (sm_100a) only and has no CPU fallback")


def depth_to_world_coords(depth: torch.Tensor, intrinsics: torch.Tensor, extrinsics_R: torch.Tensor = None,
                          extrinsics_t: torch.Tensor = None):
    """depth_transform.py:589-641.  depth (1,1,H,W) fp32 -> (H,W,3) fp32 points in pytorch3d axes."""
    if depth.shape[0] != 1:
        raise ValueError("Only batch size 1 is supported")
    height, width = depth.shape[-2:]
    if height < 2 or width < 2:
        raise RuntimeError(f'Expected depth to have at least 2 pixels in each dimension, got {height} x {width}.')
    _require_cuda(depth, "depth")
    lib = N.load()
    d = depth.reshape(1, height, width).to(torch.float32).contiguous()
    xs, ys = pixel_grid(height, width, d.device)
    out = torch.empty((height, width, 3), dtype=torch.float32, device=d.device)
    cam = N.make_camera(intrinsics)
    N.check(lib.dh_unproject(N.ptr(d), 1, height, width, C.byref(cam), N.ptr(xs), N.ptr(ys), N.ptr(out),
                             N.stream_handle(d.device)), "dh_unproject")
    if extrinsics_R is not None or extrinsics_t is not None:
        # camera -> world: R^T (p - t) (depth_transform.py:639); general extrinsics are outside the bit-exact contract
        R = torch.eye(3, device=d.device) if extrinsics_R is None else extrinsics_R.to(d.device, torch.float32)
        t = torch.zeros(3, device=d.device) if extrinsics_t is None else extrinsics_t.to(d.device, torch.float32)
        out = (out - t) @ R
    return out


def transform_points(points: torch.Tensor, rot_angle: torch.Tensor = None, rot_axis: torch.Tensor = None,
                     translation: torch.Tensor = None):
    """depth_transform.py:439-459 (torch fp32 variant used by mesh mode and the webapp): Rodrigues rotation
    about the mean of the given points + translation.  Angle in degrees."""
    _require_cuda(points, "points")
    lib = N.load()
    p = points.to(torch.float32).contiguous()
    n = p.shape[0]
    out = torch.empty_like(p)
    ws_bytes = int(lib.dh_transform_points_workspace_bytes(n))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=p.device)
    axis = (C.c_float * 3)(*[float(v) for v in rot_axis.detach().cpu().reshape(-1)[:3]])
    tr = (C.c_float * 3)(*[float(v) for v in translation.detach().cpu().reshape(-1)[:3]])
    N.check(lib.dh_transform_points(N.ptr(p), n, float(rot_angle), axis, tr, N.ptr(out), N.ptr(ws), ws_bytes,
                                    N.stream_handle(p.device)), "dh_transform_points")
    return out


def points_to_depth(points: torch.Tensor, intrinsics: torch.Tensor, output_size: Tuple[int, int],
                    extrinsics_R: torch.Tensor = None, extrinsics_t: torch.Tensor = None, point_mask: torch.Tensor = None):
    """depth_transform.py:643-747.  Z-buffered point splat: returns, like the reference,
    ``(depth_map (1,1,H,W) fp32 on points.device, depth_mask (H,W) bool ndarray, u[visible], v[visible] int64
    ndarrays, visible (N,) bool ndarray)``.  Only identity extrinsics are implemented on the device."""
    if extrinsics_R is not None or extrinsics_t is not None:
        raise NotImplementedError("points_to_depth: only identity extrinsics are supported (all reference callers)")
    _require_cuda(points, "points")
    lib = N.load()
    dev = points.device
    H, W = int(output_size[0]), int(output_size[1])
    pts = points.to(torch.float64).contiguous()
    n = pts.shape[0]
    P = H * W
    st = N.stream_handle(dev)
    cam = N.make_camera(intrinsics)
    i32 = torch.int32
    pix = torch.empty(max(n, 1), dtype=i32, device=dev)
    zkey = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    u = torch.empty(max(n, 1), dtype=i32, device=dev)
    v = torch.empty(max(n, 1), dtype=i32, device=dev)
    zbuf = torch.empty(P, dtype=torch.int64, device=dev)
    winner = torch.empty(P, dtype=i32, device=dev)
    depth_map = torch.empty((H, W), dtype=torch.float32, device=dev)
    target = torch.empty((H, W), dtype=torch.uint8, device=dev)
    visible = torch.zeros(max(n, 1), dtype=torch.uint8, device=dev)
    pm = (torch.zeros(max(n, 1), dtype=torch.uint8, device=dev) if point_mask is None
          else (point_mask.to(dev) != 0).to(torch.uint8).contiguous())
    N.check(lib.dh_project_points(N.ptr(pts), n, H, W, C.byref(cam), N.ptr(pix), N.ptr(zkey), N.ptr(u), N.ptr(v), st),
            "dh_project_points")
    N.check(lib.dh_splat_zbuffer(N.ptr(pix), N.ptr(zkey), None, n, n, max(n, 1), 1, P, N.ptr(zbuf), N.ptr(winner), st),
            "dh_splat_zbuffer")
    N.check(lib.dh_splat_resolve(N.ptr(zbuf), N.ptr(winner), 1, H, W, 0, N.ptr(pm), None, max(n, 1), N.ptr(depth_map),
                                 N.ptr(target), None, None, None, st), "dh_splat_resolve")
    N.check(lib.dh_splat_visible(N.ptr(pix), N.ptr(winner), None, n, n, max(n, 1), 1, P, 0, N.ptr(pm), N.ptr(visible), st),
            "dh_splat_visible")
    vis = visible[:n].bool()
    uv = torch.stack([u[:n][vis], v[:n][vis]]).to(torch.int64).cpu().numpy()
    return (depth_map[None, None], target.bool().cpu().numpy(), uv[0], uv[1], vis.cpu().numpy())


def _pack_mask(mask_f32: torch.Tensor) -> torch.Tensor:
    """(B,H,W) float mask (non-zero = set) -> row-padded bit planes (B,H,ceil(W/32)) int32."""
    lib = N.load()
    B, H, W = mask_f32.shape
    bits = torch.empty((B, H, (W + 31) // 32), dtype=torch.int32, device=mask_f32.device)
    N.check(lib.dh_pack_mask_bits(N.ptr(mask_f32, torch.float32, "mask"), B, H, W, N.ptr(bits), N.stream_handle(mask_f32.device)),
            "dh_pack_mask_bits")
    return bits


def _poisson_device(image: torch.Tensor, mask_bits: torch.Tensor, lap_source: Optional[torch.Tensor] = None,
                    check: bool = False, what: str = "Poisson fill") -> torch.Tensor:
    """fp64 CG fill on the device.  ``check=True`` reads the iteration counts back (one small synchronising copy) and warns
    when a system stopped without reaching the tolerance - the reference's direct solver cannot fail that way."""
    lib = N.load()
    B, H, W = image.shape
    out = torch.empty_like(image)
    ws_bytes = int(lib.dh_poisson_workspace_bytes(B, H, W))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=image.device)
    iters = torch.zeros(B, dtype=torch.int32, device=image.device)
    N.check(lib.dh_poisson_fill_source(N.ptr(image, torch.float32, "image"), N.ptr(mask_bits), None,
                                       N.ptr(lap_source, torch.float32, "lap_source") if lap_source is not None else None,
                                       B, H, W, N.ptr(out), 0, 1e-13, N.ptr(iters), N.ptr(ws), ws_bytes, N.stream_handle(image.device)),
            "dh_poisson_fill_source")
    _poisson_device.last_iters = iters
    if check:
        warn_if_not_converged(iters, what)
    return out


def warn_if_not_converged(iters: torch.Tensor, what: str) -> None:
    """iters: the solver's per-system iteration counts (negative = stopped without reaching the tolerance)."""
    it = iters.cpu().numpy()
    bad = it < 0
    if bad.any():
        import warnings
        warnings.warn(f"{what}: the conjugate-gradient solver did not reach its tolerance for {int(bad.sum())} of {len(it)} system(s) "
                      f"(stopped after {int((-it[bad] - 1).max())} iterations); the filled values are approximate", RuntimeWarning)


def poisson_solve(input_image, mask):
    """depth_transform.py:535-587 - masked Poisson fill (fp64 CG on the device; SuperLU in the reference).
    NumPy in / NumPy out like the reference; the image is processed on the current CUDA device."""
    dev = torch.device("cuda", torch.cuda.current_device())
    arr = np.asarray(input_image)
    img = torch.as_tensor(arr, dtype=torch.float32, device=dev)[None].contiguous()
    m = torch.as_tensor(np.asarray(mask) != 0, device=dev).to(torch.float32)[None].contiguous()
    out = _poisson_device(img, _pack_mask(m), check=True, what="poisson_solve")
    return out[0].cpu().numpy().astype(arr.dtype)


def transform_point_cloud(points, axis, angle_degrees, x, y, z, mask):
    """depth_transform.py:461-533 - rotate a point image about the centroid of the masked points and translate it.
    points (S,S,3) fp32 (NumPy or torch), mask (S,S); returns ``(rotated_points (S,S,3) float64 ndarray,
    modified_indices (S*S,) bool ndarray)`` like the reference (which hard-codes S = 512; any S works here)."""
    lib = N.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    pts = torch.as_tensor(np.asarray(points) if not isinstance(points, torch.Tensor) else points).to(device=dev, dtype=torch.float32)
    shape = tuple(pts.shape)
    pts = pts.reshape(-1, 3).contiguous()
    n = pts.shape[0]
    mk = torch.as_tensor(np.asarray(mask) if not isinstance(mask, torch.Tensor) else mask).to(device=dev)
    mk_flat = (mk.reshape(-1) != 0)
    if mk_flat.numel() != n:
        raise ValueError("mask must have one entry per point")
    rg = make_rigid(angle_degrees, axis, [x, y, z])
    rg.t[:] = [float(x), float(y), float(z)]          # the reference adds the Python floats as given
    out = torch.empty((n, 3), dtype=torch.float64, device=dev)
    cen = torch.empty(3, dtype=torch.float32, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    ws_bytes = int(lib.dh_transform_point_cloud_workspace_bytes(n))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    N.check(lib.dh_transform_point_cloud(N.ptr(pts), N.ptr(mk_flat.to(torch.float32).contiguous()), n, C.byref(rg), N.ptr(out), N.ptr(cen),
                                         N.ptr(cnt), N.ptr(ws), ws_bytes, N.stream_handle(dev)), "dh_transform_point_cloud")
    return out.reshape(shape).cpu().numpy(), mk_flat.cpu().numpy()


def _empty_mask_result(depth, use_input_depth_normalization):
    """No foreground at all (depth_transform.py:203-216): the normalised input disparity and an empty (0,4) int64 list."""
    disparity = 1.0 / depth
    bounds = normalize_depth(disparity, return_bounds=True)[1] if use_input_depth_normalization else None
    return normalize_depth(disparity, bounds=bounds), torch.empty((0, 4), dtype=torch.int64)


def _edit_count(rot_angles, rot_axes, translations) -> int:
    B = len(rot_angles)
    if B < 1 or len(rot_axes) != B or len(translations) != B:
        raise ValueError(f"rot_angles, rot_axes and translations must have one entry per edit (at least one), got {B}, "
                         f"{len(rot_axes)}, {len(translations)}")
    return B


def _as_scene(t: torch.Tensor, H: int, W: int) -> torch.Tensor:
    """One image of H x W elements as a (1,1,H,W) scene; anything else is left for the scene checks to reject."""
    return t.reshape(1, 1, H, W) if t.numel() == H * W else t


def _scene_planes(x, name: str) -> torch.Tensor:
    """Scenes as one (S,1,H,W) tensor: a 4-D tensor is taken as it is, a sequence of (1,1,H,W) tensors is concatenated."""
    if isinstance(x, torch.Tensor):
        if x.dim() != 4 or x.shape[1] != 1 or x.shape[0] < 1:
            raise ValueError(f"{name} must be (S,1,H,W) with at least one scene, got {tuple(x.shape)}")
        return x
    x = list(x)
    if not x:
        raise ValueError(f"{name} must hold at least one scene")
    for t in x:
        if t.shape[0] != 1:
            raise ValueError(f"one image per scene (batch size 1), got a batch of {t.shape[0]} in {name}")
    if len({tuple(t.shape) for t in x}) != 1 or x[0].dim() != 4:
        raise ValueError(f"the scenes of {name} must all be (1,1,H,W) of one size, got {[tuple(t.shape) for t in x]}")
    return x[0] if len(x) == 1 else torch.cat(x)


def _scene_args(depths, bg_depths, fg_masks, scene_index, rot_angles, rot_axes, translations):
    """Argument checks of the scene calls, before any device work: ``(depths, bg_depths, fg_masks, scene_index list, B)``."""
    depths, bg_depths, fg_masks = (_scene_planes(x, n) for x, n in ((depths, "depths"), (bg_depths, "bg_depths"), (fg_masks, "fg_masks")))
    S, H, W = depths.shape[0], depths.shape[-2], depths.shape[-1]
    for name, t in (("bg_depths", bg_depths), ("fg_masks", fg_masks)):
        if tuple(t.shape) != (S, 1, H, W):
            raise ValueError(f"{name} must be {(S, 1, H, W)} like depths, got {tuple(t.shape)}")
    B = _edit_count(rot_angles, rot_axes, translations)
    index = [int(i) for i in (scene_index.tolist() if isinstance(scene_index, torch.Tensor) else scene_index)]
    if len(index) != B:
        raise ValueError(f"scene_index must have one entry per edit ({B}), got {len(index)}")
    for i in index:
        if not 0 <= i < S:
            raise IndexError(f"scene_index {i} outside [0, {S})")
    return depths, bg_depths, fg_masks, index, B


_ROWS_CHUNK_BYTES = 16 << 20


def _rows_to_cpu(corr: torch.Tensor, counts):
    """The first counts[e] rows of corr[e] (B,P,4) for every edit, on the CPU.  Consecutive edits are copied together in chunks
    of up to 16 MB: one large copy runs at a higher rate than many small ones, while a host buffer above glibc's largest mmap
    threshold (32 MB) is mapped and faulted in anew on every call."""
    out, e = [], 0
    while e < len(counts):
        k, n = e + 1, counts[e]
        while k < len(counts) and (n + counts[k]) * 32 <= _ROWS_CHUNK_BYTES:
            n += counts[k]
            k += 1
        rows = corr[e, :counts[e]] if k == e + 1 else torch.cat([corr[j, :counts[j]] for j in range(e, k)])
        if k == e + 1:
            out.append(rows.cpu())
        else:                                                               # each edit owns its rows
            out += [r.clone() for r in torch.split(rows.cpu(), counts[e:k])]
        e = k
    return out


def _gather_planes(planes: torch.Tensor, index) -> torch.Tensor:
    """planes[index] as one contiguous (len(index),...) tensor; the edits of a single scene expand it (no copy for one edit)."""
    if len(set(index)) == 1:
        s = index[0]
        return planes[s:s + 1].expand(len(index), *planes.shape[1:]).contiguous()
    return planes.index_select(0, torch.tensor(index, device=planes.device))


def _scene_masks_present(fg_masks: torch.Tensor, index):
    """Which scenes have a foreground, read with one synchronisation (scenes no edit references are not read)."""
    used = sorted(set(index))
    masks = fg_masks if len(used) == fg_masks.shape[0] else fg_masks[torch.tensor(used, device=fg_masks.device)]
    present = masks.flatten(1).any(1).tolist()
    return dict(zip(used, present))


def _empty_mask_edits(depths, index, edits, use_input_depth_normalization, disparity, correspondences):
    """``_empty_mask_result`` of its scene for each edit in ``edits`` (computed once per scene)."""
    done = {}
    for b in edits:
        s = index[b]
        if s not in done:
            done[s] = _empty_mask_result(depths[s:s + 1], use_input_depth_normalization)
        disparity[b] = done[s][0][0]
        correspondences[b] = done[s][1].clone()


def transform_depth_pc_scenes(depths: torch.Tensor, bg_depths: torch.Tensor, fg_masks: torch.Tensor, intrinsics: torch.Tensor,
                              scene_index, rot_angles, rot_axes, translations, use_input_depth_normalization=False,
                              return_device_result: bool = False):
    """``transform_depth_pc`` for B edits over S scenes as ONE ``EditEngine`` batch.  ``depths`` / ``bg_depths`` / ``fg_masks``
    are (S,1,H,W) (or sequences of S (1,1,H,W) tensors of one size); edit b transforms scene ``scene_index[b]`` by
    (``rot_angles[b]``, ``rot_axes[b]``, ``translations[b]``; ``None`` takes the defaults of the single call).  The scene planes
    are gathered per edit on the device.  Returns ``(disparities (B,1,H,W) fp32, [correspondences (n_b,4) int64 CPU] * B)``,
    entry b equal bit for bit to ``transform_depth_pc`` on its scene; an edit of a scene without foreground gets that scene's
    empty-mask result.  With ``return_device_result=True`` the ``EditResult`` of the edits whose scene has a foreground (in edit
    order; None when there is none) is appended."""
    depths, bg_depths, fg_masks, index, B = _scene_args(depths, bg_depths, fg_masks, scene_index, rot_angles, rot_axes, translations)
    H, W = depths.shape[-2:]
    present = _scene_masks_present(fg_masks, index)
    live = [b for b in range(B) if present[index[b]]]
    if live:
        if H != W:
            raise RuntimeError(f"the 'pc' depth transform needs a square mask, got {H} x {W}")
        _require_cuda(depths, "depths")
    disparity, correspondences, res = [None] * B, [None] * B, None
    if live:
        # defaults of the reference: no rotation about +y, no translation (depth_transform.py:219-224)
        rigids = [make_rigid(0.0 if rot_angles[b] is None else rot_angles[b],
                             torch.tensor([0.0, 1.0, 0.0]) if rot_axes[b] is None else rot_axes[b],
                             torch.zeros(3) if translations[b] is None else translations[b]) for b in live]
        dev, f32 = depths.device, torch.float32
        d, bg, m = (_gather_planes(t.reshape(-1, H, W).to(device=dev, dtype=f32), [index[b] for b in live])
                    for t in (depths, bg_depths, fg_masks))
        res = get_engine(dev, len(live), H, W).run(d, bg, m, intrinsics, rigids,
                                                   use_input_depth_normalization=use_input_depth_normalization, poisson=True)
        # one copy per edit: the engine's rows are small (at most one per foreground pixel), and separate copies measured faster
        # than chunked ones here
        rows = [res.correspondences(e).cpu() for e in range(len(live))]
        if len(live) == B:                        # every edit has a foreground: rows are already in edit order
            out = res.disparity[:, None].clone(), rows
            return (*out, res) if return_device_result else out
        for e, b in enumerate(live):
            disparity[b] = res.disparity[e:e + 1]
            correspondences[b] = rows[e]
    _empty_mask_edits(depths, index, [b for b in range(B) if not present[index[b]]], use_input_depth_normalization, disparity,
                      correspondences)
    out = torch.stack(disparity), correspondences
    return (*out, res) if return_device_result else out


def transform_depth_pc(depth: torch.Tensor, bg_depth: torch.Tensor, fg_mask: torch.Tensor, intrinsics: torch.Tensor,
                       rot_angle: float = None, rot_axis: torch.Tensor = None, translation: torch.Tensor = None,
                       use_input_depth_normalization=False, return_device_result: bool = False):
    """depth_transform.py:198-363 - the default ('pc') depth transform.

    Returns ``(edited disparity (1,1,S,S) fp32 on depth.device in [0,255], correspondences (N,4) int64 CPU)``.
    With ``return_device_result=True`` a third value, the device-side ``EditResult`` (winner indices, masks,
    device copy of the correspondences), is appended for the warp / loss kernels.
    """
    disparity, corrs, res = transform_depth_pc_batch(depth, bg_depth, fg_mask, intrinsics, [rot_angle], [rot_axis], [translation],
                                                     use_input_depth_normalization, return_device_result=True)
    return (disparity, corrs[0], res) if return_device_result else (disparity, corrs[0])


def transform_depth_pc_batch(depth: torch.Tensor, bg_depth: torch.Tensor, fg_mask: torch.Tensor, intrinsics: torch.Tensor,
                             rot_angles, rot_axes, translations, use_input_depth_normalization=False,
                             return_device_result: bool = False):
    """``transform_depth_pc`` for B transforms of one scene: ``transform_depth_pc_scenes`` with one scene.  ``rot_angles`` /
    ``rot_axes`` / ``translations`` hold one entry per edit (``None`` takes the defaults of the single call).  Returns
    ``(disparities (B,1,S,S) fp32 on depth.device, [correspondences (n_b,4) int64 CPU] * B)``, plus the ``EditResult`` (None for
    an empty mask) with ``return_device_result=True``."""
    B = _edit_count(rot_angles, rot_axes, translations)
    H, W = depth.shape[-2:]
    scene = [[_as_scene(t, H, W)] for t in (depth, bg_depth, fg_mask)]
    return transform_depth_pc_scenes(*scene, intrinsics, [0] * B, rot_angles, rot_axes, translations, use_input_depth_normalization,
                                     return_device_result)


def _object_masks(fg_masks) -> torch.Tensor:
    """K object masks as one (K,H,W) tensor: a (K,1,H,W) tensor, or a sequence of K (1,1,H,W) tensors."""
    if isinstance(fg_masks, torch.Tensor):
        if fg_masks.dim() != 4 or fg_masks.shape[1] != 1 or fg_masks.shape[0] < 1:
            raise ValueError(f"fg_masks must be (K,1,H,W) with at least one object, got {tuple(fg_masks.shape)}")
        return fg_masks[:, 0]
    masks = list(fg_masks)
    if not masks:
        raise ValueError("fg_masks must hold at least one object mask")
    if len({tuple(t.shape) for t in masks}) != 1 or masks[0].dim() != 4 or tuple(masks[0].shape[:2]) != (1, 1):
        raise ValueError(f"the object masks must all be (1,1,H,W) of one size, got {[tuple(t.shape) for t in masks]}")
    return torch.cat(masks)[:, 0]


def _object_transforms(K: int, rot_angles, rot_axes, translations):
    """B edits of K objects: ``rot_angles[b][k]`` etc. move object k in edit b.  Returns B."""
    B = _edit_count(rot_angles, rot_axes, translations)
    for b in range(B):
        n = (len(rot_angles[b]), len(rot_axes[b]), len(translations[b]))
        if n != (K, K, K):
            raise ValueError(f"edit {b} must have one transform per object ({K}), got {n[0]} angles, {n[1]} axes, {n[2]} translations")
    return B


MAX_OBJECTS = 16


def transform_depth_pc_objects_batch(depth: torch.Tensor, bg_depth: torch.Tensor, fg_masks, intrinsics: torch.Tensor, rot_angles,
                                     rot_axes, translations, use_input_depth_normalization=False, return_device_result: bool = False):
    """B edits of one scene whose foreground is K disjoint objects, each object with its own rigid transform, as ONE
    ``EditEngine`` batch (``dh_edit_splat_objects``).

    ``fg_masks``: K masks of the scene, a (K,1,H,W) tensor or a sequence of K (1,1,H,W) tensors (non-zero = in the object,
    1 <= K <= 16); they must not overlap, and their union is the foreground.  ``rot_angles`` / ``rot_axes`` / ``translations``
    are (B,K) nested sequences: entry [b][k] moves object k in edit b (``None`` takes the single call's default).  Every object
    rotates about the sequential centroid of its own pixels; the z-buffer sees all moved objects together, so they occlude one
    another (an exact z tie goes to the lower source raster index).  An object without pixels is allowed and its transform is
    ignored.  With K = 1 every result equals ``transform_depth_pc_batch`` bit for bit.  Returns what ``transform_depth_pc_batch``
    returns: ``(disparities (B,1,S,S) fp32, [correspondences (n_b,4) int64 CPU] * B)``, plus the ``EditResult`` (None for an
    empty union) with ``return_device_result=True``."""
    masks = _object_masks(fg_masks)
    K = masks.shape[0]
    if K > MAX_OBJECTS:
        raise ValueError(f"at most {MAX_OBJECTS} objects per edit are supported, got {K}")
    B = _object_transforms(K, rot_angles, rot_axes, translations)
    H, W = masks.shape[-2:]
    if depth.numel() != H * W or bg_depth.numel() != H * W:
        raise ValueError(f"depth and bg_depth must be one {H} x {W} image like the masks, got {tuple(depth.shape)} and "
                         f"{tuple(bg_depth.shape)}")
    inside = masks != 0
    count = inside.sum(0)
    overlap, present = torch.stack([(count > 1).any(), (count > 0).any()]).tolist()     # the one synchronisation
    if overlap:
        raise ValueError("the object masks overlap: every pixel may belong to one object at most")
    if not present:
        disparity, corr = _empty_mask_result(depth.reshape(1, 1, H, W), use_input_depth_normalization)
        out = disparity.expand(B, 1, H, W).clone(), [corr.clone() for _ in range(B)]
        return (*out, None) if return_device_result else out
    if H != W:
        raise RuntimeError(f"the 'pc' depth transform needs a square mask, got {H} x {W}")
    _require_cuda(depth, "depth")
    dev, f32 = depth.device, torch.float32
    ids = torch.arange(1, K + 1, dtype=torch.uint8, device=inside.device).view(K, 1, 1)
    labels = (inside.to(torch.uint8) * ids).amax(0)                    # k + 1 on object k (the masks are disjoint)
    planes = [t.reshape(1, H, W).to(device=dev, dtype=f32) for t in (depth, bg_depth)] + [(count > 0).to(device=dev, dtype=f32)[None],
                                                                                           labels.to(dev)[None]]
    d, bg, m, lab = (t.expand(B, H, W).contiguous() for t in planes)
    rigids = [make_rigid(0.0 if rot_angles[b][k] is None else rot_angles[b][k],
                         torch.tensor([0.0, 1.0, 0.0]) if rot_axes[b][k] is None else rot_axes[b][k],
                         torch.zeros(3) if translations[b][k] is None else translations[b][k]) for b in range(B) for k in range(K)]
    res = get_engine(dev, B, H, W).run_objects(d, bg, m, lab, K, intrinsics, rigids,
                                               use_input_depth_normalization=use_input_depth_normalization, poisson=True)
    rows = [res.correspondences(e).cpu() for e in range(B)]
    out = res.disparity[:, None].clone(), rows
    return (*out, res) if return_device_result else out


def transform_depth_pc_objects(depth: torch.Tensor, bg_depth: torch.Tensor, fg_masks, intrinsics: torch.Tensor, rot_angles, rot_axes,
                               translations, use_input_depth_normalization=False, return_device_result: bool = False):
    """One 'pc' edit of K disjoint objects of a square scene, object k moved by (``rot_angles[k]``, ``rot_axes[k]``,
    ``translations[k]``): ``transform_depth_pc_objects_batch`` with one edit.  Returns ``(edited disparity (1,1,S,S) fp32,
    correspondences (N,4) int64 CPU)`` like ``transform_depth_pc`` (plus the ``EditResult`` with ``return_device_result=True``)."""
    disparity, corrs, res = transform_depth_pc_objects_batch(depth, bg_depth, fg_masks, intrinsics, [rot_angles], [rot_axes],
                                                             [translations], use_input_depth_normalization, return_device_result=True)
    return (disparity, corrs[0], res) if return_device_result else (disparity, corrs[0])


def transform_depth_mesh(depth: torch.Tensor, bg_depth: torch.Tensor, fg_mask: torch.Tensor, intrinsics: torch.Tensor,
                         rot_angle: float = None, rot_axis: torch.Tensor = None, translation: torch.Tensor = None,
                         use_input_depth_normalization=False):
    """depth_transform.py:91-195 - opt-in mesh mode: triangulate both depth maps, move the foreground mesh, rasterise the
    scene (hard z-buffer, back faces culled, blur 1e-5) and read depth and source coordinates off the render layers.
    Correspondences are enumerated over TARGET pixels in raster order; no mask cleaning and no hole fill (as in the
    reference).  The rasteriser follows pytorch3d's published semantics; bit parity with pytorch3d is unpinned.  Runs as
    ``transform_depth_mesh_batch`` with one transform."""
    disparity, corrs = transform_depth_mesh_batch(depth, bg_depth, fg_mask, intrinsics, [rot_angle], [rot_axis], [translation],
                                                  use_input_depth_normalization)
    return disparity, corrs[0]


def transform_depth_mesh_batch(depth: torch.Tensor, bg_depth: torch.Tensor, fg_mask: torch.Tensor, intrinsics: torch.Tensor,
                               rot_angles, rot_axes, translations, use_input_depth_normalization=False):
    """``transform_depth_mesh`` for B transforms of one scene in one native call: ``transform_depth_mesh_scenes`` with one scene.

    Both meshes are built once; the background mesh is rasterised once and every edit's moved foreground faces are rasterised
    over a copy of its z-buffer, which gives the z-buffer of the joined mesh bit for bit.  ``rot_angles`` / ``rot_axes`` /
    ``translations`` hold one entry per edit (``None`` takes the defaults of the single call).  Returns ``(disparities
    (B,1,H,W) fp32 on depth.device, [correspondences (n_b,4) int64 CPU] * B)``; entry b equals bit for bit what the
    renderer reads off the joined mesh [background, foreground moved by transform b]."""
    B = _edit_count(rot_angles, rot_axes, translations)
    H, W = depth.shape[-2:]
    scene = [[_as_scene(t, H, W)] for t in (depth, bg_depth, fg_mask)]
    return transform_depth_mesh_scenes(*scene, intrinsics, [0] * B, rot_angles, rot_axes, translations, use_input_depth_normalization)


def transform_depth_mesh_scenes(depths: torch.Tensor, bg_depths: torch.Tensor, fg_masks: torch.Tensor, intrinsics: torch.Tensor,
                                scene_index, rot_angles, rot_axes, translations, use_input_depth_normalization=False):
    """``transform_depth_mesh`` for B edits over S scenes in one native call (``dh_edit_mesh_scenes``).  Arguments and result
    as ``transform_depth_pc_scenes``: edit b moves the foreground of scene ``scene_index[b]``, entry b equals bit for bit
    ``transform_depth_mesh_batch`` on its scene.  The meshes of each scene an edit uses are built once and its background is
    rasterised once; scenes without foreground give their edits the empty-mask result and are not sent to the kernels."""
    from .renderer import MeshRenderer, fov_scales
    depths, bg_depths, fg_masks, index, B = _scene_args(depths, bg_depths, fg_masks, scene_index, rot_angles, rot_axes, translations)
    H, W = depths.shape[-2:]
    present = _scene_masks_present(fg_masks, index)
    live = [b for b in range(B) if present[index[b]]]
    disparity, correspondences = [None] * B, [None] * B
    if live:
        _require_cuda(depths, "depths")
        lib = N.load()
        dev = depths.device
        f32, i32 = torch.float32, torch.int32
        scenes = sorted({index[b] for b in live})
        slot = {s: k for k, s in enumerate(scenes)}
        bg_v, bg_f, fg_v, fg_c, fg_f = [], [], [], [], []
        for s in scenes:
            background = depth_to_mesh(depth=bg_depths[s:s + 1], intrinsics=intrinsics)
            foreground = depth_to_mesh(depth=depths[s:s + 1], intrinsics=intrinsics, mask=fg_masks[s, 0] > 0.5)
            bg_v.append(background.verts.to(f32))
            bg_f.append(background.faces.to(i32))
            fg_v.append(foreground.verts.to(f32))
            fg_c.append(foreground.vert_attributes["color"].to(f32))
            fg_f.append(foreground.faces.to(i32))
        counts = [(C.c_int32 * len(scenes))(*[t.shape[0] for t in ts]) for ts in (bg_v, bg_f, fg_v, fg_f)]
        bg_verts, bg_faces, fg_verts, fg_colors, fg_faces = (torch.cat(ts).contiguous() for ts in (bg_v, bg_f, fg_v, fg_c, fg_f))
        n = len(live)
        table = (C.c_int32 * n)(*[slot[index[b]] for b in live])
        # the host values of the single call: the angle through an fp32 tensor, axis / translation as C floats
        angles, axes, shifts = [], [], []
        for b in live:
            a, ax, t = rot_angles[b], rot_axes[b], translations[b]
            angles.append(float(torch.tensor(0.0 if a is None else float(a), dtype=f32)))
            axes += [float(v) for v in (torch.tensor([0.0, 1.0, 0.0]) if ax is None else ax).detach().cpu().reshape(-1)[:3]]
            shifts += [float(v) for v in (torch.zeros(3) if t is None else t).detach().cpu().reshape(-1)[:3]]
        # the camera of the single call: Camera(intrinsics) (identity extrinsics) through MeshRenderer, blur 1e-5, back faces culled
        sx, sy = fov_scales(intrinsics[1, 1], H, W, MeshRenderer.z_near)
        R = (C.c_float * 9)(1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0)
        T = (C.c_float * 3)(0.0, 0.0, 0.0)
        target_z = torch.empty((n, H, W), dtype=f32, device=dev)
        corr = torch.empty((n, H * W, 4), dtype=torch.int64, device=dev)
        n_corr = torch.empty(n, dtype=i32, device=dev)
        host = ((C.c_float * n)(*angles), (C.c_float * (3 * n))(*axes), (C.c_float * (3 * n))(*shifts), H, W, R, T, sx, sy, 1e-5, 1, 1, 1,
                N.ptr(target_z), N.ptr(corr), N.ptr(n_corr), None)
        if len(scenes) == 1:        # one scene: dh_edit_mesh_batch, whose kernels are faster for it than the scene-table ones
            ws_bytes = int(lib.dh_edit_mesh_batch_workspace_bytes(n, counts[0][0], counts[2][0], H, W))
        else:
            ws_bytes = int(lib.dh_edit_mesh_scenes_workspace_bytes(len(scenes), *counts, n, table, H, W))
        if ws_bytes == 0:
            raise ValueError(f"mesh mode: unsupported sizes ({len(scenes)} scenes, {n} edits, {H}x{W}, "
                             f"{bg_verts.shape[0]} + {fg_verts.shape[0]} vertices)")
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        if len(scenes) == 1:
            N.check(lib.dh_edit_mesh_batch(N.ptr(bg_verts), counts[0][0], N.ptr(bg_faces), counts[1][0], N.ptr(fg_verts), N.ptr(fg_colors),
                                           counts[2][0], N.ptr(fg_faces), counts[3][0], n, *host, N.ptr(ws), ws_bytes,
                                           N.stream_handle(dev)), "dh_edit_mesh_batch")
        else:
            N.check(lib.dh_edit_mesh_scenes(len(scenes), N.ptr(bg_verts), N.ptr(bg_faces), counts[0], counts[1], N.ptr(fg_verts),
                                            N.ptr(fg_colors), N.ptr(fg_faces), counts[2], counts[3], n, table, *host, N.ptr(ws), ws_bytes,
                                            N.stream_handle(dev)), "dh_edit_mesh_scenes")
        rows_per_edit = n_corr.tolist()                                          # the one synchronisation
        rows = _rows_to_cpu(corr, rows_per_edit)
        bounds = (normalize_depth(1.0 / _gather_planes(depths, [index[b] for b in live]), return_bounds=True)[1]
                  if use_input_depth_normalization else None)
        disp = normalize_depth(1.0 / target_z[:, None], bounds=bounds)
        if len(live) == B:                        # every edit has a foreground: rows are already in edit order
            return disp, rows
        for e, b in enumerate(live):
            disparity[b] = disp[e]
            correspondences[b] = rows[e]
    _empty_mask_edits(depths, index, [b for b in range(B) if not present[index[b]]], use_input_depth_normalization, disparity,
                      correspondences)
    return torch.stack(disparity), correspondences


def transform_depth(depth: torch.Tensor, bg_depth: torch.Tensor, fg_mask: torch.Tensor, intrinsics: torch.Tensor,
                    rot_angle: float = None, rot_axis: torch.Tensor = None, translation: torch.Tensor = None,
                    use_input_depth_normalization=False, depth_transform_mode: str = "pc"):
    """depth_transform.py:73-89."""
    if depth_transform_mode == "mesh":
        return transform_depth_mesh(depth=depth, bg_depth=bg_depth, fg_mask=fg_mask, intrinsics=intrinsics,
                                    rot_angle=rot_angle, rot_axis=rot_axis, translation=translation,
                                    use_input_depth_normalization=use_input_depth_normalization)
    elif depth_transform_mode == "pc":
        return transform_depth_pc(depth=depth, bg_depth=bg_depth, fg_mask=fg_mask, intrinsics=intrinsics,
                                  rot_angle=rot_angle, rot_axis=rot_axis, translation=translation,
                                  use_input_depth_normalization=use_input_depth_normalization)
    else:
        raise ValueError(f"Unknown depth transform mode '{depth_transform_mode}'.")
