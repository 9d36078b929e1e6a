"""Host-side driver of the fused pc path: owns the device scratch of a batch of edits and enqueues
K1 -> K2 -> masks -> correspondences -> (Poisson fill) on the current CUDA stream.

One ``EditEngine`` per (device, B, H, W).  All buffers are torch-allocated once and reused; a batch of
edits costs one host synchronisation (reading the per-edit correspondence counts).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as N

MAX_OBJECTS = 16      # objects per multi-object edit (dh_edit_splat_objects)


def ellipse_rows(k: int) -> List[int]:
    """Rows of ``cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (k, k))`` as bit masks (bit j = column j).
    Restates OpenCV's ellipse rasterisation so the product does not need cv2; tests compare with cv2."""
    if k < 1 or k > 32:
        raise ValueError(f"structuring element size {k} outside [1, 32]")
    if k == 1:
        return [1]
    r = c = k // 2
    inv_r2 = 1.0 / (r * r) if r else 0.0
    rows = []
    for i in range(k):
        dy = i - r
        bits = 0
        if abs(dy) <= r:
            dx = int(np.rint(c * np.sqrt((r * r - dy * dy) * inv_r2)))
            j1, j2 = max(c - dx, 0), min(c + dx + 1, k)
            for j in range(j1, j2):
                bits |= 1 << j
        rows.append(bits)
    return rows


def make_rigid(rot_angle, rot_axis, translation) -> N.dh_rigid:
    """Host-side reduction of the user's transform, following depth_transform.py:497-500, :518-519, :241-243
    to the letter (NumPy fp32 axis normalisation, fp64 cos/sin of np.radians(angle))."""
    if isinstance(rot_angle, torch.Tensor):
        rot_angle = rot_angle.item()
    axis = np.asarray(rot_axis.detach().cpu().numpy() if isinstance(rot_axis, torch.Tensor) else rot_axis, dtype=np.float32)
    axis = axis / np.linalg.norm(axis)
    angle = np.radians(rot_angle)
    if isinstance(translation, torch.Tensor):
        t = [translation[i].item() for i in range(3)]
    else:
        t = [float(np.float32(v)) for v in translation]
    rg = N.dh_rigid()
    rg.axis[:] = [float(a) for a in axis.astype(np.float32)]
    rg.cos_t = float(np.cos(angle))
    rg.sin_t = float(np.sin(angle))
    rg.t[:] = t
    return rg


_GRID_CACHE: Dict[Tuple[int, int, str], Tuple[torch.Tensor, torch.Tensor]] = {}


def pixel_grid(H: int, W: int, device: torch.device) -> Tuple[torch.Tensor, torch.Tensor]:
    """x (W,) / y (H,) image-plane coordinates.  Computed by torch.linspace on the CPU - the very kernel the
    reference uses (depth_transform.py:621-628) - and uploaded once per (H, W, device)."""
    key = (H, W, str(device))
    if key not in _GRID_CACHE:
        nw = (W - 1) / (max(W, H) - 1)
        nh = (H - 1) / (max(W, H) - 1)
        xs = torch.linspace(-nw, nw, steps=W, dtype=torch.float32)
        ys = torch.linspace(-nh, nh, steps=H, dtype=torch.float32)
        _GRID_CACHE[key] = (xs.to(device), ys.to(device))
    return _GRID_CACHE[key]


@dataclass
class EditResult:
    """Device-side result of a batch of edits (views into the engine's buffers; valid until the next call)."""
    B: int
    H: int
    W: int
    n_fg: torch.Tensor            # (B,) int32
    n_corr: torch.Tensor          # (B,) int32
    centroid: torch.Tensor        # (B,3) fp32; (B,K,3) for a multi-object edit
    pix: torch.Tensor             # (B,2P) int32
    zkey: torch.Tensor            # (B,2P) int64 view of the uint64 keys
    fg_index: torch.Tensor        # (B,P) int32
    winner: torch.Tensor          # (B,P) int32 view of uint32 (0xFFFFFFFF -> -1)
    winner_src: torch.Tensor      # (B,P) int32
    depth_map: torch.Tensor       # (B,H,W) fp32
    target_mask: torch.Tensor     # (B,H,W) uint8
    target_bits: torch.Tensor     # (B,H,wpr) int32 (bit-packed)
    cleaned_bits: torch.Tensor    # (B,H,wpr) int32
    corr: torch.Tensor            # (B,P,4) int64
    disparity_raw: torch.Tensor   # (B,H,W) fp32  normalize_depth(1/depth_map)
    disparity: Optional[torch.Tensor]  # (B,H,W) fp32 Poisson-filled (None if not requested)
    points: Optional[torch.Tensor]     # (B,2P,3) fp64 (debug)

    def correspondences(self, e: int = 0) -> torch.Tensor:
        """(n_corr,4) int64 on the device, reference order."""
        return self.corr[e, : int(self.n_corr_host[e])]

    n_corr_host: Optional[np.ndarray] = None
    n_fg_host: Optional[np.ndarray] = None
    object_id: Optional[torch.Tensor] = None  # (B,P) uint8: object of foreground point j (multi-object edits only)


class EditEngine:
    """Scratch + launch sequence for B edits of H x W depth maps on one device."""

    def __init__(self, device: torch.device, B: int, H: int, W: int, keep_points: bool = False):
        if H < 2 or W < 2:
            raise RuntimeError(f"Expected depth to have at least 2 pixels in each dimension, got {H} x {W}.")
        self.lib = N.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise N.NativeLibraryError("EditEngine needs a CUDA device; there is no CPU path")
        self.B, self.H, self.W = B, H, W
        P = H * W
        self.P = P
        self.wpr = (W + 31) // 32
        dev = self.device
        i32, i64, f32, u8 = torch.int32, torch.int64, torch.float32, torch.uint8
        self.ws_bytes = int(self.lib.dh_edit_workspace_bytes(B, H, W))
        self.ws = torch.empty(self.ws_bytes, dtype=u8, device=dev)
        self.pix = torch.empty((B, 2 * P), dtype=i32, device=dev)
        self.zkey = torch.empty((B, 2 * P), dtype=i64, device=dev)
        self.fg_index = torch.empty((B, P), dtype=i32, device=dev)
        self.n_fg = torch.zeros((B,), dtype=i32, device=dev)
        self.n_corr = torch.zeros((B,), dtype=i32, device=dev)
        self.centroid = torch.empty((B, 3), dtype=f32, device=dev)
        self.zbuf = torch.empty((B, P), dtype=i64, device=dev)
        self.winner = torch.empty((B, P), dtype=i32, device=dev)
        self.winner_src = torch.empty((B, P), dtype=i32, device=dev)
        self.depth_map = torch.empty((B, H, W), dtype=f32, device=dev)
        self.target_mask = torch.empty((B, H, W), dtype=u8, device=dev)
        self.target_bits = torch.empty((B, H, self.wpr), dtype=i32, device=dev)
        self.cleaned_bits = torch.empty((B, H, self.wpr), dtype=i32, device=dev)
        self.tmp_bits = torch.empty((B, H, self.wpr), dtype=i32, device=dev)
        self.corr = torch.empty((B, P, 4), dtype=i64, device=dev)
        self.corr_ws = torch.empty((B * ((P + 1023) // 1024) + 64,), dtype=i32, device=dev)      # tile counts of dh_correspondences
        self.inv_minmax = torch.empty((B, 2), dtype=f32, device=dev)
        self.in_minmax = torch.empty((B, 2), dtype=f32, device=dev)
        self.disparity_raw = torch.empty((B, H, W), dtype=f32, device=dev)
        self.disparity = torch.empty((B, H, W), dtype=f32, device=dev)
        self.points = torch.empty((B, 2 * P, 3), dtype=torch.float64, device=dev) if keep_points else None
        self.poisson_ws_bytes = int(self.lib.dh_poisson_workspace_bytes(B, H, W))
        self.poisson_ws = torch.empty(self.poisson_ws_bytes, dtype=u8, device=dev)
        self.poisson_iters = torch.zeros((B,), dtype=i32, device=dev)
        # relative residual at which the CG hole fill stops (fp64).  The filled disparity is cast to fp32: from 1e-9 downwards the
        # result does not change any more (tests/fuzz/poisson_tolerance.py), 1e-11 keeps two orders of margin for ill-conditioned holes
        self.poisson_rel_tol = 1e-11
        self.n_pinned = torch.zeros((3, B), dtype=i32).pin_memory()
        # the transforms are uploaded from this (pageable, engine-owned) array: it outlives the call, so a CUDA graph that captured
        # the launch chain re-reads the transforms stored here at every replay
        self._rigids = (N.dh_rigid * B)()
        self.obj_ws = None                # scratch of multi-object edits (run_objects)
        self.xs, self.ys = pixel_grid(H, W, dev)
        S = max(H, W)
        # depth_transform.py:311-313: MORPH_ELLIPSE elements of size img_res//250 (open) and img_res//50 (close)
        self.open_k, self.close_k = max(S // 250, 1), max(S // 50, 1)
        self.open_rows = N.u32_array(ellipse_rows(self.open_k))
        self.close_rows = N.u32_array(ellipse_rows(self.close_k))

    def run(self, depth: torch.Tensor, bg_depth: torch.Tensor, fg_mask: torch.Tensor, intrinsics: torch.Tensor,
            rigids: Sequence[N.dh_rigid], use_input_depth_normalization: bool = False, poisson: bool = True,
            sync_counts: bool = True) -> EditResult:
        """depth / bg_depth / fg_mask: (B,H,W) fp32 contiguous on this device.  rigids: B host structs."""
        lib, B, H, W, P = self.lib, self.B, self.H, self.W, self.P
        if len(rigids) != B:
            raise ValueError(f"expected {B} rigid transforms, got {len(rigids)}")
        for name, t in (("depth", depth), ("bg_depth", bg_depth), ("fg_mask", fg_mask)):
            if tuple(t.shape) != (B, H, W):
                raise ValueError(f"{name} must have shape {(B, H, W)}, got {tuple(t.shape)}")
        st = N.stream_handle(self.device)
        cam = N.make_camera(intrinsics)
        rg = self._rigids
        for i, r in enumerate(rigids):
            rg[i] = r
        f32 = torch.float32
        # K1 + K2 (unproject, transform, project, exact (z, index) splat, depth map / target mask / winner sources / min-max)
        N.check(lib.dh_edit_splat(
            N.ptr(depth, f32, "depth"), N.ptr(bg_depth, f32, "bg_depth"), N.ptr(fg_mask, f32, "fg_mask"), B, H, W,
            C.byref(cam), rg, N.ptr(self.xs), N.ptr(self.ys), N.ptr(self.pix), N.ptr(self.zkey), N.ptr(self.fg_index),
            N.ptr(self.n_fg), N.ptr(self.centroid), N.ptr(self.points) if self.points is not None else None,
            N.ptr(self.zbuf), N.ptr(self.winner), N.ptr(self.depth_map), N.ptr(self.target_mask), N.ptr(self.target_bits),
            N.ptr(self.winner_src), N.ptr(self.inv_minmax), N.ptr(self.ws), self.ws_bytes, st), "dh_edit_splat")
        return self._finish(depth, self.centroid, None, use_input_depth_normalization, poisson, sync_counts)

    def run_objects(self, depth: torch.Tensor, bg_depth: torch.Tensor, fg_mask: torch.Tensor, labels: torch.Tensor, K: int,
                    intrinsics: torch.Tensor, rigids: Sequence[N.dh_rigid], use_input_depth_normalization: bool = False,
                    poisson: bool = True, sync_counts: bool = True) -> EditResult:
        """``run`` for edits of K disjoint objects (``dh_edit_splat_objects``).  fg_mask (B,H,W) fp32 is the union of the objects,
        labels (B,H,W) uint8 holds k + 1 on the pixels of object k (0 elsewhere), rigids B*K host structs, edit-major.  The
        result's ``centroid`` is (B,K,3) and ``object_id`` (B,P) uint8 gives the object of each foreground point."""
        lib, B, H, W, P = self.lib, self.B, self.H, self.W, self.P
        if not 1 <= K <= MAX_OBJECTS:
            raise ValueError(f"between 1 and {MAX_OBJECTS} objects per edit are supported, got {K}")
        if len(rigids) != B * K:
            raise ValueError(f"expected {B * K} rigid transforms ({B} edits of {K} objects), got {len(rigids)}")
        for name, t in (("depth", depth), ("bg_depth", bg_depth), ("fg_mask", fg_mask), ("labels", labels)):
            if tuple(t.shape) != (B, H, W):
                raise ValueError(f"{name} must have shape {(B, H, W)}, got {tuple(t.shape)}")
        if self.obj_ws is None:           # allocated on first use: the single-object path never needs it
            self.obj_ws_bytes = int(lib.dh_edit_objects_workspace_bytes(B, H, W))
            self.obj_ws = torch.empty(self.obj_ws_bytes, dtype=torch.uint8, device=self.device)
            self.object_id = torch.empty((B, P), dtype=torch.uint8, device=self.device)
            self.obj_centroid = torch.empty((B * MAX_OBJECTS * 3,), dtype=torch.float32, device=self.device)
            self._obj_rigids = (N.dh_rigid * (B * MAX_OBJECTS))()
        st = N.stream_handle(self.device)
        cam = N.make_camera(intrinsics)
        rg = self._obj_rigids
        for i, r in enumerate(rigids):
            rg[i] = r
        f32 = torch.float32
        N.check(lib.dh_edit_splat_objects(
            N.ptr(depth, f32, "depth"), N.ptr(bg_depth, f32, "bg_depth"), N.ptr(fg_mask, f32, "fg_mask"),
            N.ptr(labels, torch.uint8, "labels"), B, K, H, W, C.byref(cam), rg, N.ptr(self.xs), N.ptr(self.ys), N.ptr(self.pix),
            N.ptr(self.zkey), N.ptr(self.fg_index), N.ptr(self.object_id), N.ptr(self.n_fg), N.ptr(self.obj_centroid),
            N.ptr(self.points) if self.points is not None else None, N.ptr(self.zbuf), N.ptr(self.winner), N.ptr(self.depth_map),
            N.ptr(self.target_mask), N.ptr(self.target_bits), N.ptr(self.winner_src), N.ptr(self.inv_minmax), N.ptr(self.obj_ws),
            self.obj_ws_bytes, st), "dh_edit_splat_objects")
        centroid = self.obj_centroid[: B * K * 3].view(B, K, 3)
        return self._finish(depth, centroid, self.object_id, use_input_depth_normalization, poisson, sync_counts)

    def _finish(self, depth: torch.Tensor, centroid: torch.Tensor, object_id: Optional[torch.Tensor],
                use_input_depth_normalization: bool, poisson: bool, sync_counts: bool) -> EditResult:
        """Everything after the splat: mask cleaning, correspondences, disparity, hole fill, and the count read-back."""
        lib, B, H, W, P = self.lib, self.B, self.H, self.W, self.P
        st = N.stream_handle(self.device)
        N.check(lib.dh_mask_clean(N.ptr(self.target_bits), N.ptr(self.cleaned_bits), N.ptr(self.tmp_bits), B, H, W,
                                  self.close_rows, self.close_k, self.open_rows, self.open_k, st), "dh_mask_clean")
        N.check(lib.dh_correspondences(N.ptr(self.pix), N.ptr(self.winner), N.ptr(self.fg_index), N.ptr(self.n_fg),
                                       N.ptr(self.cleaned_bits), B, H, W, 2 * P, N.ptr(self.corr), N.ptr(self.n_corr),
                                       N.ptr(self.corr_ws), self.corr_ws.numel() * 4, st), "dh_correspondences")
        bounds = self.inv_minmax
        if use_input_depth_normalization:
            N.check(lib.dh_inv_minmax(N.ptr(depth), B, P, N.ptr(self.in_minmax), st), "dh_inv_minmax")
            bounds = self.in_minmax
        N.check(lib.dh_disparity(N.ptr(self.depth_map), B, P, N.ptr(bounds), N.ptr(self.disparity_raw), st), "dh_disparity")
        disparity = None
        if poisson:
            N.check(lib.dh_poisson_fill(N.ptr(self.disparity_raw), N.ptr(self.cleaned_bits), N.ptr(self.target_bits), B, H, W,
                                        N.ptr(self.disparity), 0, self.poisson_rel_tol, N.ptr(self.poisson_iters),
                                        N.ptr(self.poisson_ws), self.poisson_ws_bytes, st), "dh_poisson_fill")
            disparity = self.disparity
        res = EditResult(B=B, H=H, W=W, n_fg=self.n_fg, n_corr=self.n_corr, centroid=centroid, pix=self.pix,
                         zkey=self.zkey, fg_index=self.fg_index, winner=self.winner, winner_src=self.winner_src,
                         depth_map=self.depth_map, target_mask=self.target_mask, target_bits=self.target_bits,
                         cleaned_bits=self.cleaned_bits, corr=self.corr, disparity_raw=self.disparity_raw,
                         disparity=disparity, points=self.points, object_id=object_id)
        if sync_counts:
            self.n_pinned[0].copy_(self.n_corr, non_blocking=True)
            self.n_pinned[1].copy_(self.n_fg, non_blocking=True)
            if poisson:
                self.n_pinned[2].copy_(self.poisson_iters, non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            res.n_corr_host = self.n_pinned[0].numpy().copy()
            res.n_fg_host = self.n_pinned[1].numpy().copy()
            if poisson:
                from .depth_transform import warn_if_not_converged
                warn_if_not_converged(self.n_pinned[2], "hole fill of the edited disparity")
        return res

    def unpack_bits(self, bits: torch.Tensor) -> torch.Tensor:
        """(B,H,wpr) packed -> (B,H,W) uint8."""
        out = torch.empty((self.B, self.H, self.wpr * 32), dtype=torch.uint8, device=self.device)
        N.check(self.lib.dh_unpack_bits(N.ptr(bits), bits.numel(), N.ptr(out), N.stream_handle(self.device)), "dh_unpack_bits")
        return out[:, :, : self.W]


_ENGINES: Dict[Tuple[str, int, int, int, bool], EditEngine] = {}


def get_engine(device: torch.device, B: int, H: int, W: int, keep_points: bool = False) -> EditEngine:
    key = (str(torch.device(device)), B, H, W, keep_points)
    if key not in _ENGINES:
        _ENGINES[key] = EditEngine(device, B, H, W, keep_points)
    return _ENGINES[key]
