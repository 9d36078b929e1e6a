"""NumPy oracle of multi-object 'pc' edits: the foreground is K disjoint object masks of one square scene, each object moved by
its own rigid transform about its own centroid.  There is no reference for K > 1; this is the natural generalisation of
depth_transform.py:198-363 (oracle/dh_oracle.py ``transform_depth_pc``), built from the same primitives:

- points 0..P-1 are the background pixels, points P..P+n-1 the pixels of the union of the masks in source raster order;
- point P + j belongs to the object whose mask holds its pixel and is rotated about the fp32 sequential centroid of that
  object's points (raster order, ``np.mean`` over the object alone), then translated, in ``rigid_transform_fg``'s order;
- z-buffer, ties, target mask ("the winner is a foreground point of any object"), correspondences, morphology, disparity and
  Poisson fill are those of ``transform_depth_pc``.

With one mask every intermediate equals ``transform_depth_pc``."""
from __future__ import annotations

import os
import sys
from typing import Dict, Sequence

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import dh_oracle as O          # noqa: E402

f32, f64 = np.float32, np.float64
MAX_OBJECTS = 16


def object_masks(fg_masks) -> np.ndarray:
    """(K,1,S,S), (K,S,S) or a sequence of K (1,1,S,S) / (S,S) masks -> (K,S,S) bool (non-zero = in the object)."""
    if isinstance(fg_masks, np.ndarray):
        m = fg_masks
        if m.ndim == 4:
            m = m[:, 0]
    else:
        m = np.stack([np.asarray(x).reshape(np.asarray(x).shape[-2:]) for x in fg_masks])
    return np.asarray(m) != 0


def transform_depth_pc_objects(depth: np.ndarray, bg_depth: np.ndarray, fg_masks, K: np.ndarray, rot_angles: Sequence[float],
                               rot_axes: Sequence[Sequence[float]], translations: Sequence[Sequence[float]],
                               use_input_depth_normalization: bool = False, loop: bool = False,
                               poisson: bool = True) -> Dict[str, np.ndarray]:
    """``transform_depth_pc`` with K object masks and K transforms (``rot_angles[k]`` etc. move object k).  Returns the same
    intermediates, with ``centroid`` (K,3) fp32 (NaN for an object without pixels) and ``object`` (n,) int64: the object of each
    foreground point."""
    depth = np.asarray(depth, dtype=f32)
    bg_depth = np.asarray(bg_depth, dtype=f32)
    masks = object_masks(fg_masks)
    n_obj = masks.shape[0]
    if not 1 <= n_obj <= MAX_OBJECTS:
        raise ValueError(f"between 1 and {MAX_OBJECTS} object masks are supported, got {n_obj}")
    if not len(rot_angles) == len(rot_axes) == len(translations) == n_obj:
        raise ValueError(f"one transform per object ({n_obj}) expected, got {len(rot_angles)}, {len(rot_axes)}, {len(translations)}")
    if (masks.sum(0) > 1).any():
        raise ValueError("the object masks overlap")
    S = masks.shape[-1]
    if masks.shape[1] != masks.shape[2]:
        raise RuntimeError(f"Expected fg_mask to be square, got shape {masks.shape[1]} x {masks.shape[2]}.")
    mask = masks.any(0)
    out: Dict[str, np.ndarray] = {}
    with np.errstate(all="ignore"):
        bounds = None
        if use_input_depth_normalization:
            d = (f32(1.0) / depth).astype(f32)
            bounds = (d.min(), d.max())
        if not mask.any():
            out["correspondences"] = np.zeros((0, 4), np.int64)
            out["disparity"] = O.normalize_depth((f32(1.0) / depth).astype(f32), bounds)
            return out
        bg_pts = O.depth_to_world_coords(bg_depth, K).reshape(-1, 3)
        pts = O.depth_to_world_coords(depth, K).reshape(-1, 3)
        F = np.nonzero(mask.reshape(-1))[0]
        obj = np.argmax(masks.reshape(n_obj, -1)[:, F], axis=0).astype(np.int64)
        r = np.empty((F.shape[0], 3), dtype=f64)
        cen = np.full((n_obj, 3), np.nan, dtype=f32)
        for k in range(n_obj):
            sel = obj == k
            if sel.any():
                r[sel], cen[k] = O.rigid_transform_fg(pts[F[sel]], rot_axes[k], rot_angles[k], translations[k])
        points = np.vstack([bg_pts.astype(f64), r])
        P = S * S
        point_mask = np.arange(points.shape[0]) >= P
        depth_map, target_mask, tx, ty, visible, winner = O.points_to_depth(points, K, (S, S), point_mask, loop=loop)
        u, v = O.project_points(points, K, (S, S))
        disparity_raw = O.normalize_depth((f32(1.0) / depth_map).astype(f32), bounds)
    vis_fg = visible[P:]
    src = F[vis_fg]
    cleaned = O.clean_target_mask(target_mask, S)
    keep = cleaned[ty, tx]
    corr = np.stack([src % S, src // S, tx, ty], axis=-1)[keep].astype(np.int64)
    inpaint = cleaned ^ target_mask
    out.update(points=points, centroid=cen, object=obj, pix=v * S + u, winner=winner, depth_map=depth_map,
               target_mask=target_mask, visible=visible, cleaned=cleaned, correspondences=corr,
               disparity_raw=disparity_raw, inpaint_mask=inpaint, fg_index=F)
    if poisson:
        out["disparity"] = O.poisson_solve(disparity_raw, inpaint.astype(np.uint8)).astype(f32)
    return out


def sector_masks(mask: np.ndarray, n: int, cx: float = None, cy: float = None) -> np.ndarray:
    """Split a (S,S) mask into n angular sectors about (cx, cy) (default: the mask's pixel centre) -> (n,S,S) float32."""
    m = np.asarray(mask) != 0
    ys, xs = np.nonzero(m)
    if cx is None:
        cx, cy = (xs.mean(), ys.mean()) if len(xs) else (0.0, 0.0)
    yy, xx = np.mgrid[0:m.shape[0], 0:m.shape[1]]
    ang = (np.arctan2(yy - cy, xx - cx) + np.pi) / (2 * np.pi)
    sector = np.minimum((ang * n).astype(np.int64), n - 1)
    return np.stack([(m & (sector == k)).astype(np.float32) for k in range(n)])
