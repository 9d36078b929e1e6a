"""TEST INFRASTRUCTURE ONLY - CPU restatement (NumPy) of the reference's activation-lifting / 3D-warp path.

This module is the *oracle*: an independent, resolution-generic restatement of the arithmetic the
reference executes on its default ``'pc'`` path, written from the closed forms in SURVEY.md
Appendix A.  It is pinned against the real reference by ``oracle/make_golden.py`` (golden vectors
under ``tests/golden/``) and by ``tests/test_oracle_vs_reference.py`` (runs when ``/root/reference``
is present).  It must never be imported by the product package ``diffusionhandles_b200``.

Reference lines restated here (all under ``/root/reference/diffhandles``):

* ``get_depth_intrinsics``            guided_stable_diffuser.py:129-153
* ``depth_to_world_coords``           depth_transform.py:589-641
* ``transform_point_cloud``           depth_transform.py:461-533   (``512`` generalised to S)
* point-set assembly                  depth_transform.py:255-274
* ``points_to_depth``                 depth_transform.py:643-747   (z-buffer loop :697-712)
* masks / correspondences             depth_transform.py:283-343
* inpaint mask + ``poisson_solve``    depth_transform.py:346-363, :535-587
* ``normalize_depth``                 depth_transform.py:15-28
* ``process_correspondences``         guided_stable_diffuser.py:490-584
* losses                              losses.py:4-84
* guidance weight schedule            guided_stable_diffuser.py:336-373, :622-665
* latent update, CFG, DDIM update     guided_stable_diffuser.py:434, :470-474 (scheduler arithmetic: diffusers 0.23, absent:
                                      parity unpinned, see the section header)

Numerics contract (SURVEY.md finding 8): the oracle reproduces the reference *as executed under this
image* (NumPy >= 2 promotion rules: ``float32_array * np.float64 scalar -> float64``).
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Sequence, Tuple

import numpy as np

f32 = np.float32
f64 = np.float64


# --------------------------------------------------------------------------------------------
# intrinsics / grids
# --------------------------------------------------------------------------------------------
def get_depth_intrinsics() -> np.ndarray:
    """guided_stable_diffuser.py:129-153 - pinhole K, 55 degree FoV, principal point 0, fp32."""
    f = 1.0 / np.tan(0.5 * 55.0 * (np.pi / 180.0))
    return np.array([[f, 0, 0], [0, f, 0], [0, 0, 1]], dtype=f32)


def linspace_f32(start: float, end: float, steps: int) -> np.ndarray:
    """``torch.linspace(start, end, steps, dtype=float32)`` on CPU (depth_transform.py:623-628).

    torch's CPU kernel is symmetric with ONE rounding per element: ``step = fl32((end-start)/(steps-1))``;
    ``x_i = fma(step, i, start)`` for ``i < steps//2`` and ``x_i = fma(-step, steps-1-i, end)`` otherwise.
    The fma is emulated in fp64 (a 24-bit x 20-bit product and one add are exact there for the sizes
    used, so the final cast is the single rounding).
    """
    s, e = f32(start), f32(end)
    if steps == 1:
        return np.array([s], dtype=f32)
    step = f32((e - s) / f32(steps - 1))
    i = np.arange(steps, dtype=np.int64)
    half = steps // 2
    lo = f64(s) + f64(step) * i.astype(f64)
    hi = f64(e) - f64(step) * (steps - 1 - i).astype(f64)
    return np.where(i < half, lo, hi).astype(f32)


def pixel_grid(H: int, W: int) -> Tuple[np.ndarray, np.ndarray]:
    """x (W,) and y (H,) image-plane coordinates, depth_transform.py:621-628."""
    nw = (W - 1) / (max(W, H) - 1)
    nh = (H - 1) / (max(W, H) - 1)
    return linspace_f32(-nw, nw, W), linspace_f32(-nh, nh, H)


def inv3x3_f32(K: np.ndarray) -> np.ndarray:
    """fp32 inverse of the intrinsics.  For the contract class (diagonal K, zero principal point) the
    inverse is ``diag(1/k00, 1/k11, 1/k22)`` with one fp32 divide per entry, which is what LAPACK's
    getrf/getri produce for a diagonal matrix (SURVEY.md A.1)."""
    K = np.asarray(K, dtype=f32)
    off = K.copy()
    np.fill_diagonal(off, 0)
    if not np.any(off):
        return np.diag((f32(1.0) / np.diag(K)).astype(f32)).astype(f32)
    return np.linalg.inv(K.astype(f64)).astype(f32)  # outside the bit-exact contract


# --------------------------------------------------------------------------------------------
# A.1 unprojection
# --------------------------------------------------------------------------------------------
def depth_to_world_coords(depth: np.ndarray, K: np.ndarray) -> np.ndarray:
    """depth (H,W) fp32 -> (H,W,3) fp32 world points (identity extrinsics), depth_transform.py:589-641.

    ``points = M @ ((D * Kinv) @ [x, y, 1])`` with diagonal K: X = -fl(fl(d*kx)*x), Y = -fl(fl(d*ky)*y),
    Z = fl(fl(d*kz)*1).
    """
    depth = np.asarray(depth, dtype=f32)
    H, W = depth.shape
    if H < 2 or W < 2:
        raise RuntimeError(f"Expected depth to have at least 2 pixels in each dimension, got {H} x {W}.")
    Kinv = inv3x3_f32(K)
    xs, ys = pixel_grid(H, W)
    if Kinv[0, 1] == 0 and Kinv[0, 2] == 0 and Kinv[1, 0] == 0 and Kinv[1, 2] == 0 and Kinv[2, 0] == 0 and Kinv[2, 1] == 0:
        X = -((depth * Kinv[0, 0]).astype(f32) * xs[None, :]).astype(f32)
        Y = -((depth * Kinv[1, 1]).astype(f32) * ys[:, None]).astype(f32)
        Z = (depth * Kinv[2, 2]).astype(f32)
    else:  # general K: left-to-right fp32 accumulation (not a bit-exact contract, SURVEY.md A.1)
        DK = depth[..., None, None] * Kinv[None, None]
        one = np.ones_like(depth)
        coord = np.stack([np.broadcast_to(xs[None, :], depth.shape), np.broadcast_to(ys[:, None], depth.shape), one], -1)
        p = ((DK[..., 0] * coord[..., 0:1]).astype(f32) + (DK[..., 1] * coord[..., 1:2]).astype(f32)).astype(f32)
        p = (p + (DK[..., 2] * coord[..., 2:3]).astype(f32)).astype(f32)
        X, Y, Z = -p[..., 0], -p[..., 1], p[..., 2]
    return np.stack([X, Y, Z], axis=-1).astype(f32)


# --------------------------------------------------------------------------------------------
# A.2 rigid transform of the foreground points
# --------------------------------------------------------------------------------------------
def sequential_sum_f32(v: np.ndarray) -> np.ndarray:
    """Strictly sequential fp32 sum over axis 0 (what ``np.mean(points[mask], axis=0)`` does for an
    (M,3) C-contiguous fp32 array: the reduction axis is the outer loop)."""
    return np.cumsum(v, axis=0, dtype=f32)[-1] if len(v) else np.zeros(v.shape[1:], f32)


def normalize_axis(axis: Sequence[float]) -> np.ndarray:
    """``axis / np.linalg.norm(axis)`` in fp32 (depth_transform.py:500)."""
    a = np.asarray(axis, dtype=f32)
    return (a / np.linalg.norm(a)).astype(f32)


def rigid_transform_fg(p: np.ndarray, axis: Sequence[float], angle_degrees: float,
                       t: Sequence[float], centroid: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray]:
    """Rodrigues rotation about the centroid + translation for the N_fg masked points (raster order).

    p (N_fg,3) fp32 -> (N_fg,3) fp64, centroid (3,) fp32.  depth_transform.py:492-531, SURVEY.md A.2/A.9.
    With ``centroid`` given, the points are rotated about it instead of about their own centroid.
    """
    p = np.asarray(p, dtype=f32)
    n = p.shape[0]
    a = normalize_axis(axis)
    angle = np.radians(angle_degrees)
    c, s = np.cos(angle), np.sin(angle)                     # fp64 scalars
    cen = (sequential_sum_f32(p) / f32(n)).astype(f32) if centroid is None else np.asarray(centroid, f32)
    q = (p - cen).astype(f32)
    cr = np.stack([
        ((a[1] * q[:, 2]).astype(f32) - (a[2] * q[:, 1]).astype(f32)).astype(f32),
        ((a[2] * q[:, 0]).astype(f32) - (a[0] * q[:, 2]).astype(f32)).astype(f32),
        ((a[0] * q[:, 1]).astype(f32) - (a[1] * q[:, 0]).astype(f32)).astype(f32)], axis=-1)
    # dot32: fma(q2,a2, fma(q0,a0, q1*a1)); exact (order independent) for a single-non-zero axis (A.2 caveat)
    d = (q[:, 1].astype(f64) * f64(a[1])).astype(f32)
    d = (q[:, 0].astype(f64) * f64(a[0]) + d.astype(f64)).astype(f32)
    d = (q[:, 2].astype(f64) * f64(a[2]) + d.astype(f64)).astype(f32)
    t3 = (a[None, :] * d[:, None]).astype(f32)
    r = (q.astype(f64) * c + cr.astype(f64) * s) + t3.astype(f64) * (1 - c)
    r = (r + cen.astype(f64)) + np.array([t[0], t[1], t[2]], dtype=f64)
    return r, cen


def transform_point_cloud(points: np.ndarray, axis, angle_degrees: float, x: float, y: float, z: float, mask: np.ndarray):
    """depth_transform.py:461-533 with the hard-coded 512 generalised: rotates ALL points about the fp32 sequential
    centroid of the masked ones.  Returns ((S,S,3) fp64, (S*S,) bool)."""
    points = np.asarray(points, dtype=f32)
    m = np.asarray(mask).astype(bool)
    flat = points.reshape(-1, 3)
    cen = (sequential_sum_f32(flat[m.reshape(-1)]) / f32(int(m.sum()))).astype(f32)
    r, _ = rigid_transform_fg(flat, axis, angle_degrees, (x, y, z), centroid=cen)
    return r.reshape(points.shape), m.reshape(-1)


# --------------------------------------------------------------------------------------------
# A.4 projection, A.5 z-buffer
# --------------------------------------------------------------------------------------------
def project_points(points: np.ndarray, K: np.ndarray, output_size: Tuple[int, int]) -> Tuple[np.ndarray, np.ndarray]:
    """points (N,3) fp64 (pytorch3d axes) -> integer pixel coordinates u (col), v (row); depth_transform.py:666-687.
    Clip first, then round-half-even."""
    H, W = output_size
    K = np.asarray(K, dtype=f32).astype(f64)
    P = np.asarray(points, dtype=f64)
    px, py, pz = -P[:, 0], -P[:, 1], P[:, 2]
    with np.errstate(all="ignore"):
        if K[0, 1] == 0 and K[0, 2] == 0 and K[1, 0] == 0 and K[1, 2] == 0 and K[2, 0] == 0 and K[2, 1] == 0:
            projx, projy, projz = K[0, 0] * px, K[1, 1] * py, K[2, 2] * pz
        else:
            projx = K[0, 0] * px + K[0, 1] * py + K[0, 2] * pz
            projy = K[1, 0] * px + K[1, 1] * py + K[1, 2] * pz
            projz = K[2, 0] * px + K[2, 1] * py + K[2, 2] * pz
        u = projx / projz
        v = projy / projz
        m = max(H, W) - 1
        u = (u * 0.5 + 0.5) * m
        v = (v * 0.5 + 0.5) * m
        u = np.rint(np.clip(u, 0, W - 1)).astype(np.int64)
        v = np.rint(np.clip(v, 0, H - 1)).astype(np.int64)
    return u, v


def zbuffer_closed_form(z: np.ndarray, pix: np.ndarray, n_pix: int) -> np.ndarray:
    """winner[q] = argmin over {i: pix_i = q} of (z_i, i) (lexicographic), -1 for empty pixels.
    Closed form of the strict-``<`` sequential loop at depth_transform.py:697-712 (SURVEY.md A.5)."""
    z = np.asarray(z, dtype=f64)
    idx = np.arange(z.shape[0], dtype=np.int64)
    ok = ~np.isnan(z)
    order = np.lexsort((idx[ok], z[ok], pix[ok]))
    sp = pix[ok][order]
    first = np.ones(sp.shape[0], dtype=bool)
    first[1:] = sp[1:] != sp[:-1]
    winner = np.full(n_pix, -1, dtype=np.int64)
    winner[sp[first]] = idx[ok][order][first]
    return winner


def zbuffer_loop(z: np.ndarray, pix: np.ndarray, n_pix: int) -> np.ndarray:
    """Literal sequential port of the reference loop (strict ``<`` in index order).  Slow; used to pin
    the closed form and as the honest CPU baseline of the splat."""
    depth = np.full(n_pix, np.inf)
    winner = np.full(n_pix, -1, dtype=np.int64)
    zl, pl = z.tolist(), pix.tolist()
    for i in range(len(zl)):
        q = pl[i]
        if zl[i] < depth[q]:
            depth[q] = zl[i]
            winner[q] = i
    return winner


def points_to_depth(points: np.ndarray, K: np.ndarray, output_size: Tuple[int, int],
                    point_mask: Optional[np.ndarray] = None, loop: bool = False):
    """Restatement of depth_transform.py:643-747 (identity extrinsics).

    Returns ``(depth_map (H,W) fp32 [+inf = empty], depth_mask (H,W) bool, u[visible], v[visible],
    visible (N,) bool, winner (H*W,) int64)``.
    """
    H, W = output_size
    points = np.asarray(points, dtype=f64)
    N = points.shape[0]
    if point_mask is None:
        point_mask = np.zeros(N, dtype=np.uint8)
    pm = np.asarray(point_mask).astype(bool)
    u, v = project_points(points, K, output_size)
    pix = v * W + u
    z = points[:, 2] + 0.0
    winner = (zbuffer_loop if loop else zbuffer_closed_form)(z, pix, H * W)
    has = winner >= 0
    depth_map = np.full(H * W, np.inf, dtype=f64)
    depth_map[has] = z[winner[has]]
    depth_mask = np.zeros(H * W, dtype=bool)
    depth_mask[has] = pm[winner[has]]
    visible = np.zeros(N, dtype=bool)
    visible[winner[has]] = True
    visible &= pm
    return (depth_map.astype(f32).reshape(H, W), depth_mask.reshape(H, W), u[visible], v[visible], visible, winner)


# --------------------------------------------------------------------------------------------
# A.6 masks, morphology, correspondences
# --------------------------------------------------------------------------------------------
def ellipse_element(k: int) -> np.ndarray:
    """``cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (k, k))`` restated (OpenCV morph.dispatch.cpp):
    r = k//2, c = k//2; row i spans [c-dx, c+dx] with dx = round(c*sqrt((r*r-dy*dy)/r^2)), dy = i-r."""
    if k <= 0:
        raise ValueError("structuring element size must be positive")
    if k == 1:
        return np.ones((1, 1), np.uint8)
    r, c = k // 2, k // 2
    inv_r2 = 1.0 / (r * r) if r else 0.0
    el = np.zeros((k, k), np.uint8)
    for i in range(k):
        dy = i - r
        if abs(dy) <= r:
            dx = int(np.rint(c * math.sqrt((r * r - dy * dy) * inv_r2)))
            j1, j2 = max(c - dx, 0), min(c + dx + 1, k)
            el[i, j1:j2] = 1
    return el


def _morph(img: np.ndarray, el: np.ndarray, dilate: bool) -> np.ndarray:
    """Binary erode/dilate with OpenCV semantics: anchor = (k//2, k//2),
    ``dst(y,x) = op over el(i,j)!=0 of src(y+i-ay, x+j-ax)``; out-of-image samples do not contribute."""
    img = np.asarray(img).astype(bool)
    H, W = img.shape
    kh, kw = el.shape
    ay, ax = kh // 2, kw // 2
    out = np.zeros((H, W), bool) if dilate else np.ones((H, W), bool)
    for i in range(kh):
        for j in range(kw):
            if not el[i, j]:
                continue
            dy, dx = i - ay, j - ax
            ys0, ys1 = max(0, -dy), min(H, H - dy)
            xs0, xs1 = max(0, -dx), min(W, W - dx)
            if ys0 >= ys1 or xs0 >= xs1:
                continue
            src = img[ys0 + dy:ys1 + dy, xs0 + dx:xs1 + dx]
            if dilate:
                out[ys0:ys1, xs0:xs1] |= src
            else:
                out[ys0:ys1, xs0:xs1] &= src
    return out


def morph_dilate(img, el):
    return _morph(img, el, True)


def morph_erode(img, el):
    return _morph(img, el, False)


def clean_target_mask(target_mask: np.ndarray, img_res: int,
                      close_el: Optional[np.ndarray] = None, open_el: Optional[np.ndarray] = None) -> np.ndarray:
    """OPEN_{S//250}(CLOSE_{S//50}(mask)) with MORPH_ELLIPSE elements, depth_transform.py:308-321.
    For S < 250 (S < 50) the reference's element size would be 0, which OpenCV rejects; the reference itself
    only runs at S = 512.  Sizes are clamped to >= 1 (a 1x1 element is the identity) for those resolutions."""
    if close_el is None:
        close_el = ellipse_element(max(img_res // 50, 1))
    if open_el is None:
        open_el = ellipse_element(max(img_res // 250, 1))
    m = morph_erode(morph_dilate(target_mask, close_el), close_el)
    m = morph_dilate(morph_erode(m, open_el), open_el)
    return m


def normalize_depth(x: np.ndarray, bounds=None) -> np.ndarray:
    """255*(x-min)/(max-min) in fp32, depth_transform.py:15-28 (one image)."""
    x = np.asarray(x, dtype=f32)
    if bounds is None:
        mn, mx = x.min(), x.max()
    else:
        mn, mx = f32(bounds[0]), f32(bounds[1])
    with np.errstate(all="ignore"):
        return ((f32(255) * (x - mn).astype(f32)).astype(f32) / f32(mx - mn)).astype(f32)


def poisson_solve(image: np.ndarray, mask: np.ndarray) -> np.ndarray:
    """Masked 5-point Poisson fill, depth_transform.py:535-587 (vectorised assembly, same SuperLU solve).
    Image-border neighbours are simply absent (diagonal stays 4)."""
    import scipy.sparse
    import scipy.sparse.linalg
    image = np.asarray(image)
    mask = np.asarray(mask).astype(bool)
    ys, xs = np.where(mask)
    n = len(ys)
    out = image.copy()
    if n == 0:
        return out
    H, W = image.shape
    index = -np.ones((H, W), dtype=np.int64)
    index[ys, xs] = np.arange(n)
    rows, cols, vals = [np.arange(n)], [np.arange(n)], [np.full(n, 4.0)]
    b = np.zeros(n)
    for dy, dx in ((-1, 0), (1, 0), (0, -1), (0, 1)):
        ny, nx = ys + dy, xs + dx
        inside = (ny >= 0) & (ny < H) & (nx >= 0) & (nx < W)
        nyc, nxc = np.clip(ny, 0, H - 1), np.clip(nx, 0, W - 1)
        unk = inside & mask[nyc, nxc]
        known = inside & ~mask[nyc, nxc]
        rows.append(np.nonzero(unk)[0]); cols.append(index[nyc[unk], nxc[unk]]); vals.append(np.full(unk.sum(), -1.0))
        b[known] += image[nyc[known], nxc[known]]
    A = scipy.sparse.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n))
    sol = scipy.sparse.linalg.spsolve(A, b)
    out[ys, xs] = sol
    return out


def solve_laplacian_depth(fg_depth: np.ndarray, bg_depth: np.ndarray, mask: np.ndarray) -> np.ndarray:
    """utils.py:49-102: Poisson fill of ``fg_depth`` inside ``mask`` whose source term is the Laplacian of ``bg_depth``
    (scipy.ndimage.convolve with the 5-point kernel, zero padding, result in the input dtype)."""
    import scipy.ndimage
    import scipy.sparse
    import scipy.sparse.linalg
    fg = np.asarray(fg_depth)
    mask = np.asarray(mask).astype(bool)
    ys, xs = np.where(mask)
    n = len(ys)
    out = fg.copy()
    if n == 0:
        return out
    H, W = fg.shape
    lap = scipy.ndimage.convolve(np.asarray(bg_depth), np.array([[0, 1, 0], [1, -4, 1], [0, 1, 0]]), mode="constant")
    index = -np.ones((H, W), dtype=np.int64)
    index[ys, xs] = np.arange(n)
    rows, cols, vals = [np.arange(n)], [np.arange(n)], [np.full(n, 4.0)]
    b = np.zeros(n)
    for dy, dx in ((-1, 0), (1, 0), (0, -1), (0, 1)):
        ny, nx = ys + dy, xs + dx
        inside = (ny >= 0) & (ny < H) & (nx >= 0) & (nx < W)
        nyc, nxc = np.clip(ny, 0, H - 1), np.clip(nx, 0, W - 1)
        unk = inside & mask[nyc, nxc]
        known = inside & ~mask[nyc, nxc]
        rows.append(np.nonzero(unk)[0]); cols.append(index[nyc[unk], nxc[unk]]); vals.append(np.full(unk.sum(), -1.0))
        b[known] += fg[nyc[known], nxc[known]]
    b -= lap[ys, xs]
    A = scipy.sparse.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n))
    out[ys, xs] = scipy.sparse.linalg.spsolve(A, b)
    return out


def transform_depth_pc(depth: np.ndarray, bg_depth: np.ndarray, fg_mask: np.ndarray, K: np.ndarray,
                       rot_angle: float = 0.0, rot_axis: Sequence[float] = (0.0, 1.0, 0.0),
                       translation: Sequence[float] = (0.0, 0.0, 0.0),
                       use_input_depth_normalization: bool = False, loop: bool = False,
                       poisson: bool = True) -> Dict[str, np.ndarray]:
    """Resolution-generic restatement of depth_transform.py:198-363.  depth/bg_depth/fg_mask are (S,S).

    Returns every intermediate the CUDA path is compared against:
    ``points`` (N,3) fp64, ``pix`` (N,), ``winner`` (S*S,), ``depth_map`` (S,S) fp32, ``target_mask``,
    ``visible`` (N,), ``cleaned`` (S,S) bool, ``correspondences`` (N_corr,4) int64 [x_src,y_src,x_dst,y_dst],
    ``disparity_raw`` (S,S) fp32, ``inpaint_mask`` (S,S) bool, ``disparity`` (S,S) fp32 (Poisson-filled).
    """
    depth = np.asarray(depth, dtype=f32)
    bg_depth = np.asarray(bg_depth, dtype=f32)
    mask = np.asarray(fg_mask).astype(bool)
    S = mask.shape[-1]
    if mask.shape[0] != mask.shape[1]:
        raise RuntimeError(f"Expected fg_mask to be square, got shape {mask.shape[0]} x {mask.shape[1]}.")
    out: Dict[str, np.ndarray] = {}
    with np.errstate(all="ignore"):
        bounds = None
        if use_input_depth_normalization:
            d = (f32(1.0) / depth).astype(f32)
            bounds = (d.min(), d.max())
        if not mask.any():
            out["correspondences"] = np.zeros((0, 4), np.int64)
            out["disparity"] = normalize_depth((f32(1.0) / depth).astype(f32), bounds)
            return out
        bg_pts = depth_to_world_coords(bg_depth, K).reshape(-1, 3)
        pts = depth_to_world_coords(depth, K).reshape(-1, 3)
        F = np.nonzero(mask.reshape(-1))[0]
        r, cen = rigid_transform_fg(pts[F], rot_axis, rot_angle, translation)
        points = np.vstack([bg_pts.astype(f64), r])
        P = S * S
        point_mask = np.arange(points.shape[0]) >= P
        depth_map, target_mask, tx, ty, visible, winner = points_to_depth(points, K, (S, S), point_mask, loop=loop)
        u, v = project_points(points, K, (S, S))
        disparity_raw = normalize_depth((f32(1.0) / depth_map).astype(f32), bounds)
    vis_fg = visible[P:]
    src = F[vis_fg]
    cleaned = clean_target_mask(target_mask, S)
    keep = cleaned[ty, tx]
    corr = np.stack([src % S, src // S, tx, ty], axis=-1)[keep].astype(np.int64)
    inpaint = cleaned ^ target_mask
    out.update(points=points, centroid=cen, pix=v * S + u, winner=winner, depth_map=depth_map,
               target_mask=target_mask, visible=visible, cleaned=cleaned, correspondences=corr,
               disparity_raw=disparity_raw, inpaint_mask=inpaint, fg_index=F)
    if poisson:
        out["disparity"] = poisson_solve(disparity_raw, inpaint.astype(np.uint8)).astype(f32)
    return out


# --------------------------------------------------------------------------------------------
# A.7 process_correspondences
# --------------------------------------------------------------------------------------------
def binary_erosion_cross(mask: np.ndarray, iterations: int) -> np.ndarray:
    """scipy.ndimage.binary_erosion(mask, iterations=n): 3x3 cross, border_value=0 (erodes from the border)."""
    m = np.asarray(mask).astype(bool)
    for _ in range(iterations):
        p = np.pad(m, 1, constant_values=False)
        m = p[1:-1, 1:-1] & p[:-2, 1:-1] & p[2:, 1:-1] & p[1:-1, :-2] & p[1:-1, 2:]
    return m


def process_correspondences(corr: np.ndarray, img_res: int, bg_erosion: int = 0, grid: int = 64) -> Dict[str, np.ndarray]:
    """guided_stable_diffuser.py:490-584 in closed form (bounds filter -> // (img_res//64) -> masks -> nonzero)."""
    corr = np.asarray(corr, dtype=np.int64).reshape(-1, 4)
    ox, oy, tx, ty = corr[:, 0], corr[:, 1], corr[:, 2], corr[:, 3]
    ok = (tx >= 0) & (tx < img_res) & (ty >= 0) & (ty < img_res)
    r = img_res // grid
    ox, oy, tx, ty = ox[ok] // r, oy[ok] // r, tx[ok] // r, ty[ok] // r
    bo = np.ones((grid, grid), bool)
    bt = np.ones((grid, grid), bool)
    if len(ox):
        bo[oy, ox] = False
        bt[ty, tx] = False
    if bg_erosion > 0:
        bo = binary_erosion_cross(bo, bg_erosion)
        bt = binary_erosion_cross(bt, bg_erosion)
    by, bx = np.nonzero(bo & bt)
    byo, bxo = np.nonzero(bo)
    byt, bxt = np.nonzero(bt)
    return {"original_x": ox, "original_y": oy, "transformed_x": tx, "transformed_y": ty,
            "background_x": bx, "background_y": by, "background_x_orig": bxo, "background_y_orig": byo,
            "background_x_trans": bxt, "background_y_trans": byt}


# --------------------------------------------------------------------------------------------
# row 9: the activation warp (list form and dense form)
# --------------------------------------------------------------------------------------------
def warp_gather_list(A: np.ndarray, y: np.ndarray, x: np.ndarray) -> np.ndarray:
    """W[c,n] = A[c, y[n], x[n]] - exactly the reference gather (losses.py:46-47, :80)."""
    return np.ascontiguousarray(A[:, y, x])


def dense_source_map(corr: np.ndarray, img_res: int, side: int,
                     winner_src: Optional[np.ndarray] = None) -> np.ndarray:
    """Per-level dense source map (side*side,) int32: ``src(q)`` = source cell of the FIRST correspondence
    in reference order (lowest n) whose destination cell is q; -1 where there is none (SURVEY.md 8(a) row 9).

    With ``winner_src`` (img_res*img_res int64: source pixel of every target pixel's splat winner, -1 = hole)
    cells without a correspondence fall back to the lowest-index target pixel of the cell that has a
    winner ("full winner-index map": background stays in place, foreground moves).
    """
    r = img_res // side
    corr = np.asarray(corr, dtype=np.int64).reshape(-1, 4)
    m = np.full(side * side, -1, dtype=np.int64)
    if winner_src is not None:
        ws = np.asarray(winner_src, dtype=np.int64).reshape(img_res, img_res)
        # visit target pixels in reverse raster order so the lowest index is written last
        ty, tx = np.divmod(np.arange(img_res * img_res - 1, -1, -1), img_res)
        s = ws[ty, tx]
        ok = s >= 0
        cell = (ty[ok] // r) * side + tx[ok] // r
        m[cell] = ((s[ok] // img_res) // r) * side + (s[ok] % img_res) // r
    if len(corr):
        d = (corr[:, 3] // r) * side + corr[:, 2] // r
        s = (corr[:, 1] // r) * side + corr[:, 0] // r
        m[d[::-1]] = s[::-1]
    return m.astype(np.int32)


def warp_gather_dense(A: np.ndarray, src_map: np.ndarray) -> np.ndarray:
    """D[c,q] = A[c, src_map[q]] if src_map[q] >= 0 else 0.   A (C,h,w) -> (C,h,w)."""
    C, h, w = A.shape
    flat = A.reshape(C, h * w)
    safe = np.where(src_map >= 0, src_map, 0)
    out = flat[:, safe]
    out[:, src_map < 0] = 0
    return out.reshape(C, h, w)


# --------------------------------------------------------------------------------------------
# A.8 losses (closed forms for patch_size == 1; dtype selects fp32 restatement or fp64 truth)
# --------------------------------------------------------------------------------------------
def bilinear_axis_table(n_in: int, n_out: int):
    """torch ``F.interpolate(mode='bilinear', align_corners=False)`` per-axis taps:
    src = max(scale*(i+0.5)-0.5, 0), i0 = floor(src), i1 = i0 + (i0 < n_in-1), lam = src - i0 (fp32)."""
    scale = f32(n_in) / f32(n_out)
    i = np.arange(n_out, dtype=f32)
    src = np.maximum((scale * (i + f32(0.5))).astype(f32) - f32(0.5), f32(0)).astype(f32)
    i0 = np.minimum(src.astype(np.int64), n_in - 1)
    i1 = i0 + (i0 < n_in - 1)
    lam = (src - i0.astype(f32)).astype(f32)
    return i0, i1, lam


def bilinear_resize(A: np.ndarray, size: Tuple[int, int], dtype=f32) -> np.ndarray:
    C, h, w = A.shape
    Ho, Wo = size
    if (h, w) == (Ho, Wo):
        return A.astype(dtype)
    y0, y1, ly = bilinear_axis_table(h, Ho)
    x0, x1, lx = bilinear_axis_table(w, Wo)
    A = A.astype(dtype)
    ly, lx = ly.astype(dtype)[None, :, None], lx.astype(dtype)[None, None, :]
    top = A[:, y0][:, :, x0] * (1 - lx) + A[:, y0][:, :, x1] * lx
    bot = A[:, y1][:, :, x0] * (1 - lx) + A[:, y1][:, :, x1] * lx
    return (top * (1 - ly) + bot * ly).astype(dtype)


def bilinear_resize_transpose(G: np.ndarray, in_size: Tuple[int, int], dtype=f64) -> np.ndarray:
    """Adjoint of ``bilinear_resize``: G (C,Ho,Wo) -> (C,h,w)."""
    C, Ho, Wo = G.shape
    h, w = in_size
    if (h, w) == (Ho, Wo):
        return G.astype(dtype)
    y0, y1, ly = bilinear_axis_table(h, Ho)
    x0, x1, lx = bilinear_axis_table(w, Wo)
    My = np.zeros((Ho, h), dtype); Mx = np.zeros((Wo, w), dtype)
    np.add.at(My, (np.arange(Ho), y0), 1 - ly.astype(dtype)); np.add.at(My, (np.arange(Ho), y1), ly.astype(dtype))
    np.add.at(Mx, (np.arange(Wo), x0), 1 - lx.astype(dtype)); np.add.at(Mx, (np.arange(Wo), x1), lx.astype(dtype))
    return np.einsum("cyx,yh,xw->chw", G.astype(dtype), My, Mx).astype(dtype)


def box_sum(M: np.ndarray, patch: int) -> np.ndarray:
    """Window sums of ``AvgPool2d(patch, stride=1, padding=patch//2)`` (zero padded, losses.py:64) at the first H x W
    output positions: out[.., q] = sum_{d in [0,patch)} M[.., q - patch//2 + d].  (For an even patch torch's output has
    one more row and column; the losses only ever index rows/columns < H.)"""
    C, H, W = M.shape
    pad = patch // 2
    Mp = np.pad(M, ((0, 0), (pad, patch), (pad, patch)))
    out = np.zeros_like(M)
    for dy in range(patch):
        for dx in range(patch):
            out = out + Mp[:, dy:dy + H, dx:dx + W]
    return out


def box_sum_transpose(Q: np.ndarray, patch: int) -> np.ndarray:
    """Adjoint of ``box_sum``: out[.., j] = sum of Q over the output positions q (< H) whose window contains j."""
    C, H, W = Q.shape
    pad = patch // 2
    Qp = np.pad(Q, ((0, 0), (patch, patch), (patch, patch)))
    out = np.zeros_like(Q)
    for dy in range(patch):
        for dx in range(patch):
            out = out + Qp[:, pad - dy + patch:pad - dy + patch + H, pad - dx + patch:pad - dx + patch + W]
    return out


def foreground_loss(cur: np.ndarray, orig: np.ndarray, pc: Dict[str, np.ndarray],
                    size=(64, 64), dtype=f64, x1="original_x", y1="original_y",
                    x2="transformed_x", y2="transformed_y", patch: int = 1):
    """losses.py:4-17 + :51-84.  Returns (loss, dL/dcur at native resolution).

    patch 1: L = mean_c mean_n |up(orig)[c,src_n] - up(cur)[c,dst_n]|.
    patch p: the two maps are first replaced by their local averages over the indexed cells,
             F[c,q] = (box_p(w * up)[c,q] / p^2) / (box_p(w)[q] / p^2 + 1e-10),  w = 1 on the indexed cells
             (losses.py:57-77), and the gradient flows back through the average of the current map.
    An empty index list gives loss NaN (mean over nothing) and gradient ZERO, as torch's autograd does."""
    C, h, w = cur.shape
    uo = bilinear_resize(orig, size, dtype)
    uc = bilinear_resize(cur, size, dtype)
    ys, xs, yd, xd = pc[y1], pc[x1], pc[y2], pc[x2]
    N = len(xs)
    if N == 0:
        return dtype(np.nan), np.zeros(cur.shape, dtype)
    if patch != 1:
        w1 = np.zeros((1,) + tuple(size), dtype); w2 = np.zeros((1,) + tuple(size), dtype)
        w1[0, ys, xs] = 1; w2[0, yd, xd] = 1
        pp = dtype(patch * patch)
        den1 = (box_sum(w1, patch) / pp + dtype(1e-10)).astype(dtype)
        den2 = (box_sum(w2, patch) / pp + dtype(1e-10)).astype(dtype)
        uo = ((box_sum(w1 * uo, patch) / pp).astype(dtype) / den1).astype(dtype)
        uc = ((box_sum(w2 * uc, patch) / pp).astype(dtype) / den2).astype(dtype)
    # patch 1: the local average of an indexed cell is f / (1 + 1e-10) (losses.py:75-77) - the identity in fp32, a 1e-10
    # relative factor in fp64
    one_eps = dtype(1) + dtype(1e-10) if patch == 1 else dtype(1)
    d = uo[:, ys, xs] / one_eps - uc[:, yd, xd] / one_eps
    loss = np.abs(d).mean(axis=-1).mean()
    g_up = np.zeros((C, size[0] * size[1]), dtype)
    cell = yd * size[1] + xd
    contrib = -np.sign(d) / dtype(C * N) / one_eps
    for c in range(C) if C <= 8 else ():
        np.add.at(g_up[c], cell, contrib[c])
    if C > 8:
        # accumulate per destination cell with a sparse one-hot matmul
        import scipy.sparse
        Sm = scipy.sparse.csr_matrix((np.ones(N), (np.arange(N), cell)), shape=(N, size[0] * size[1]))
        g_up = np.asarray(contrib @ Sm)
    g_up = g_up.reshape(C, *size)
    if patch != 1:
        g_up = (w2 * box_sum_transpose((g_up / den2 / pp).astype(dtype), patch)).astype(dtype)
    g = bilinear_resize_transpose(g_up, (h, w), dtype)
    return dtype(loss), g


def background_loss(cur: np.ndarray, orig: np.ndarray, pc: Dict[str, np.ndarray],
                    size=(64, 64), loss_type: str = "global_avg", dtype=f64, patch: int = 1):
    """losses.py:19-49.  Returns (loss, dL/dcur).  ``patch`` only matters for 'local_avg'."""
    if loss_type == "local_avg":
        return foreground_loss(cur, orig, pc, size, dtype, "background_x", "background_y", "background_x", "background_y", patch)
    if loss_type != "global_avg":
        raise ValueError(f"Unknown background loss type: {loss_type}")
    C, h, w = cur.shape
    uo = bilinear_resize(orig, size, dtype)
    uc = bilinear_resize(cur, size, dtype)
    y1, x1 = pc["background_y_orig"], pc["background_x_orig"]
    y2, x2 = pc["background_y_trans"], pc["background_x_trans"]
    if len(x2) == 0:
        return dtype(np.nan), np.zeros(cur.shape, dtype)          # NaN loss, nothing to scatter the gradient to
    if len(x1) == 0:
        return dtype(np.nan), np.zeros(cur.shape, dtype)          # NaN difference: torch's abs backward takes sign(NaN) = 0
    delta = uo[:, y1, x1].mean(-1) - uc[:, y2, x2].mean(-1)
    loss = np.abs(delta).mean()
    g_up = np.zeros((C, size[0] * size[1]), dtype)
    # a cell listed k times receives k quanta (np.add.at accumulates over repeated indices, fancy assignment would not)
    np.add.at(g_up, (slice(None), np.asarray(y2) * size[1] + np.asarray(x2)), (-np.sign(delta) / dtype(C * len(x2)))[:, None])
    return dtype(loss), bilinear_resize_transpose(g_up.reshape(C, *size), (h, w), dtype)


def loss_sign_ambiguity(cur: np.ndarray, orig: np.ndarray, pc: Dict[str, np.ndarray], size=(64, 64),
                        bg_loss_type: str = "global_avg", eps: float = 2e-6, patch: int = 1, bg_patch: Optional[int] = None) -> np.ndarray:
    """bool (C,h,w): native cells whose gradient depends on sign(d) of a difference with |d| < eps.

    The losses are L1: their gradient is a sum of +-1/(C N) terms.  Where a difference is within fp32 rounding
    of zero, its sign - and with it one gradient quantum - legitimately depends on the arithmetic (fp32 vs fp64,
    FMA contraction); the reference itself differs between its CPU and CUDA runs there.  Parity tests compare the
    gradients on the complement of this mask and require the mask to be a vanishing fraction of the tensor.
    With a patch > 1 the difference is taken between local averages and one quantum spreads over the patch."""
    C, h, w = cur.shape
    bg_patch = patch if bg_patch is None else bg_patch
    uo = bilinear_resize(orig, size, f64)
    uc = bilinear_resize(cur, size, f64)

    def local(ys, xs, yd, xd, p):
        a, b = uo, uc
        w2 = np.zeros((1,) + tuple(size), f64)
        w2[0, yd, xd] = 1
        if p != 1:
            w1 = np.zeros((1,) + tuple(size), f64)
            w1[0, ys, xs] = 1
            a = box_sum(w1 * uo, p) / (box_sum(w1, p) + 1e-10 * p * p)
            b = box_sum(w2 * uc, p) / (box_sum(w2, p) + 1e-10 * p * p)
        d = a[:, ys, xs] - b[:, yd, xd]
        amb = np.zeros((C, size[0] * size[1]), bool)
        cc, nn = np.nonzero(np.abs(d) < eps)
        amb[cc, (yd * size[1] + xd)[nn]] = True
        amb = amb.reshape(C, *size)
        if p != 1:
            amb = (box_sum_transpose(amb.astype(f64), p) > 0) & (w2 > 0)
        return amb

    amb_up = np.zeros((C,) + tuple(size), bool)
    if len(pc["original_x"]):
        amb_up |= local(pc["original_y"], pc["original_x"], pc["transformed_y"], pc["transformed_x"], patch)
    if bg_loss_type == "local_avg" and len(pc["background_x"]):
        amb_up |= local(pc["background_y"], pc["background_x"], pc["background_y"], pc["background_x"], bg_patch)
    amb = bilinear_resize_transpose(amb_up.astype(f64), (h, w), f64) > 0
    if bg_loss_type == "global_avg" and len(pc["background_x_orig"]) and len(pc["background_x_trans"]):
        delta = uo[:, pc["background_y_orig"], pc["background_x_orig"]].mean(-1) - uc[:, pc["background_y_trans"], pc["background_x_trans"]].mean(-1)
        amb[np.abs(delta) < eps] = True
    return amb


def guidance_weight_schedule(fg_weight: float = 1.5, bg_weight: float = 1.25, guidance_max_step: int = 38,
                             schedule_type: str = "constant"):
    """guided_stable_diffuser.py:336-373 + StepGuidanceWeightSchedule :622-665 as a function (t_idx, it) -> (fgw, bgw)."""
    fgw, bgw = fg_weight * 30, bg_weight * 30
    if schedule_type == "constant":
        ff, bf = np.linspace(fgw, fgw, guidance_max_step), np.linspace(bgw, bgw, guidance_max_step)
    elif schedule_type == "linear":
        ff, bf = np.linspace(fgw, 0.0, guidance_max_step), np.linspace(bgw, 0.0, guidance_max_step)
    elif schedule_type == "quadratic":
        ff, bf = np.linspace(np.sqrt(fgw), 0.0, guidance_max_step) ** 2, np.linspace(np.sqrt(bgw), 0.0, guidance_max_step) ** 2
    else:
        raise ValueError(f"Unknown guidance schedule type: {schedule_type}")
    den = []
    for t in range(guidance_max_step):
        fw, bw = ([0.0, 0.0, 7.5], [0.0, 0.0, 1.5]) if t % 3 == 0 else \
                 ([0.0, 5.0, 0.0], [0.0, 1.5, 0.0]) if t % 3 == 1 else ([0.0, 5.0, 7.5], [0.0, 1.5, 1.5])
        den.append(((np.array(fw) * ff[t]).tolist(), (np.array(bw) * bf[t]).tolist()))
    den.append(([0.0] * 3, [0.0] * 3))
    opt = [([2.5] * 3, [1.25] * 3), ([1.25] * 3, [2.5] * 3), ([1.25] * 3, [1.25] * 3), ([2.5] * 3, [2.5] * 3)]

    def schedule(t_idx: int, it: int):
        if t_idx < 0 or it < 0:
            raise ValueError(f"Could not find weights for denoising step {t_idx} and optimization step {it}.")
        df, db = den[min(t_idx, guidance_max_step)]
        of, ob = opt[min(it, 3)]
        return [a * b for a, b in zip(df, of)], [a * b for a, b in zip(db, ob)]
    return schedule


# --------------------------------------------------------------------------------------------
# the elementwise steps of guided_inference around the U-Net (SURVEY.md 8(f) rank 4)
#
# PARITY UNPINNED for the scheduler arithmetic: it lives in diffusers (pyproject.toml:30 pins 0.23.*), which is not
# installed here and not under /root/reference.  Restated from the published algorithm (DDIM, Song et al. 2021, eq. 12, as
# DDIMScheduler.step of diffusers 0.23 evaluates it: epsilon prediction, eta = 0, no clipping) and anchored on the
# reference's call sites (guided_stable_diffuser.py:31-32 constructor, :262-267 and :470-474 CFG + step, :434 latent update)
# and on the published endpoints of Stable Diffusion's scaled-linear table (alphas_cumprod[0] = 0.99915, [999] = 0.00466).
# --------------------------------------------------------------------------------------------
def ddim_alphas_cumprod(num_train_timesteps: int = 1000, beta_start: float = 0.00085, beta_end: float = 0.012) -> np.ndarray:
    """``torch.cumprod(1 - torch.linspace(beta_start**0.5, beta_end**0.5, N, dtype=float32)**2, 0)`` ("scaled_linear"): the
    products are accumulated in fp64 and rounded to fp32 per element, as torch's CPU cumprod does."""
    root = linspace_f32(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps)
    alphas = f32(1.0) - root * root
    return np.cumprod(alphas.astype(f64)).astype(f32)


def ddim_timesteps(num_inference_steps: int, num_train_timesteps: int = 1000, steps_offset: int = 0) -> np.ndarray:
    """"leading" spacing: multiples of N // n, descending."""
    ratio = num_train_timesteps // num_inference_steps
    return (np.arange(num_inference_steps)[::-1] * ratio).astype(np.int64) + steps_offset


def cfg_combine(noise_uncond: np.ndarray, noise_text: np.ndarray, guidance_scale: float = 7.5) -> np.ndarray:
    """guided_stable_diffuser.py:470-471 (fp32, each op rounded)."""
    u, t = noise_uncond.astype(f32), noise_text.astype(f32)
    return u + f32(guidance_scale) * (t - u)


def ddim_coefficients(timestep: int, alphas_cumprod: np.ndarray, num_inference_steps: int,
                      final_alpha_cumprod: Optional[float] = None) -> Tuple[np.float32, np.float32, np.float32, np.float32]:
    """(sqrt(1 - a_t), sqrt(a_t), sqrt(a_prev), sqrt(1 - a_prev)) in fp32 with correctly rounded square roots.  diffusers evaluates
    ``a ** 0.5`` on 0-d CPU tensors, i.e. with torch's CPU sqrt, which (MKL VML here) may differ from the correctly rounded value
    by one ulp - comparisons of the coefficients therefore allow 1 ulp."""
    n_train = alphas_cumprod.shape[0]
    prev = timestep - n_train // num_inference_steps
    a_t = f32(alphas_cumprod[timestep])
    a_prev = f32(alphas_cumprod[prev]) if prev >= 0 else f32(alphas_cumprod[0] if final_alpha_cumprod is None else final_alpha_cumprod)
    return np.sqrt(f32(1.0) - a_t), np.sqrt(a_t), np.sqrt(a_prev), np.sqrt(f32(1.0) - a_prev)


def ddim_step(model_output: np.ndarray, timestep: int, sample: np.ndarray, alphas_cumprod: np.ndarray, num_inference_steps: int,
              final_alpha_cumprod: Optional[float] = None, reciprocal_division: bool = False, coefficients=None) -> np.ndarray:
    """x_{t-1} = sqrt(a_prev) * x0 + sqrt(1 - a_prev) * eps with x0 = (x_t - sqrt(1 - a_t) * eps) / sqrt(a_t); every coefficient
    and every elementwise op in fp32.  ``reciprocal_division``: multiply by fl32(1 / sqrt(a_t)) instead of dividing (what
    torch's CUDA kernels do for a host-scalar divisor).  ``coefficients``: use these four fp32 values instead of
    ``ddim_coefficients`` (to separate the elementwise arithmetic from the 1-ulp question of the square roots)."""
    if coefficients is None:
        coefficients = ddim_coefficients(timestep, alphas_cumprod, num_inference_steps, final_alpha_cumprod)
    sqrt_beta_t, sqrt_alpha_t, sqrt_alpha_prev, sqrt_beta_prev = (f32(c) for c in coefficients)
    eps, x = model_output.astype(f32), sample.astype(f32)
    num = x - sqrt_beta_t * eps
    x0 = num * (f32(1.0) / sqrt_alpha_t) if reciprocal_division else num / sqrt_alpha_t
    return sqrt_alpha_prev * x0 + sqrt_beta_prev * eps


def latent_update(latents: np.ndarray, grad: np.ndarray, step_size: float = 0.1) -> np.ndarray:
    """guided_stable_diffuser.py:434: latents - grad * 0.1 in fp32 (0.1 rounded to fp32 first, as torch does for a Python scalar)."""
    return latents.astype(f32) - grad.astype(f32) * f32(step_size)


# --------------------------------------------------------------------------------------------
# synthetic workloads of SURVEY.md 8(d)
# --------------------------------------------------------------------------------------------
def smooth_scene(S: int = 512, seed: int = 0):
    """A scene closer to the reference's fixtures than the config-1 recipe: smooth curved surfaces (no per-pixel noise, so
    neighbouring points project to neighbouring pixels and z-fights come from geometry), an irregular foreground made of
    overlapping ellipses with a hole, a thin bar and a detached blob.  Plain arithmetic on seeded NumPy draws, rounded to
    fp32 once, so every box regenerates the same arrays."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:S, 0:S].astype(np.float64) / S
    bg = 3.6 + 1.1 * yy + 0.25 * (xx - 0.5) ** 2 + 0.08 * yy * xx
    mask = np.zeros((S, S), bool)
    fg = np.full((S, S), 10.0)
    for _ in range(3):
        cx, cy = rng.uniform(0.35, 0.65), rng.uniform(0.4, 0.7)
        ax, ay = rng.uniform(0.08, 0.2), rng.uniform(0.08, 0.2)
        r2 = ((xx - cx) / ax) ** 2 + ((yy - cy) / ay) ** 2
        inside = r2 < 1.0
        bump = 2.4 + 0.3 * (cy - 0.5) - 0.35 * np.sqrt(np.maximum(0.0, 1.0 - r2)) + 0.15 * (xx - cx)
        fg = np.where(inside, np.minimum(fg, bump), fg)
        mask |= inside
    hx, hy = rng.uniform(0.45, 0.55), rng.uniform(0.5, 0.6)
    mask &= ~(((xx - hx) / 0.03) ** 2 + ((yy - hy) / 0.04) ** 2 < 1.0)            # a hole
    bar = (np.abs(yy - 0.3) < 1.5 / S) & (xx > 0.2) & (xx < 0.8)                   # a 3-pixel bar
    blob = ((xx - 0.15) / 0.04) ** 2 + ((yy - 0.8) / 0.05) ** 2 < 1.0               # a detached blob
    fg = np.where(bar & ~mask, 2.0 + 0.2 * xx, fg)
    fg = np.where(blob & ~mask, 2.8 - 0.2 * yy, fg)
    mask |= bar | blob
    depth = np.where(mask, fg, bg)
    return depth.astype(f32), bg.astype(f32), mask.astype(f32)


def synthetic_scene(S: int = 512, seed: int = 0, cx: Optional[float] = None, cy: Optional[float] = None,
                    radius: Optional[float] = None, quantize: Optional[float] = None, kind: str = "disc"):
    """Config-1 recipe (scaled with S): bg_depth = 4 + row/S + 0.05*rand, fg = 2 + 0.3*rand inside a disc;
    ``kind='smooth'`` gives ``smooth_scene``."""
    if kind == "smooth":
        return smooth_scene(S, seed)
    import torch
    g = torch.Generator().manual_seed(seed)
    rows = torch.arange(S, dtype=torch.float32)[:, None]
    bg = 4 + rows / S + 0.05 * torch.rand(S, S, generator=g)
    fgv = 2 + 0.3 * torch.rand(S, S, generator=g)
    k = S / 512.0
    cx = 256 * k if cx is None else cx
    cy = 280 * k if cy is None else cy
    radius = 120 * k if radius is None else radius
    col = torch.arange(S, dtype=torch.float32)[None, :]
    mask = ((col - cx) ** 2 + (rows - cy) ** 2) < radius ** 2
    depth = torch.where(mask, fgv, bg)
    if quantize:
        depth = torch.round(depth / quantize) * quantize
        bg = torch.round(bg / quantize) * quantize
    return depth.numpy().astype(f32), bg.numpy().astype(f32), mask.numpy().astype(f32)


# --------------------------------------------------------------------------------------------
# mesh mode: hard z-buffer triangle rasteriser (pytorch3d rasterize_meshes semantics, SURVEY.md Appendix B).
# PARITY UNPINNED: pytorch3d is not installed and no reference test pins its output; this restates the PUBLISHED
# algorithm in fp32 with one rounding per operation, and is what the CUDA rasteriser is compared with.
# --------------------------------------------------------------------------------------------
def fov_scales(k11: float, H: int, W: int, znear: float = 0.1):
    """NDC scales (sx, sy) of pytorch3d's FoVPerspectiveCameras built the way pytorch3d_renderer.py:890-913 does
    (fov from the intrinsics, aspect ratio 1), evaluated with torch fp32 ops like the reference."""
    import torch
    k = torch.tensor(k11, dtype=torch.float32)
    if H != W:
        k = k * (H / max(H, W))
    fov = 2 * torch.rad2deg(torch.atan(1 / k))
    fov = (np.pi / 180) * fov
    tan_half = torch.tan(fov / 2)
    max_y = tan_half * znear
    min_y = -max_y
    max_x = max_y * 1.0
    min_x = -max_x
    return float(2.0 * znear / (max_x - min_x)), float(2.0 * znear / (max_y - min_y))


def _ndc_range(S1: int, S2: int):
    r = f32(2.0)
    if S1 > S2:
        r = f32(f32(f32(S1) * r) / f32(S2))
    return r


def _pix_to_ndc(i, S1: int, S2: int):
    r = _ndc_range(S1, S2)
    off = f32(r / f32(2.0))
    return (-off + ((r * np.asarray(i, f32)).astype(f32) + off).astype(f32) / f32(S1)).astype(f32)


def _edge(px, py, ax, ay, bx, by):
    return ((px - ax).astype(f32) * (by - ay).astype(f32)).astype(f32) - ((py - ay).astype(f32) * (bx - ax).astype(f32)).astype(f32)


def _seg_dist2(px, py, ax, ay, bx, by):
    bax, bay = f32(bx - ax), f32(by - ay)
    l2 = f32(f32(bax * bax) + f32(bay * bay))
    if l2 <= f32(1e-8):
        dx, dy = (px - bx).astype(f32), (py - by).astype(f32)
        return ((dx * dx).astype(f32) + (dy * dy).astype(f32)).astype(f32)
    t = (((bax * (px - ax).astype(f32)).astype(f32) + (bay * (py - ay).astype(f32)).astype(f32)).astype(f32) / l2).astype(f32)
    t = np.minimum(np.maximum(t, f32(0)), f32(1)).astype(f32)
    qx, qy = (ax + (t * bax).astype(f32)).astype(f32), (ay + (t * bay).astype(f32)).astype(f32)
    dx, dy = (px - qx).astype(f32), (py - qy).astype(f32)
    return ((dx * dx).astype(f32) + (dy * dy).astype(f32)).astype(f32)


def rasterize_meshes(verts: np.ndarray, faces: np.ndarray, H: int, W: int, sx: float, sy: float, blur_radius: float = 0.0,
                     cull_backfaces: bool = False, perspective_correct: bool = True, clip_barycentric: bool = True):
    """Returns pix_to_face (H,W) int32 (-1 empty), zbuf (H,W) fp32, bary (H,W,3) fp32 (-1 empty)."""
    verts = np.asarray(verts, f32)
    with np.errstate(all="ignore"):
        Z = verts[:, 2]
        den = np.where(Z < 0, -np.maximum(np.abs(Z), f32(1e-8)), np.maximum(np.abs(Z), f32(1e-8))).astype(f32)
        nx = ((f32(sx) * verts[:, 0]).astype(f32) / den).astype(f32)
        ny = ((f32(sy) * verts[:, 1]).astype(f32) / den).astype(f32)
    eps = f32(1e-8)
    bs = f32(np.sqrt(f32(blur_radius)))
    blur = f32(blur_radius)
    best_z = np.full((H, W), np.inf, f32)
    best_f = np.full((H, W), -1, np.int64)
    best_b = np.full((H, W, 3), -1, f32)
    xs_ndc = _pix_to_ndc(np.arange(W), W, H)      # indexed by xidx
    ys_ndc = _pix_to_ndc(np.arange(H), H, W)
    for f, (i0, i1, i2) in enumerate(np.asarray(faces, np.int64)):
        x0, y0, z0, x1, y1, z1, x2, y2, z2 = nx[i0], ny[i0], Z[i0], nx[i1], ny[i1], Z[i1], nx[i2], ny[i2], Z[i2]
        if max(z0, z1, z2) < 0:
            continue
        xmin, xmax = f32(min(x0, x1, x2) - bs), f32(max(x0, x1, x2) + bs)
        ymin, ymax = f32(min(y0, y1, y2) - bs), f32(max(y0, y1, y2) + bs)
        area = _edge(np.asarray(x0), np.asarray(y0), x1, y1, x2, y2)
        if (cull_backfaces and area < 0) or (-eps <= area <= eps):
            continue
        xi = np.nonzero((xs_ndc <= xmax) & (xs_ndc >= xmin))[0]
        yi = np.nonzero((ys_ndc <= ymax) & (ys_ndc >= ymin))[0]
        if len(xi) == 0 or len(yi) == 0:
            continue
        py, px = np.meshgrid(ys_ndc[yi], xs_ndc[xi], indexing="ij")
        px, py = px.astype(f32).ravel(), py.astype(f32).ravel()
        yy, xx = np.meshgrid(yi, xi, indexing="ij")
        with np.errstate(all="ignore"):
            a = f32(_edge(np.asarray(x2), np.asarray(y2), x0, y0, x1, y1) + eps)
            w0 = (_edge(px, py, x1, y1, x2, y2) / a).astype(f32)
            w1 = (_edge(px, py, x2, y2, x0, y0) / a).astype(f32)
            w2 = (_edge(px, py, x0, y0, x1, y1) / a).astype(f32)
            if perspective_correct:
                t0 = ((w0 * z1).astype(f32) * z2).astype(f32)
                t1 = ((z0 * w1).astype(f32) * z2).astype(f32)
                t2 = (f32(z0 * z1) * w2).astype(f32)
                dn = np.maximum(((t0 + t1).astype(f32) + t2).astype(f32), eps).astype(f32)
                w0, w1, w2 = (t0 / dn).astype(f32), (t1 / dn).astype(f32), (t2 / dn).astype(f32)
            c0, c1, c2 = w0, w1, w2
            if clip_barycentric:
                c0, c1, c2 = (np.maximum(f32(0), np.minimum(f32(1), w)).astype(f32) for w in (w0, w1, w2))
                sm = np.maximum(((c0 + c1).astype(f32) + c2).astype(f32), f32(1e-5)).astype(f32)
                c0, c1, c2 = (c0 / sm).astype(f32), (c1 / sm).astype(f32), (c2 / sm).astype(f32)
            pz = (((c0 * z0).astype(f32) + (c1 * z1).astype(f32)).astype(f32) + (c2 * z2).astype(f32)).astype(f32)
            inside = (w0 > 0) & (w1 > 0) & (w2 > 0)
            d = np.minimum(_seg_dist2(px, py, x0, y0, x1, y1), np.minimum(_seg_dist2(px, py, x0, y0, x2, y2), _seg_dist2(px, py, x1, y1, x2, y2)))
            ok = (pz >= 0) & (inside | (d < blur))
        rows, cols = (H - 1 - yy.ravel()), (W - 1 - xx.ravel())
        for k in np.nonzero(ok)[0]:
            r, c = rows[k], cols[k]
            if pz[k] < best_z[r, c]:          # faces are visited in index order: strict '<' == lexicographic (pz, face)
                best_z[r, c] = pz[k]; best_f[r, c] = f; best_b[r, c] = (c0[k], c1[k], c2[k])
    zbuf = np.where(best_f >= 0, best_z, f32(-1)).astype(f32)
    return best_f.astype(np.int32), zbuf, best_b


def interpolate_face_attributes(attr: np.ndarray, faces: np.ndarray, pix_to_face: np.ndarray, bary: np.ndarray) -> np.ndarray:
    """(H,W,D+1): hard blend of the interpolated vertex attribute, alpha last, background 0."""
    attr = np.asarray(attr, f32)
    H, W = pix_to_face.shape
    out = np.zeros((H, W, attr.shape[1] + 1), f32)
    hit = pix_to_face >= 0
    fv = np.asarray(faces, np.int64)[pix_to_face[hit]]
    b = bary[hit]
    val = (((attr[fv[:, 0]] * b[:, 0:1]).astype(f32) + (attr[fv[:, 1]] * b[:, 1:2]).astype(f32)).astype(f32) + (attr[fv[:, 2]] * b[:, 2:3]).astype(f32)).astype(f32)
    out[hit, :-1] = val
    out[hit, -1] = 1
    return out
