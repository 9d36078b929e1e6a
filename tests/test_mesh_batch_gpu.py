"""GPU (-m gpu): mesh mode for B transforms of one scene (depth_transform.transform_depth_mesh_batch / dh_edit_mesh_batch).
The background mesh is rasterised once and every edit's moved foreground goes on top of a copy of its z-buffer; every edit
must equal the joined-mesh renderer (MeshRenderer on [bg, moved fg], one dh_rasterize_meshes per edit) bit for bit -
disparities and correspondences, values and order - and the NumPy oracle on the joined mesh."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import dh_oracle as O
from helpers import load_photogen, photogen_filled_bg

pytestmark = pytest.mark.gpu

META, GET = load_photogen()
SCENES = sorted(META)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def K(dev):
    from diffusionhandles_b200.guided_stable_diffuser import GuidedStableDiffuser
    return GuidedStableDiffuser.get_depth_intrinsics(device=dev)


def _bits_equal(a, b):
    """bit-for-bit equality of two fp32 tensors (NaN payloads and the sign of zero included)"""
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# mixed transforms: (angle, axis, translation); None takes the single call's defaults
EDITS = [
    (35.0, torch.tensor([0.0, 1.0, 0.0]), torch.tensor([0.2, 0.0, 0.1])),
    (0.0, torch.tensor([0.0, 1.0, 0.0]), torch.tensor([0.0, 0.0, -20.0])),        # behind the camera: no correspondences
    (35.0, torch.tensor([0.0, 1.0, 0.0]), torch.tensor([0.2, 0.0, 0.1])),         # the first one again
    (-50.0, torch.tensor([0.3, 1.0, -0.2]), torch.tensor([-0.3, 0.1, 0.4])),
    (10.0, torch.tensor([1.0, 0.0, 0.0]), torch.tensor([60.0, 0.0, 0.0])),        # off-screen: no correspondences
    (None, None, None),
    (80.0, torch.tensor([0.0, 0.0, 1.0], dtype=torch.float64), torch.tensor([0.05, -0.1, -0.3], dtype=torch.float64)),
    (12.5, torch.tensor([0.0, -1.0, 0.0]), None),
]
GONE = (1, 4)           # the edits that leave no foreground on screen


def _scene(dev, H, W, seed):
    S = max(H, W)
    depth, bg, mask = O.synthetic_scene(S, seed)
    return tuple(torch.from_numpy(np.ascontiguousarray(a[:H, :W])).to(dev)[None, None] for a in (depth, bg, mask))


def _batch_vs_singles(td, tb, tm, K, edits, unn=False):
    from diffusionhandles_b200 import depth_transform as dt
    angles, axes, shifts = zip(*edits)
    disp, corrs = dt.transform_depth_mesh_batch(td, tb, tm, K, list(angles), list(axes), list(shifts), use_input_depth_normalization=unn)
    H, W = td.shape[-2:]
    assert disp.shape == (len(edits), 1, H, W) and disp.device == td.device and len(corrs) == len(edits)
    for b, edit in enumerate(edits):
        d1, c1 = _joined_mesh_edit(td, tb, tm, K, edit, unn)
        assert _bits_equal(disp[b:b + 1], d1), b
        assert corrs[b].device.type == "cpu" and corrs[b].dtype == torch.int64
        assert torch.equal(corrs[b], c1), (b, corrs[b].shape, c1.shape)
    return disp, corrs


@pytest.mark.parametrize("H,W", [(24, 24), (48, 48), (64, 64), (48, 64)])
@pytest.mark.parametrize("B", [1, 3, 8])
def test_batch_matches_single_path(dev, K, H, W, B):
    td, tb, tm = _scene(dev, H, W, 60 + H + W)
    edits = EDITS[:B]
    _, corrs = _batch_vs_singles(td, tb, tm, K, edits)
    assert corrs[0].shape[0] > 5                                   # the foreground is visible in the first edit
    for b in GONE:
        if b < B:
            assert corrs[b].shape == (0, 4), b
    if B >= 3:
        assert torch.equal(corrs[0], corrs[2])                    # identical transforms in one batch


# ------------------------------------------------------------------------------------------------
# the native call on hand-built meshes
# ------------------------------------------------------------------------------------------------
def _meshes(dev, K, td, tb, tm):
    from diffusionhandles_b200 import depth_transform as dt
    return dt.depth_to_mesh(tb, K), dt.depth_to_mesh(td, K, mask=tm[0, 0] > 0.5)


def _native_batch(dev, K, bg, fg, edits, H, W):
    """dh_edit_mesh_batch on the two meshes: (target_z (B,H,W), [corr rows], pix_to_face (B,H,W))"""
    from diffusionhandles_b200 import _native as N
    from diffusionhandles_b200.renderer import fov_scales
    lib = N.load()
    B = len(edits)
    f32, i32 = torch.float32, torch.int32
    bv, bf = bg.verts.to(f32).contiguous(), bg.faces.to(i32).contiguous()
    fv, fc, ff = fg.verts.to(f32).contiguous(), fg.vert_attributes["color"].to(f32).contiguous(), fg.faces.to(i32).contiguous()
    sx, sy = fov_scales(K[1, 1], H, W)
    ang = (C.c_float * B)(*[a for a, _, _ in edits])
    axs = (C.c_float * (3 * B))(*[v for _, ax, _ in edits for v in ax])
    trs = (C.c_float * (3 * B))(*[v for _, _, t in edits for v in t])
    z = torch.empty((B, H, W), dtype=f32, device=dev)
    corr = torch.empty((B, H * W, 4), dtype=torch.int64, device=dev)
    n = torch.empty(B, dtype=i32, device=dev)
    p2f = torch.empty((B, H, W), dtype=i32, device=dev)
    ws_bytes = int(lib.dh_edit_mesh_batch_workspace_bytes(B, bv.shape[0], fv.shape[0], H, W))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    N.check(lib.dh_edit_mesh_batch(N.ptr(bv), bv.shape[0], N.ptr(bf), bf.shape[0], N.ptr(fv), N.ptr(fc), fv.shape[0], N.ptr(ff),
                                   ff.shape[0], B, ang, axs, trs, H, W, (C.c_float * 9)(1, 0, 0, 0, 1, 0, 0, 0, 1), (C.c_float * 3)(0, 0, 0),
                                   sx, sy, 1e-5, 1, 1, 1, N.ptr(z), N.ptr(corr), N.ptr(n), N.ptr(p2f), N.ptr(ws), ws_bytes,
                                   N.stream_handle(dev)), "dh_edit_mesh_batch")
    counts = n.tolist()
    return z, [corr[b, :c].cpu() for b, c in enumerate(counts)], p2f


def _joined_render(dev, K, bg, fg, edit, H, W):
    """transform_points, then the renderer on the joined mesh [bg, moved fg]; None in the edit takes transform_depth_mesh's
    defaults"""
    from diffusionhandles_b200 import depth_transform as dt
    from diffusionhandles_b200.mesh import Mesh
    from diffusionhandles_b200.renderer import Camera, MeshRenderer, SplatRendererArgs
    a, ax, t = edit
    angle = torch.tensor(0.0 if a is None else float(a), dtype=torch.float32)
    axis = torch.tensor([0.0, 1.0, 0.0]) if ax is None else torch.as_tensor(ax)
    shift = torch.zeros(3) if t is None else torch.as_tensor(t)
    moved = Mesh(dt.transform_points(fg.verts, angle, axis, shift), fg.faces)
    moved.add_vert_attribute("color", fg.vert_attributes["color"])
    r = MeshRenderer(['world_position', 'flat_vertex_color'],
                     SplatRendererArgs(device=dev, output_res=(H, W), cull_backfaces=True, blur_radius=1e-5))
    r.update_scene({'meshes': [bg, moved], 'cameras': [Camera(intrinsics=K)]})
    layers = r.render()
    return moved, layers, r.fragments[0][0]


def _joined_mesh_edit(td, tb, tm, K, edit, unn):
    """One edit through the joined-mesh renderer: (disparity (1,1,H,W), correspondences (n,4) int64 CPU) read off the
    'world_position' z and the carried 'flat_vertex_color' layers, one row per target pixel that shows the foreground, in target
    raster order, sources rounded half-to-even; an empty mask gives the normalised input disparity."""
    from diffusionhandles_b200 import depth_transform as dt
    if not tm.any():
        return dt._empty_mask_result(td, unn)
    H, W = td.shape[-2:]
    bg, fg = _meshes(td.device, K, td, tb, tm)
    _, layers, _ = _joined_render(td.device, K, bg, fg, edit, H, W)
    target_depth = layers['world_position'][None, ..., 2]
    carried = layers['flat_vertex_color'][0]
    ty, tx = torch.nonzero(carried[..., 2] > 0.5, as_tuple=True)
    source = torch.round(carried[ty, tx, :2] * carried.new_tensor([W - 1, H - 1])).to(torch.int64)
    correspondences = torch.stack([source[:, 0], source[:, 1], tx, ty], dim=-1).cpu()
    bounds = dt.normalize_depth(1.0 / td, return_bounds=True)[1] if unn else None
    return dt.normalize_depth(1.0 / target_depth, bounds=bounds), correspondences


def test_tie_order_background_wins(dev, K):
    """A foreground lying exactly on the background (the same vertices, bit for bit) under an identity transform: every
    foreground face ties with a background face, and the background must win each tie as in the joined mesh.  The vertex
    coordinates are rounded to multiples of 2^-10 and the foreground has 8 x 8 = 64 vertices, so the centroid, p - c and
    (p - c) + c are exact and the identity transform leaves the vertices bit-identical."""
    from diffusionhandles_b200.mesh import Mesh
    S = 32
    depth, bg, mask = O.synthetic_scene(S, 70)
    mask = np.zeros((S, S), np.float32)
    mask[12:20, 10:18] = 1.0
    tb, tm = torch.from_numpy(bg).to(dev)[None, None], torch.from_numpy(mask).to(dev)[None, None]
    bg_mesh, fg_mesh = _meshes(dev, K, tb, tb, tm)                 # foreground depth == background depth
    v = torch.round(bg_mesh.verts * 1024) / 1024 + 0.0               # (+ 0.0 folds -0 into +0)
    bg_col = bg_mesh.vert_attributes["color"]
    bg_mesh = Mesh(v, bg_mesh.faces)
    bg_mesh.add_vert_attribute("color", bg_col)
    fg_verts = v.reshape(S, S, 3)[torch.from_numpy(mask > 0.5).to(dev)]
    assert fg_verts.shape[0] == 64
    col = fg_mesh.vert_attributes["color"]
    fg_mesh = Mesh(fg_verts.contiguous(), fg_mesh.faces)
    fg_mesh.add_vert_attribute("color", col)
    edits = [(0.0, (0.0, 1.0, 0.0), (0.0, 0.0, 0.0)), (0.0, (0.0, 1.0, 0.0), (0.0, 0.0, -0.5)), (0.0, (1.0, 0.0, 0.0), (0.0, 0.0, 0.0))]
    z, corrs, p2f = _native_batch(dev, K, bg_mesh, fg_mesh, edits, S, S)
    F_bg = bg_mesh.faces.shape[0]
    for b, e in enumerate(edits):
        moved, layers, p2f_joined = _joined_render(dev, K, bg_mesh, fg_mesh, e, S, S)
        if b != 1:
            assert torch.equal(moved.verts, fg_mesh.verts)          # an exact identity: every foreground face ties
        assert torch.equal(p2f[b], p2f_joined), b
        assert _bits_equal(z[b], layers['world_position'][0, ..., 2]), b
    assert (p2f[0] < F_bg).all() and (p2f[2] < F_bg).all()          # the background won every tie ...
    assert corrs[0].shape == (0, 4) and corrs[2].shape == (0, 4)     # ... so nothing is carried
    assert (p2f[1] >= F_bg).sum() > 20 and corrs[1].shape[0] > 20    # moved towards the camera, the foreground wins


def test_against_oracle(dev, K):
    """target z and the carried source pixels of a small batch against the NumPy rasteriser and interpolation on the joined
    mesh of each edit."""
    from diffusionhandles_b200 import depth_transform as dt
    S = 24
    td, tb, tm = _scene(dev, S, S, 71)
    bg_mesh, fg_mesh = _meshes(dev, K, td, tb, tm)
    edits = [(35.0, (0.0, 1.0, 0.0), (0.2, 0.0, 0.1)), (-20.0, (0.2, 1.0, 0.0), (-0.1, 0.05, 0.3)), (0.0, (0.0, 1.0, 0.0), (0.0, 0.0, 0.0))]
    z, corrs, p2f = _native_batch(dev, K, bg_mesh, fg_mesh, edits, S, S)
    sx, sy = O.fov_scales(float(K[1, 1]), S, S)
    F_bg, V_bg = bg_mesh.faces.shape[0], bg_mesh.verts.shape[0]
    faces = torch.cat([bg_mesh.faces, fg_mesh.faces + V_bg]).cpu().numpy()
    colors = torch.cat([bg_mesh.vert_attributes["color"], fg_mesh.vert_attributes["color"]]).cpu().numpy()
    for b, (a, ax, t) in enumerate(edits):
        moved = dt.transform_points(fg_mesh.verts, torch.tensor(a, dtype=torch.float32), torch.tensor(ax), torch.tensor(t))
        verts = torch.cat([bg_mesh.verts, moved]).cpu().numpy()
        o_p2f, _, o_b = O.rasterize_meshes(verts, faces, S, S, sx, sy, 1e-5, True, True, True)
        assert np.array_equal(p2f[b].cpu().numpy(), o_p2f), b
        assert (o_p2f >= F_bg).sum() > 10, b
        world = O.interpolate_face_attributes(verts, faces, o_p2f, o_b)
        assert np.array_equal(z[b].cpu().numpy(), world[..., 2]), b
        carried = O.interpolate_face_attributes(colors, faces, o_p2f, o_b)
        ty, tx = np.nonzero(carried[..., 2] > 0.5)
        src = np.rint((carried[ty, tx, :2] * np.array([S - 1, S - 1], np.float32)).astype(np.float32)).astype(np.int64)
        expect = np.stack([src[:, 0], src[:, 1], tx, ty], -1).astype(np.int64)
        assert np.array_equal(corrs[b].numpy(), expect), b


@pytest.mark.parametrize("scene", SCENES)
def test_real_scene_batch(dev, K, scene):
    """Each photogen scene's edits (its transforms.json) as ONE batch against per-edit transform_depth(..., 'mesh')."""
    from diffusionhandles_b200 import depth_transform as dt
    depth, _, mask = GET(scene)
    bg2 = photogen_filled_bg(scene, GET)
    td, tb, tm = (torch.from_numpy(a).to(dev)[None, None] for a in (depth, bg2, mask))
    edits = [(e["rotation_angle"], torch.tensor(e["rotation_axis"]), torch.tensor(e["translation"])) for e in META[scene]["edits"].values()]
    disp, corrs = dt.transform_depth_mesh_batch(td, tb, tm, K, *map(list, zip(*edits)))
    assert disp.shape == (len(edits), 1, 512, 512)
    for b, (a, ax, t) in enumerate(edits):
        d1, c1 = dt.transform_depth(td, tb, tm, K, rot_angle=a, rot_axis=ax, translation=t, depth_transform_mode="mesh")
        assert _bits_equal(disp[b:b + 1], d1) and torch.equal(corrs[b], c1), (scene, b)


def test_edges(dev, K):
    """An empty mask, a mask with pixels but no complete 2x2 block (vertices, no faces) and use_input_depth_normalization."""
    from diffusionhandles_b200 import depth_transform as dt
    S = 32
    td, tb, tm = _scene(dev, S, S, 72)
    edits = EDITS[:3]
    disp, corrs = _batch_vs_singles(td, tb, torch.zeros_like(tm), K, edits)
    assert all(c.shape == (0, 4) for c in corrs)
    diag = torch.zeros_like(tm)
    idx = torch.arange(4, 28, device=dev)
    diag[0, 0, idx, idx] = 1.0                                     # a diagonal line: no 2x2 block is complete
    from diffusionhandles_b200.depth_transform import depth_to_mesh
    fg = depth_to_mesh(td, K, mask=diag[0, 0] > 0.5)
    assert fg.verts.shape[0] == 24 and fg.faces.shape[0] == 0
    disp, corrs = _batch_vs_singles(td, tb, diag, K, edits)
    assert all(c.shape == (0, 4) for c in corrs)
    _batch_vs_singles(td, tb, tm, K, EDITS[:4], unn=True)
    _batch_vs_singles(td, tb, tm, K, EDITS[:4], unn=False)


def test_facade_edit_geometry_batch(dev, K):
    from diffusionhandles_b200 import DiffusionHandles
    from diffusionhandles_b200.guided_stable_diffuser import GuidedStableDiffuser
    conf = SimpleNamespace(guided_diffuser=None, depth_transform_mode='mesh')
    dh = DiffusionHandles(conf, diffuser=SimpleNamespace(get_depth_intrinsics=GuidedStableDiffuser.get_depth_intrinsics))
    td, tb, tm = _scene(dev, 48, 48, 73)
    angles, axes, shifts = (list(x) for x in zip(*EDITS[:5]))
    disp, corrs = dh.edit_geometry_batch(td, tm, tb, angles, axes, shifts)
    for b in range(5):
        d1, c1 = dh.edit_geometry(td, tm, tb, angles[b], axes[b], shifts[b])
        assert _bits_equal(disp[b:b + 1], d1) and torch.equal(corrs[b], c1), b


def test_transform_foreground_batch_mesh_mode(dev, golden_pc):
    """transform_foreground_batch in mesh mode with an injected tiny diffuser: batched mesh geometry, then the batched guided
    loop; each edit against transform_foreground."""
    from test_loss_batch_gpu import _PerSample, _tiny
    from diffusionhandles_b200 import DiffusionHandles
    from diffusionhandles_b200.depth_transform import transform_depth
    meta, g = golden_pc
    m = meta["cfg1"]
    T = 3
    conf, unet, gsd, gen, latents0, _, cond, uncond = _tiny(dev, T)
    conf.save_denoising_steps = False
    gsd.unet = _PerSample(unet)
    dh = DiffusionHandles(SimpleNamespace(guided_diffuser=conf, depth_transform_mode='mesh'), diffuser=gsd).to(dev)
    depth, bg, mask = O.synthetic_scene(**m["scene"])
    td, tb, tm = (torch.from_numpy(a).to(dev)[None, None] for a in (depth, bg, mask))
    acts = [torch.randn((T, c, s, s), generator=gen, device=dev) for c, s in ((6, 32), (5, 64), (4, 64))]
    angles = [m["angle"], 10.0]
    axes = [torch.tensor(m["axis"]), torch.tensor([1.0, 0.0, 0.0])]
    shifts = [torch.tensor(m["translation"]), torch.tensor(m["translation"]) * 0.5]
    images, disp = dh.transform_foreground_batch(td, cond, tm, tb, uncond, latents0, acts, angles, axes, shifts)
    assert disp.shape == (2, 1, 512, 512) and images.shape == (2, 4, 64, 64)
    K = gsd.get_depth_intrinsics(device=dev)
    for e in range(2):
        d1, _ = transform_depth(td, tb, tm, K, angles[e], axes[e], shifts[e], depth_transform_mode="mesh")
        assert _bits_equal(disp[e:e + 1], d1), e
        img, d2 = dh.transform_foreground(td, cond, tm, tb, uncond, latents0, acts, rot_angle=angles[e], rot_axis=axes[e],
                                          translation=shifts[e])
        assert _bits_equal(d2, d1)
        assert torch.allclose(images[e:e + 1], img, rtol=1e-5, atol=1e-5 * float(img.abs().max())), (e, float((images[e] - img[0]).abs().max()))
