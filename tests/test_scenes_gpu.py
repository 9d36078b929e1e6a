"""GPU (-m gpu): edits of several scenes in one call.  Every edit must come out bit for bit as its own scene's call gives it:
transform_depth_pc_scenes against transform_depth (and the reference's correspondence hashes), transform_depth_mesh_scenes /
dh_edit_mesh_scenes against transform_depth_mesh_batch / dh_edit_mesh_batch on the edit's scene, set_foreground_scenes against
set_foreground, per-edit identity lists in the batched loss against the stacked form, and transform_foreground_scenes against
transform_foreground of each edit's scene."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import dh_oracle as O
from helpers import load_photogen, photogen_filled_bg, sha
from test_mesh_batch_gpu import EDITS, _bits_equal, _meshes, _native_batch, _scene

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


@pytest.fixture(scope="module")
def photogen(dev):
    """The 20 scenes as (S,1,512,512) planes (background: the reference's set_foreground, by the oracle) and their 90 edits as
    (scene_index, angles, axes, translations)."""
    depths, bgs, masks, index, angles, axes, shifts = [], [], [], [], [], [], []
    for s, scene in enumerate(SCENES):
        depth, _, mask = GET(scene)
        depths.append(depth)
        bgs.append(photogen_filled_bg(scene, GET))
        masks.append(mask)
        for e in META[scene]["edits"].values():
            index.append(s)
            angles.append(e["rotation_angle"])
            axes.append(torch.tensor(e["rotation_axis"]))
            shifts.append(torch.tensor(e["translation"]))
    planes = tuple(torch.from_numpy(np.stack(a)).to(dev)[:, None] for a in (depths, bgs, masks))
    return planes, (index, angles, axes, shifts)


def _refs():
    return [e for scene in SCENES for e in META[scene]["edits"].values()]


def test_photogen_pc_scenes(dev, K, photogen):
    """All 90 edits of the 20 scenes in ONE transform_depth_pc_scenes call: the reference's correspondences, and each disparity
    equal to transform_depth on its scene."""
    from diffusionhandles_b200 import depth_transform as dt
    (d, b, m), (index, angles, axes, shifts) = photogen
    assert len(index) == 90
    disp, corrs = dt.transform_depth_pc_scenes(d, b, m, K, index, angles, axes, shifts)
    assert disp.shape == (90, 1, 512, 512) and len(corrs) == 90
    for e, ref in enumerate(_refs()):
        assert corrs[e].shape[0] == ref["n_corr"] and sha(corrs[e].numpy()) == ref["sha_corr"], e
        s = index[e]
        d1, c1 = dt.transform_depth(d[s:s + 1], b[s:s + 1], m[s:s + 1], K, rot_angle=angles[e], rot_axis=axes[e], translation=shifts[e])
        assert _bits_equal(disp[e:e + 1], d1) and torch.equal(corrs[e], c1), e


def _concat_meshes(meshes):
    f32, i32 = torch.float32, torch.int32
    cat = lambda ts: torch.cat(ts).contiguous()                               # noqa: E731
    arrays = (cat([bg.verts.to(f32) for bg, _ in meshes]), cat([bg.faces.to(i32) for bg, _ in meshes]),
              cat([fg.verts.to(f32) for _, fg in meshes]), cat([fg.vert_attributes["color"].to(f32) for _, fg in meshes]),
              cat([fg.faces.to(i32) for _, fg in meshes]))
    counts = [(C.c_int32 * len(meshes))(*[int(x) for x in c]) for c in zip(*[(bg.verts.shape[0], bg.faces.shape[0], fg.verts.shape[0],
                                                                              fg.faces.shape[0]) for bg, fg in meshes])]
    return arrays, counts


def _native_scenes(dev, K, meshes, index, edits, H, W):
    """dh_edit_mesh_scenes over the scene table ``meshes`` [(bg, fg)]: (target_z (B,H,W), [corr rows], pix_to_face (B,H,W))"""
    from diffusionhandles_b200 import _native as N
    from diffusionhandles_b200.renderer import fov_scales
    lib = N.load()
    B, n = len(edits), len(meshes)
    (bv, bf, fv, fc, ff), counts = _concat_meshes(meshes)
    sx, sy = fov_scales(K[1, 1], H, W)
    idx = (C.c_int32 * B)(*index)
    ang = (C.c_float * B)(*[float(a) for a, _, _ in edits])
    axs = (C.c_float * (3 * B))(*[float(v) for _, ax, _ in edits for v in ax])
    trs = (C.c_float * (3 * B))(*[float(v) for _, _, t in edits for v in t])
    z = torch.empty((B, H, W), dtype=torch.float32, device=dev)
    corr = torch.empty((B, H * W, 4), dtype=torch.int64, device=dev)
    nc = torch.empty(B, dtype=torch.int32, device=dev)
    p2f = torch.empty((B, H, W), dtype=torch.int32, device=dev)
    ws_bytes = int(lib.dh_edit_mesh_scenes_workspace_bytes(n, *counts, B, idx, H, W))
    assert ws_bytes > 0
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    N.check(lib.dh_edit_mesh_scenes(n, N.ptr(bv), N.ptr(bf), counts[0], counts[1], N.ptr(fv), N.ptr(fc), N.ptr(ff), counts[2], counts[3],
                                    B, idx, ang, axs, trs, H, W, (C.c_float * 9)(1, 0, 0, 0, 1, 0, 0, 0, 1), (C.c_float * 3)(0, 0, 0),
                                    sx, sy, 1e-5, 1, 1, 1, N.ptr(z), N.ptr(corr), N.ptr(nc), N.ptr(p2f), N.ptr(ws), ws_bytes,
                                    N.stream_handle(dev)), "dh_edit_mesh_scenes")
    counts_out = nc.tolist()
    return z, [corr[b, :c].cpu() for b, c in enumerate(counts_out)], p2f


def _assert_scenes_equal_batches(dev, K, meshes, index, edits, H, W):
    """every edit of one scene call against dh_edit_mesh_batch on its scene with its transform alone"""
    z, corrs, p2f = _native_scenes(dev, K, meshes, index, edits, H, W)
    for e, (s, edit) in enumerate(zip(index, edits)):
        z1, c1, p1 = _native_batch(dev, K, *meshes[s], [edit], H, W)
        assert _bits_equal(z[e], z1[0]), (e, s)
        assert torch.equal(corrs[e], c1[0]), (e, s)
        assert torch.equal(p2f[e], p1[0]), (e, s)
    return z, corrs, p2f


def test_photogen_mesh_scenes(dev, K, photogen):
    """The same 90 edits through transform_depth_mesh_scenes: each equal to transform_depth_mesh_batch on its own scene;
    pix_to_face through the ABI against dh_edit_mesh_batch per scene."""
    from diffusionhandles_b200 import depth_transform as dt
    (d, b, m), (index, angles, axes, shifts) = photogen
    disp, corrs = dt.transform_depth_mesh_scenes(d, b, m, K, index, angles, axes, shifts)
    assert disp.shape == (90, 1, 512, 512)
    for s in range(len(SCENES)):
        edits = [e for e in range(90) if index[e] == s]
        d1, c1 = dt.transform_depth_mesh_batch(d[s:s + 1], b[s:s + 1], m[s:s + 1], K, [angles[e] for e in edits], [axes[e] for e in edits],
                                               [shifts[e] for e in edits])
        for k, e in enumerate(edits):
            assert _bits_equal(disp[e:e + 1], d1[k:k + 1]) and torch.equal(corrs[e], c1[k]), (s, e)
    meshes = [_meshes(dev, K, d[s:s + 1], b[s:s + 1], m[s:s + 1]) for s in range(len(SCENES))]
    edits = [(float(torch.tensor(a, dtype=torch.float32)), ax, t) for a, ax, t in zip(angles, axes, shifts)]
    z, corrs_abi, p2f = _native_scenes(dev, K, meshes, index, edits, 512, 512)
    for s in range(len(SCENES)):
        es = [e for e in range(90) if index[e] == s]
        z1, c1, p1 = _native_batch(dev, K, *meshes[s], [edits[e] for e in es], 512, 512)
        for k, e in enumerate(es):
            assert _bits_equal(z[e], z1[k]) and torch.equal(corrs_abi[e], c1[k]) and torch.equal(p2f[e], p1[k]), (s, e)
            assert torch.equal(corrs_abi[e], corrs[e]), (s, e)


def test_mesh_scenes_edge_cases(dev, K):
    """Non-square images, unsorted and repeated scene indices, a scene without foreground vertices next to ones with large
    foregrounds, and a scene no edit references; the Python call with an empty-mask scene among them."""
    from diffusionhandles_b200 import depth_transform as dt
    H, W = 48, 64
    planes = [_scene(dev, H, W, seed) for seed in (80, 81, 82, 83)]
    empty = (planes[1][0], planes[1][1], torch.zeros_like(planes[1][2]))
    scenes = [planes[0], empty, planes[2], planes[3]]
    meshes = [_meshes(dev, K, *p) for p in scenes]
    assert meshes[1][1].verts.shape[0] == 0 and meshes[0][1].faces.shape[0] > 100
    index = [3, 0, 1, 0, 3, 0, 1]                   # scene 2 unreferenced
    edits = [(a if a is not None else 0.0, ax if ax is not None else (0.0, 1.0, 0.0), t if t is not None else (0.0, 0.0, 0.0))
             for a, ax, t in EDITS[:len(index)]]
    z, corrs, _ = _assert_scenes_equal_batches(dev, K, meshes, index, edits, H, W)
    assert corrs[0].shape[0] > 5 and corrs[5].shape[0] > 5                     # scenes 3 and 0 visible
    assert corrs[2].shape == (0, 4) and corrs[6].shape == (0, 4)                # scene 1 has no foreground
    # the Python call: the empty-mask scene gets the empty-mask result, the others their batch call's bits
    d, b, m = (torch.cat([p[k] for p in scenes]) for k in range(3))
    for unn in (False, True):
        disp, cs = dt.transform_depth_mesh_scenes(d, b, m, K, index, *map(list, zip(*EDITS[:len(index)])), use_input_depth_normalization=unn)
        for e, s in enumerate(index):
            a, ax, t = EDITS[e]
            d1, c1 = dt.transform_depth_mesh_batch(d[s:s + 1], b[s:s + 1], m[s:s + 1], K, [a], [ax], [t], use_input_depth_normalization=unn)
            assert _bits_equal(disp[e:e + 1], d1) and torch.equal(cs[e], c1[0]), (unn, e, s)


def _tie_scene(dev, K):
    """The foreground lying exactly on the background (test_mesh_batch_gpu.test_tie_order_background_wins): 8 x 8 vertices on a
    2^-10 grid, so an identity transform leaves them bit-identical and every foreground face ties with a background face."""
    from diffusionhandles_b200.mesh import Mesh
    S = 32
    _, bg, _ = O.synthetic_scene(S, 70)
    mask = np.zeros((S, S), np.float32)
    mask[12:20, 10:18] = 1.0
    tb, tm = torch.from_numpy(bg).to(dev)[None, None], torch.from_numpy(mask).to(dev)[None, None]
    bg_mesh, fg_mesh = _meshes(dev, K, tb, tb, tm)
    v = torch.round(bg_mesh.verts * 1024) / 1024 + 0.0
    bg_col = bg_mesh.vert_attributes["color"]
    bg_mesh = Mesh(v, bg_mesh.faces)
    bg_mesh.add_vert_attribute("color", bg_col)
    col = fg_mesh.vert_attributes["color"]
    fg_mesh = Mesh(v.reshape(S, S, 3)[torch.from_numpy(mask > 0.5).to(dev)].contiguous(), fg_mesh.faces)
    fg_mesh.add_vert_attribute("color", col)
    return bg_mesh, fg_mesh


def test_mesh_scenes_tie_order_across_scenes(dev, K):
    """Exact background / foreground z-ties in one scene next to another scene: the background of the tie scene wins every
    tie, in every edit of that scene, wherever the edit sits in the batch."""
    S = 32
    tie = _tie_scene(dev, K)
    other = _meshes(dev, K, *_scene(dev, S, S, 84))
    identity = (0.0, (0.0, 1.0, 0.0), (0.0, 0.0, 0.0))
    closer = (0.0, (0.0, 1.0, 0.0), (0.0, 0.0, -0.5))
    index = [1, 0, 1, 0, 1]
    edits = [identity, (35.0, (0.0, 1.0, 0.0), (0.2, 0.0, 0.1)), closer, identity, identity]
    z, corrs, p2f = _assert_scenes_equal_batches(dev, K, [other, tie], index, edits, S, S)
    F_bg = tie[0].faces.shape[0]
    for e in (0, 4):
        assert (p2f[e] < F_bg).all() and corrs[e].shape == (0, 4), e             # the background won every tie
    assert (p2f[2] >= F_bg).sum() > 20 and corrs[2].shape[0] > 20               # moved towards the camera, the foreground wins


def test_set_foreground_scenes(dev, photogen):
    """set_foreground of the 20 scenes in one dilation and one Poisson launch: each equal to set_foreground of its scene."""
    from diffusionhandles_b200 import DiffusionHandles
    (d, _, m), _ = photogen
    b = torch.from_numpy(np.stack([GET(s)[1] for s in SCENES])).to(dev)[:, None]
    dh = DiffusionHandles()
    out = dh.set_foreground_scenes(d, m, b)
    assert out.shape == (20, 1, 512, 512) and out.dtype == torch.float32
    for s in range(len(SCENES)):
        assert _bits_equal(out[s:s + 1], dh.set_foreground(d[s:s + 1], m[s:s + 1], b[s:s + 1])), SCENES[s]


def test_loss_batch_per_edit_identity_lists(dev):
    """Per-edit identity lists (B (C,h,w) tensors, two edits sharing one) give the values and gradients of the stacked
    (B,C,h,w) form bit for bit, in one batch launch; the shared layer form (C,h,w) mixes with them."""
    from test_loss_batch_gpu import _assert_bit_identical, _batch_kernels, _edit_lists, _single, _twin
    from test_loss_plan_and_variants_gpu import _inputs, _pc, variant_cases
    from diffusionhandles_b200 import losses
    name = "two_resized_cnt"
    case = variant_cases()[name]
    grid, shapes, lt = case[0], case[1], case[2]
    curs, origs, fgw, bgw = _inputs(name, shapes)
    gen = torch.Generator().manual_seed(11)
    cur_b = [torch.stack([c, torch.randn(c.shape, generator=gen), c * 0.5]).to(dev) for c in curs]
    idents = [[o.to(dev), torch.randn(o.shape, generator=gen).to(dev)] for o in origs]        # two identities per layer
    lists = [[ids[0], ids[1], ids[0]] for ids in idents]                                      # edits 0 and 2 share identity 0
    stacked = [torch.stack(rows) for rows in lists]
    pcs = [_pc(*_edit_lists(name, case, k), grid) for k in range(3)]
    mixed = [idents[0][0], lists[1], stacked[2]]                                               # shared, list, stacked
    results = []
    for org in (stacked, lists, mixed):
        res = {}
        ran = _batch_kernels(lambda: res.setdefault("b", losses.guidance_loss_and_grad_batch(cur_b, org, pcs, fgw, bgw, bg_loss_type=lt)))
        assert list(ran) == [_twin(case[4])] and len(ran[_twin(case[4])]) == 1, ran
        t, p, g = res["b"]
        results.append((t.cpu().numpy(), p.cpu().numpy(), [x.cpu().numpy() for x in g]))
    singles = [_single(dev, [c[e] for c in cur_b], [rows[e] for rows in lists], pcs[e], fgw, bgw, lt, grid) for e in range(3)]
    _assert_bit_identical(results[1], singles, "per-edit list")
    t0, p0, g0 = results[0]
    t1, p1, g1 = results[1]
    assert np.array_equal(t0, t1, equal_nan=True) and np.array_equal(p0, p1, equal_nan=True)
    assert all(np.array_equal(a, b) for a, b in zip(g0, g1))
    singles = [_single(dev, [c[e] for c in cur_b], [idents[0][0], lists[1][e], stacked[2][e]], pcs[e], fgw, bgw, lt, grid)
               for e in range(3)]
    _assert_bit_identical(results[2], singles, "mixed")
    with pytest.raises(ValueError):
        losses.guidance_loss_and_grad_batch(cur_b, [rows[:2] for rows in lists], pcs, fgw, bgw, bg_loss_type=lt)


def test_transform_foreground_scenes(dev, monkeypatch):
    """Three edits of two synthetic scenes (config-4 recipe) with per-scene prompt embeddings, null-text sequences, initial noises
    and identities, through one transform_foreground_scenes: each edit agrees with transform_foreground on its own scene;
    one batched loss call per guided iteration and no torch.stack of the identities."""
    from test_loss_batch_gpu import _PerSample, _tiny
    from diffusionhandles_b200 import DiffusionHandles, guided_loop
    from diffusionhandles_b200.depth_transform import transform_depth
    from diffusionhandles_b200.synthetic import synthetic_scene
    T = 3
    conf, unet, gsd, gen, latents0, _, cond, uncond = _tiny(dev, T)
    conf.save_denoising_steps = False
    gsd.unet = _PerSample(unet)
    dh = DiffusionHandles(SimpleNamespace(guided_diffuser=conf, depth_transform_mode='pc'), diffuser=gsd).to(dev)
    planes = [tuple(torch.from_numpy(a).to(dev)[None, None] for a in synthetic_scene(512, seed)) for seed in (0, 1)]
    depths, bgs, masks = ([p[k] for p in planes] for k in range(3))
    conds = [cond, -cond]
    unconds = [uncond, uncond * 0.5 + 0.01]
    noises = [latents0, latents0 * 0.9]
    idents = [[torch.randn((T, c, s, s), generator=gen, device=dev) for c, s in ((6, 32), (5, 64), (4, 64))] for _ in range(2)]
    angle = np.linspace(-90.0, 90.0, 16)
    index = [1, 0, 1]
    angles = [float(angle[k]) for k in (3, 5, 9)]
    axes = [torch.tensor([0.0, 1.0, 0.0])] * 3
    shifts = [torch.tensor([0.1 * k - 0.8, 0.0, 0.05 * k]) for k in (3, 5, 9)]
    calls = {"loss": 0, "stack_of_identity": 0}
    ident_storages = {t.untyped_storage().data_ptr() for ids in idents for t in ids}
    real_loss, real_stack = guided_loop.guidance_loss_and_grad_batch, torch.stack

    def loss(*a, **k):
        calls["loss"] += 1
        return real_loss(*a, **k)

    def stack(tensors, *a, **k):
        tensors = list(tensors)
        if any(isinstance(t, torch.Tensor) and t.untyped_storage().data_ptr() in ident_storages for t in tensors):
            calls["stack_of_identity"] += 1
        return real_stack(tensors, *a, **k)
    with monkeypatch.context() as mp:
        mp.setattr(guided_loop, "guidance_loss_and_grad_batch", loss)
        mp.setattr(torch, "stack", stack)
        images, disp = dh.transform_foreground_scenes(depths, conds, masks, bgs, unconds, noises, idents, index, angles, axes, shifts)
    assert calls == {"loss": conf.num_optsteps * conf.guidance_max_step, "stack_of_identity": 0}, calls
    assert disp.shape == (3, 1, 512, 512) and images.shape == (3, 4, 64, 64)
    K = gsd.get_depth_intrinsics(device=dev)
    for e, s in enumerate(index):
        d1, _ = transform_depth(depths[s], bgs[s], masks[s], K, angles[e], axes[e], shifts[e])
        assert _bits_equal(disp[e:e + 1], d1), e
        img, _ = dh.transform_foreground(depths[s], conds[s], masks[s], bgs[s], unconds[s], noises[s], idents[s], rot_angle=angles[e],
                                         rot_axis=axes[e], translation=shifts[e])
        assert torch.allclose(images[e:e + 1], img, rtol=1e-5, atol=1e-5 * float(img.abs().max())), (e, float((images[e] - img[0]).abs().max()))
    # one scene: transform_foreground_batch is the one-scene case and shares the scene's values
    images1, _ = dh.transform_foreground_batch(depths[0], conds[0], masks[0], bgs[0], unconds[0], noises[0], idents[0], angles[:2],
                                               axes[:2], shifts[:2])
    images2, _ = dh.transform_foreground_scenes(depths, conds, masks, bgs, unconds, noises, idents, [0, 0], angles[:2], axes[:2], shifts[:2])
    assert torch.allclose(images1, images2, rtol=1e-5, atol=1e-5 * float(images1.abs().max()))
