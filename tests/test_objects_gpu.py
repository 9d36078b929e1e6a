"""GPU: multi-object 'pc' edits (dh_edit_splat_objects, transform_depth_pc_objects[_batch], DiffusionHandles.*_objects).

- K = 1 equals today's single-object edit bit for bit in every intermediate, on the golden configurations and all 90 photogen edits;
- K = 2, 3 and 8 equal the NumPy oracle (tests/objects_oracle.py) bit for bit: centroids, object ids, foreground points, winners,
  depth map, masks, correspondences and raw disparity; the filled disparity to 1e-3 on 0..255;
- a batch of 16 edits equals 16 single calls; the full edit with stand-in models equals guided_inference on the geometry."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from helpers import f32_translation, load_photogen, photogen_filled_bg
from objects_oracle import sector_masks, transform_depth_pc_objects
from oracle import dh_oracle as O

pytestmark = pytest.mark.gpu

META, GET = load_photogen()
SCENES = sorted(META)
KNP = O.get_depth_intrinsics()


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def K(dev):
    from diffusionhandles_b200.guided_stable_diffuser import GuidedStableDiffuser
    return GuidedStableDiffuser.get_depth_intrinsics(device=dev)


def _label_planes(masks: np.ndarray):
    """(n,S,S) disjoint masks -> union fp32 and labels uint8 (k + 1 on object k)."""
    inside = masks != 0
    labels = np.zeros(masks.shape[1:], np.uint8)
    for k in range(masks.shape[0]):
        labels[inside[k]] = k + 1
    return inside.any(0).astype(np.float32), labels


def _run_objects(dev, K, depth, bg, masks, transforms, keep_points=True):
    """The engine on B edits of one scene: transforms[b] = [(angle, axis, translation)] * n objects."""
    from diffusionhandles_b200.engine import get_engine, make_rigid
    B, S = len(transforms), depth.shape[-1]
    union, labels = _label_planes(masks)
    d, b, m, lab = (torch.from_numpy(np.ascontiguousarray(a)).to(dev)[None].expand(B, S, S).contiguous() for a in (depth, bg, union, labels))
    rigids = [make_rigid(a, list(ax), list(t)) for tr in transforms for a, ax, t in tr]
    eng = get_engine(dev, B, S, S, keep_points=keep_points)
    return eng, eng.run_objects(d, b, m, lab, masks.shape[0], K, rigids)


def _snapshot(eng, res):
    """Host copies of every intermediate of a result (the engine's buffers are reused by the next call)."""
    P = eng.P
    out = []
    for e in range(res.B):
        n = int(res.n_fg_host[e])
        snap = dict(n_fg=n, fg_index=res.fg_index[e, :n].cpu().numpy(), pix=res.pix[e, P:P + n].cpu().numpy(),
                    zkey=res.zkey[e, P:P + n].cpu().numpy(), winner=res.winner[e].cpu().numpy().astype(np.int64),
                    winner_src=res.winner_src[e].cpu().numpy(), depth_map=res.depth_map[e].cpu().numpy(),
                    target_mask=res.target_mask[e].cpu().numpy(), cleaned=eng.unpack_bits(res.cleaned_bits)[e].cpu().numpy(),
                    corr=res.correspondences(e).cpu().numpy(), disparity_raw=res.disparity_raw[e].cpu().numpy(),
                    disparity=res.disparity[e].cpu().numpy(), centroid=res.centroid[e].cpu().numpy())
        if res.points is not None:
            snap["points"] = res.points[e, P:P + n].cpu().numpy()
        if res.object_id is not None:
            snap["object"] = res.object_id[e, :n].cpu().numpy().astype(np.int64)
        out.append(snap)
    return out


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8) if a.dtype.kind == "f" else a


def _assert_snap_equal(got, ref, what):
    for k in ref:
        if k in ("object",):
            continue
        if k == "centroid":
            assert np.array_equal(_bits(got[k].reshape(-1)), _bits(ref[k].reshape(-1))), (what, k)
        elif isinstance(ref[k], np.ndarray):
            assert got[k].shape == ref[k].shape and np.array_equal(_bits(got[k]), _bits(ref[k])), (what, k)
        else:
            assert got[k] == ref[k], (what, k)


def _run_single(dev, K, depth, bg, mask, transforms):
    from diffusionhandles_b200.engine import get_engine, make_rigid
    B, S = len(transforms), depth.shape[-1]
    d, b, m = (torch.from_numpy(np.ascontiguousarray(a)).to(dev)[None].expand(B, S, S).contiguous() for a in (depth, bg, mask))
    eng = get_engine(dev, B, S, S, keep_points=True)
    return eng, eng.run(d, b, m, K, [make_rigid(a, list(ax), list(t)) for a, ax, t in transforms])


def _assert_one_object_is_single(dev, K, depth, bg, mask, transforms, what):
    eng, res = _run_single(dev, K, depth, bg, mask, transforms)
    ref = _snapshot(eng, res)
    eng, res = _run_objects(dev, K, depth, bg, (mask != 0)[None].astype(np.float32), [[t] for t in transforms])
    got = _snapshot(eng, res)
    for e in range(len(transforms)):
        assert (got[e]["object"] == 0).all()
        _assert_snap_equal(got[e], ref[e], (what, e))


def test_one_object_is_single_edit_golden(dev, K, golden_pc):
    """K = 1 against EditEngine.run on the golden configurations, every intermediate bit for bit."""
    meta, _ = golden_pc
    configs = [c for c in meta.values() if isinstance(c, dict) and {"scene", "angle", "axis", "translation"} <= set(c)]
    for cfg in configs:
        depth, bg, mask = O.synthetic_scene(**cfg["scene"])
        t = f32_translation(cfg["translation"])
        _assert_one_object_is_single(dev, K, depth, bg, mask, [(cfg["angle"], cfg["axis"], t)], cfg)


def test_one_object_is_single_edit_photogen(dev, K):
    """K = 1 against EditEngine.run on all 90 photogen edits (one batch per scene), and the public call against
    transform_depth_pc on the first edit of every scene."""
    from diffusionhandles_b200 import depth_transform as dt
    n = 0
    for scene in SCENES:
        depth, _, mask = GET(scene)
        bg = photogen_filled_bg(scene, GET)
        edits = [(e["rotation_angle"], e["rotation_axis"], f32_translation(e["translation"])) for e in META[scene]["edits"].values()]
        _assert_one_object_is_single(dev, K, depth, bg, mask, edits, scene)
        n += len(edits)
        a, ax, t = edits[0]
        td, tb, tm = (torch.from_numpy(x).to(dev)[None, None] for x in (depth, bg, mask))
        d1, c1 = dt.transform_depth_pc(td, tb, tm, K, a, torch.tensor(ax), torch.tensor(t))
        d2, c2 = dt.transform_depth_pc_objects(td, tb, tm, K, [a], [torch.tensor(ax)], [torch.tensor(t)])
        assert torch.equal(d1.view(torch.int32), d2.view(torch.int32)) and torch.equal(c1, c2), scene
    assert n == 90


def _same_f32(a, b):
    """Bit for bit, except that any NaN matches any NaN (the device and NumPy produce NaNs of different signs)."""
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(_bits(np.where(na, 0, a)), _bits(np.where(nb, 0, b)))


def _assert_matches_oracle(snap, o, S, what):
    P = S * S
    n = snap["n_fg"]
    assert n == len(o["fg_index"]) and np.array_equal(snap["fg_index"], o["fg_index"]), what
    assert np.array_equal(snap["object"], o["object"]), what
    assert np.array_equal(snap["centroid"], o["centroid"], equal_nan=True), (what, snap["centroid"], o["centroid"])   # NaN: empty
    assert np.array_equal(_bits(snap["points"]), _bits(o["points"][P:])), what
    assert np.array_equal(snap["pix"], o["pix"][P:]), what
    assert np.array_equal(snap["winner"], o["winner"]), what
    assert np.array_equal(_bits(snap["depth_map"]), _bits(o["depth_map"])), what
    assert np.array_equal(snap["target_mask"].astype(bool), o["target_mask"]), what
    assert np.array_equal(snap["cleaned"].astype(bool), o["cleaned"]), what
    assert np.array_equal(snap["corr"], o["correspondences"]), what
    assert _same_f32(snap["disparity_raw"], o["disparity_raw"]), what
    if "disparity" in o:
        assert np.abs(snap["disparity"] - o["disparity"]).max() <= 1e-3, what


def _check_cases(dev, K, depth, bg, masks, transforms, what, poisson_first=True):
    eng, res = _run_objects(dev, K, depth, bg, masks, transforms)
    snaps = _snapshot(eng, res)
    for e, tr in enumerate(transforms):
        o = transform_depth_pc_objects(depth, bg, masks, KNP, [a for a, _, _ in tr], [ax for _, ax, _ in tr], [t for _, _, t in tr],
                                       poisson=poisson_first and e == 0)
        _assert_matches_oracle(snaps[e], o, depth.shape[-1], (what, e))
    return snaps


def _recipe(k):
    """Transform k of the config-4 recipe: angle linspace(-90, 90, 16)[k] about +y, translation (0.1 k - 0.8, 0, 0.05 k)."""
    angle = np.linspace(-90.0, 90.0, 16)
    return float(angle[k % 16]), (0.0, 1.0, 0.0), f32_translation((0.1 * (k % 16) - 0.8, 0.0, 0.05 * (k % 16)))


@pytest.mark.parametrize("n_obj", [2, 3, 8])
def test_sectors_against_oracle(dev, K, n_obj):
    """The config-1 disc split into angular sectors, each sector with its own config-4 transform."""
    depth, bg, mask = O.synthetic_scene(256, 0)
    masks = sector_masks(mask, n_obj)
    transforms = [[_recipe(3 * b + k) for k in range(n_obj)] for b in range(2)]
    _check_cases(dev, K, depth, bg, masks, transforms, ("sectors", n_obj))


def test_photogen_two_objects_against_oracle(dev, K):
    """Photogen masks split into two objects, driven by two of the scene's own transforms (four scenes)."""
    for scene in SCENES[:4]:
        depth, _, mask = GET(scene)
        bg = photogen_filled_bg(scene, GET)
        edits = [(e["rotation_angle"], e["rotation_axis"], f32_translation(e["translation"])) for e in META[scene]["edits"].values()]
        masks = sector_masks(mask, 2)
        tr = [[edits[0], edits[-1]]]
        _check_cases(dev, K, depth, bg, masks, tr, scene, poisson_first=False)


def _two_discs(S=128, bad_bg=False):
    """Two discs at one depth in front of a plane; optionally a background with subnormal, tiny and huge depths (odd points)."""
    yy, xx = np.mgrid[0:S, 0:S]
    a = ((xx - 0.3 * S) ** 2 + (yy - 0.5 * S) ** 2 <= (0.12 * S) ** 2)
    b = ((xx - 0.7 * S) ** 2 + (yy - 0.5 * S) ** 2 <= (0.12 * S) ** 2)
    bg = np.full((S, S), 4.0, np.float32)
    depth = bg.copy()
    depth[a | b] = 2.0
    if bad_bg:
        bg[5:9, 5:40] = 1e-40
        bg[100:104, 10:20] = 5e-31
        bg[60, 60:70] = 1e35
    return depth, bg, np.stack([a, b]).astype(np.float32)


def test_discs_into_each_other(dev, K):
    """Two discs translated into each other at one depth: cross-object occlusion decided by exact z ties (lower source raster
    index wins); a third object that does not move, an empty fourth object, and an object pushed off-screen."""
    depth, bg, ab = _two_discs()
    S = depth.shape[0]
    z = (0.0, 1.0, 0.0)
    # each disc moves 0.2 S pixels at depth 2 (u = (-X k0 / Z / 2 + 1 / 2)(S - 1)): in one edit towards the other, onto it
    shift = float(np.float32(0.2 * S * 2.0 * 2.0 / (float(KNP[0, 0]) * (S - 1))))
    masks = np.concatenate([ab, np.zeros((2, S, S), np.float32)])
    masks[2, 10:20, 60:70] = 1.0                                           # a small third object
    depth[10:20, 60:70] = 3.0
    transforms = [[(0.0, z, (shift, 0.0, 0.0)), (0.0, z, (-shift, 0.0, 0.0)), (0.0, z, (0.0, 0.0, 0.0)), (45.0, z, (1.0, 0.0, 0.0))],
                  [(0.0, z, (-shift, 0.0, 0.0)), (0.0, z, (shift, 0.0, 0.0)), (0.0, z, (5.0, -5.0, 0.0)), (10.0, z, (0.0, 0.0, 0.0))]]
    snaps = _check_cases(dev, K, depth, bg, masks, transforms, "discs")
    assert np.isnan(snaps[0]["centroid"][3]).all()                        # the empty object
    # in one of the edits the discs meet: fewer foreground winners than foreground points
    assert min((s["winner"] >= S * S).sum() for s in snaps) < (masks[:2] != 0).sum()


def test_odd_background_against_oracle(dev, K):
    """A background with subnormal, tiny and huge depths (the generic per-point path) under a three-object edit."""
    depth, bg, ab = _two_discs(bad_bg=True)
    S = depth.shape[0]
    masks = np.concatenate([ab, np.zeros((1, S, S), np.float32)])
    masks[2, 100:110, 100:120] = 1.0
    transforms = [[_recipe(2), _recipe(9), _recipe(14)]]
    _check_cases(dev, K, depth, bg, masks, transforms, "odd background", poisson_first=False)   # (1 / 1e-40 is inf: no fill)


def test_batch_equals_singles(dev, K):
    """A batch of 16 edits of three objects equals 16 single calls bit for bit (public entry points)."""
    from diffusionhandles_b200 import depth_transform as dt
    depth, bg, mask = O.synthetic_scene(256, 0)
    masks = torch.from_numpy(sector_masks(mask, 3)).to(dev)[:, None]
    td, tb = (torch.from_numpy(a).to(dev)[None, None] for a in (depth, bg))
    ang = [[_recipe(b + 5 * k)[0] for k in range(3)] for b in range(16)]
    axs = [[torch.tensor(_recipe(b + 5 * k)[1]) for k in range(3)] for b in range(16)]
    tra = [[torch.tensor(_recipe(b + 5 * k)[2]) for k in range(3)] for b in range(16)]
    disp, corrs = dt.transform_depth_pc_objects_batch(td, tb, masks, K, ang, axs, tra)
    assert disp.shape == (16, 1, 256, 256) and len(corrs) == 16
    for b in range(16):
        d1, c1 = dt.transform_depth_pc_objects(td, tb, [masks[k:k + 1] for k in range(3)], K, ang[b], axs[b], tra[b])
        assert torch.equal(disp[b:b + 1].view(torch.int32), d1.view(torch.int32)) and torch.equal(corrs[b], c1), b


def test_transform_foreground_objects(dev):
    """The full edit with the tiny stand-in models: transform_foreground_objects equals guided_inference called on the geometry of
    edit_geometry_objects; with one object it equals transform_foreground."""
    from test_loss_batch_gpu import _tiny
    from diffusionhandles_b200 import DiffusionHandles
    from diffusionhandles_b200.synthetic import synthetic_scene
    T = 3
    conf, unet, gsd, gen, latents0, _, cond, uncond = _tiny(dev, T)
    conf.save_denoising_steps = False
    dh = DiffusionHandles(SimpleNamespace(guided_diffuser=conf, depth_transform_mode='pc'), diffuser=gsd).to(dev)
    depth, bg, mask = (torch.from_numpy(a).to(dev)[None, None] for a in synthetic_scene(512, 0))
    masks = torch.from_numpy(sector_masks(mask[0, 0].cpu().numpy(), 2)).to(dev)[:, None]
    ident = [torch.randn((T, c, s, s), generator=gen, device=dev) for c, s in ((6, 32), (5, 64), (4, 64))]
    ang = [_recipe(3)[0], _recipe(9)[0]]
    axs = [torch.tensor(_recipe(3)[1]), torch.tensor(_recipe(9)[1])]
    tra = [torch.tensor(_recipe(3)[2]), torch.tensor(_recipe(9)[2])]
    img, disp = dh.transform_foreground_objects(depth, cond, masks, bg, uncond, latents0, ident, ang, axs, tra)
    d2, corr = dh.edit_geometry_objects(depth, masks, bg, ang, axs, tra)
    assert torch.equal(disp.view(torch.int32), d2.view(torch.int32))
    with torch.no_grad():
        ref = gsd.guided_inference(latents=latents0, depth=d2, uncond_embeddings=uncond, prompt=cond, activations_orig=ident,
                                   correspondences=corr, save_denoising_steps=False)
    assert torch.allclose(img, ref, rtol=1e-5, atol=1e-5 * float(ref.abs().max()))
    img1, disp1 = dh.transform_foreground_objects(depth, cond, mask, bg, uncond, latents0, ident, [ang[0]], [axs[0]], [tra[0]])
    img0, disp0 = dh.transform_foreground(depth, cond, mask, bg, uncond, latents0, ident, rot_angle=ang[0], rot_axis=axs[0],
                                          translation=tra[0])
    assert torch.equal(disp1.view(torch.int32), disp0.view(torch.int32))
    assert torch.allclose(img1, img0, rtol=1e-5, atol=1e-5 * float(img0.abs().max()))
