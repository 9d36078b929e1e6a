"""CPU: the limits of multi-object edits - the C ABI of dh_edit_splat_objects and its workspace query (fake device pointers, every
call rejected before any CUDA call), the argument errors of the Python entry points, raised before any device work, and the oracle
with one object against transform_depth_pc."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from objects_oracle import sector_masks, transform_depth_pc_objects          # noqa: E402
from oracle import dh_oracle as O                                            # noqa: E402

OK, INVALID, WORKSPACE = 0, -1, -4
FAKE = 0x1000          # 256-byte aligned, never dereferenced
H = W = 16


@pytest.fixture(scope="module")
def lib():
    from diffusionhandles_b200 import _native as N
    try:
        return N.load()
    except N.NativeLibraryError as e:
        pytest.skip(str(e))


def _call(lib, K=2, B=1, labels=FAKE, ws_bytes=None, h=H, w=W, centroid=FAKE):
    from diffusionhandles_b200 import _native as N
    cam = N.dh_camera()
    rigids = (N.dh_rigid * max(B * max(K, 1), 1))()
    if ws_bytes is None:
        ws_bytes = int(lib.dh_edit_objects_workspace_bytes(B, h, w))
    return lib.dh_edit_splat_objects(FAKE, FAKE, FAKE, labels, B, K, h, w, C.byref(cam), rigids, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE,
                                     centroid, None, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, ws_bytes, None)


def test_abi_rejections(lib):
    assert _call(lib, K=0) == INVALID
    assert _call(lib, K=17) == INVALID
    assert _call(lib, K=-1) == INVALID
    assert _call(lib, labels=None) == INVALID
    assert _call(lib, centroid=None) == INVALID
    assert _call(lib, B=0, ws_bytes=1 << 20) == INVALID
    assert _call(lib, h=1) == INVALID
    full = int(lib.dh_edit_objects_workspace_bytes(1, H, W))
    assert _call(lib, ws_bytes=full - 1) == WORKSPACE
    assert _call(lib, K=16, ws_bytes=0) == WORKSPACE


def test_workspace_query(lib):
    assert lib.dh_edit_objects_workspace_bytes(0, H, W) == 0
    assert lib.dh_edit_objects_workspace_bytes(1, 0, W) == 0
    one, four = (int(lib.dh_edit_objects_workspace_bytes(b, H, W)) for b in (1, 4))
    assert one > int(lib.dh_edit_workspace_bytes(1, H, W)) and four > one


def _scene(n_obj=2, S=H):
    depth, bg, mask = O.synthetic_scene(S, 0)
    masks = torch.from_numpy(sector_masks(mask, n_obj))[:, None]
    return torch.from_numpy(depth)[None, None], torch.from_numpy(bg)[None, None], masks


def _intr():
    from diffusionhandles_b200.guided_stable_diffuser import GuidedStableDiffuser
    return GuidedStableDiffuser.get_depth_intrinsics()


def test_python_argument_errors():
    """Every error below is raised for CPU tensors, i.e. before any CUDA call."""
    from diffusionhandles_b200 import depth_transform as dt
    depth, bg, masks = _scene(2)
    K = _intr()
    ax = torch.tensor([0.0, 1.0, 0.0])
    t = torch.zeros(3)
    with pytest.raises(ValueError, match="overlap"):
        over = masks.clone()
        over[1] = over[1] + over[0]
        dt.transform_depth_pc_objects(depth, bg, over, K, [0.0, 0.0], [ax, ax], [t, t])
    with pytest.raises(ValueError):
        dt.transform_depth_pc_objects(depth, bg, masks, K, [0.0], [ax, ax], [t, t])
    with pytest.raises(ValueError):
        dt.transform_depth_pc_objects(depth, bg, masks, K, [0.0, 0.0], [ax], [t, t])
    with pytest.raises(ValueError):
        dt.transform_depth_pc_objects_batch(depth, bg, masks, K, [[0.0, 0.0], [0.0]], [[ax, ax]] * 2, [[t, t]] * 2)
    with pytest.raises(ValueError):
        dt.transform_depth_pc_objects_batch(depth, bg, masks, K, [], [], [])
    many = torch.zeros((17, 1, H, W))
    with pytest.raises(ValueError, match="16"):
        dt.transform_depth_pc_objects(depth, bg, many, K, [0.0] * 17, [ax] * 17, [t] * 17)
    with pytest.raises(ValueError):
        dt.transform_depth_pc_objects(depth, bg, torch.zeros((0, 1, H, W)), K, [], [], [])
    with pytest.raises(ValueError):
        dt.transform_depth_pc_objects(depth, bg, [masks[0:1], masks[1:2, :, :8]], K, [0.0, 0.0], [ax, ax], [t, t])
    rect = torch.zeros((2, 1, H, W + 2))
    rect[0, 0, 2:5, 2:5] = 1
    with pytest.raises(RuntimeError, match="square"):
        dt.transform_depth_pc_objects(torch.ones((1, 1, H, W + 2)), torch.ones((1, 1, H, W + 2)), rect, K, [0.0, 0.0], [ax, ax], [t, t])


def test_empty_union_on_cpu():
    """No object has a pixel: the empty-mask result of transform_depth_pc, without a device."""
    from diffusionhandles_b200 import depth_transform as dt
    depth, bg, masks = _scene(2)
    ax, t = torch.tensor([0.0, 1.0, 0.0]), torch.zeros(3)
    disp, corr = dt.transform_depth_pc_objects(depth, bg, torch.zeros_like(masks), _intr(), [10.0, 0.0], [ax, ax], [t, t])
    ref, ref_corr = dt._empty_mask_result(depth, False)
    assert torch.equal(disp, ref) and corr.shape == (0, 4) and ref_corr.shape == (0, 4)


def test_facade_mesh_mode_rejected():
    from types import SimpleNamespace
    from diffusionhandles_b200 import DiffusionHandles
    from diffusionhandles_b200.diffusion_handles import DEFAULT_CONF
    conf = SimpleNamespace(guided_diffuser=DEFAULT_CONF.guided_diffuser, depth_transform_mode='mesh')
    dh = DiffusionHandles(conf, diffuser=SimpleNamespace(get_depth_intrinsics=lambda device=None: _intr()))
    depth, bg, masks = _scene(2)
    ax, t = torch.tensor([0.0, 1.0, 0.0]), torch.zeros(3)
    with pytest.raises(NotImplementedError):
        dh.edit_geometry_objects(depth, masks, bg, [0.0, 0.0], [ax, ax], [t, t])


def _assert_same(a, b):
    assert set(a) - {"object"} == set(b), (sorted(a), sorted(b))
    for k in b:
        if k == "centroid":
            assert np.array_equal(a[k][0], b[k]), k
        else:
            assert np.array_equal(a[k], b[k], equal_nan=a[k].dtype.kind == "f"), k


def test_oracle_one_object_is_transform_depth_pc(golden_pc):
    """The oracle of K objects with one mask reproduces transform_depth_pc in every intermediate, on the golden configurations
    (the Poisson fill of the first one too)."""
    meta, _ = golden_pc
    Kc = O.get_depth_intrinsics()
    configs = [c for c in meta.values() if isinstance(c, dict) and {"scene", "angle", "axis", "translation"} <= set(c)]
    assert configs
    for i, cfg in enumerate(configs):
        depth, bg, mask = O.synthetic_scene(**cfg["scene"])
        args = (cfg["angle"], cfg["axis"], tuple(float(np.float32(v)) for v in cfg["translation"]))
        kw = dict(use_input_depth_normalization=bool(cfg.get("norm", False)), poisson=i == 0)
        ref = O.transform_depth_pc(depth, bg, mask, Kc, *args, **kw)
        got = transform_depth_pc_objects(depth, bg, mask[None], Kc, [args[0]], [args[1]], [args[2]], **kw)
        _assert_same(got, ref)


@pytest.mark.parametrize("seed", [0, 1])
def test_oracle_one_object_small_scenes(seed):
    """Same on small synthetic scenes, including a transform that clamps points onto border pixels."""
    Kc = O.get_depth_intrinsics()
    depth, bg, mask = O.synthetic_scene(64, seed)
    for args in ((30.0, (0.0, 1.0, 0.0), (0.3, 0.0, 0.2)), (-75.0, (1.0, 0.5, 0.0), (3.0, -2.0, 0.5))):
        t = tuple(float(np.float32(v)) for v in args[2])
        ref = O.transform_depth_pc(depth, bg, mask, Kc, args[0], args[1], t)
        got = transform_depth_pc_objects(depth, bg, mask[None], Kc, [args[0]], [args[1]], [t])
        _assert_same(got, ref)


def test_oracle_one_object_photogen():
    """All 20 photogen scenes x their 90 edits: the oracle with one mask equals transform_depth_pc (without the Poisson fill,
    which is the same function of the same inputs)."""
    from helpers import f32_translation, load_photogen, photogen_filled_bg
    meta, get = load_photogen()
    Kc = O.get_depth_intrinsics()
    n = 0
    for scene in sorted(meta):
        depth, _, mask = get(scene)
        bg = photogen_filled_bg(scene, get)
        for e in meta[scene]["edits"].values():
            args = (e["rotation_angle"], e["rotation_axis"], f32_translation(e["translation"]))
            ref = O.transform_depth_pc(depth, bg, mask, Kc, *args, poisson=False)
            got = transform_depth_pc_objects(depth, bg, mask[None], Kc, [args[0]], [args[1]], [args[2]], poisson=False)
            _assert_same(got, ref)
            n += 1
    assert n == 90
