"""GPU (``-m gpu``): batched general-patch guidance losses (``dh_guidance_loss_patch_batch`` through
``losses.guidance_loss_and_grad_batch``).  Every input that the single-edit call sends to the general patch kernel (patch_size > 1,
'local_avg' on resized layers, maps smaller than grid/8, map areas that are not a multiple of 4) runs B edits as one main launch
and one finish launch per 16 edits, and every edit must give the bits its own single-edit call gives."""
import os
import re
import sys
from collections import Counter

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.dirname(os.path.abspath(__file__))):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from test_loss_batch_gpu import _assert_bit_identical, _edit_lists, _tiny  # noqa: E402
from test_loss_plan_and_variants_gpu import _check_against_oracle, _inputs, _lists, _pc, variant_cases  # noqa: E402

gpu = pytest.mark.gpu
_PATCH = [n for n, c in variant_cases().items() if c[4] == "loss_patch_kernel"]
_KERNEL = re.compile(r"\b(loss_patch(?:_finish)?(?:_batch)?_kernel)\b")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _patch_launches(fn):
    """Counter of the patch kernels launched inside fn() ('loss_patch_kernel', 'loss_patch_batch_kernel', and their finish
    kernels), from the kernel records of a torch.profiler trace, and the grid sizes of the batch launches."""
    import json
    import tempfile
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    found, grids = Counter(), []
    for e in events:
        m = _KERNEL.search(e.get("name", "")) if e.get("cat") == "kernel" else None
        if m:
            found[m.group(1)] += 1
            if m.group(1) == "loss_patch_batch_kernel":
                grids.append(e.get("args", {}).get("grid", [0])[0])
    return found, grids


def _expected(n_edits):
    """One edit runs the single-edit kernels; every started chunk of 16 edits one batch launch and one batch finish."""
    if n_edits == 1:
        return Counter({"loss_patch_kernel": 1, "loss_patch_finish_kernel": 1})
    chunks = -(-n_edits // 16)
    return Counter({"loss_patch_batch_kernel": chunks, "loss_patch_finish_batch_kernel": chunks})


def _to_np(res):
    t, p, g = res
    return t.cpu().numpy(), p.cpu().numpy(), [x.cpu().numpy() for x in g]


def _identities(origs, n_edits, mode, dev, gen):
    """The recorded activations in one of the three accepted forms, and the (C,h,w) tensor of edit e of layer l."""
    if mode == "shared":
        org = [o.to(dev) for o in origs]
        return org, lambda l, e: org[l]
    others = [[torch.randn(o.shape, generator=gen).to(dev) for _ in range(n_edits - 1)] for o in origs]
    if mode == "stacked":
        org = [torch.stack([o.to(dev)] + oth) for o, oth in zip(origs, others)]
        return org, lambda l, e: org[l][e]
    # a per-edit list: edit e reads tensor e // 2, so consecutive edits share one identity
    per = [[o.to(dev)] + oth for o, oth in zip(origs, others)]
    org = [[per[l][e // 2] for e in range(n_edits)] for l in range(len(origs))]
    return org, lambda l, e: org[l][e]


def _run(dev, name, grid, shapes, lt, patch, lists, n_edits, mode="shared", fgw=None, bgw=None):
    """guidance_loss_and_grad_batch over n_edits edits and guidance_loss_and_grad on every edit alone.  Edit 0 has the inputs
    of _inputs(name); lists[e] are the five cell lists of edit e."""
    from diffusionhandles_b200 import losses
    curs, origs, fgw0, bgw0 = _inputs(name, shapes)
    fgw, bgw = fgw0 if fgw is None else fgw, bgw0 if bgw is None else bgw
    gen = torch.Generator().manual_seed(7)
    cur_b = [torch.stack([c] + [torch.randn(c.shape, generator=gen) for _ in range(n_edits - 1)]).to(dev) for c in curs]
    org, org_of = _identities(origs, n_edits, mode, dev, gen)
    pcs = [_pc(*lists[e], grid) for e in range(n_edits)]
    kw = dict(bg_loss_type=lt, activations_size=(grid, grid), patch_size=patch)
    res = {}
    ran, grids = _patch_launches(lambda: res.setdefault("b", losses.guidance_loss_and_grad_batch(cur_b, org, pcs, fgw, bgw, **kw)))
    singles = [_to_np(losses.guidance_loss_and_grad([c[e] for c in cur_b], [org_of(l, e) for l in range(len(shapes))], pcs[e],
                                                    fgw, bgw, **kw)) for e in range(n_edits)]
    assert ran == _expected(n_edits), (name, n_edits, ran)
    assert all(0 < g <= torch.cuda.get_device_properties(dev).multi_processor_count for g in grids), grids
    return _to_np(res["b"]), singles


def _three(grid, binary, own):
    """Edit 0: `own`; edit 1: lists of another seed; edit 2: no foreground pair."""
    other = _lists(np.random.default_rng(101), grid, binary)
    e = np.zeros(0, np.int64)
    return [own, other, (e, e) + tuple(other[2:])]


@gpu
@pytest.mark.parametrize("name", _PATCH)
def test_every_patch_case_as_a_batch_of_three(dev, name):
    """Every general-patch case of the variant table as a batch of three edits (its lists, another seed's, an empty foreground
    list): one batch launch and one finish launch, every edit its own bits, NaN foreground terms for the empty edit."""
    case = variant_cases()[name]
    grid, shapes, lt, patch = case[:4]
    lists = [_edit_lists(name, case, k) for k in range(3)]
    batch, singles = _run(dev, name, grid, shapes, lt, patch, lists, 3)
    _assert_bit_identical(batch, singles, name)
    assert np.isnan(batch[1][2][0::2]).all() and not np.isnan(batch[1][2][1::2]).any()
    assert all(np.isfinite(g[2]).all() for g in batch[2])
    if name == "patch3_resized":
        _check_against_oracle(name, case, float(batch[0][0]), batch[1][0], [g[0] for g in batch[2]])


@gpu
def test_empty_foreground_edit_has_a_zero_gradient(dev):
    """With the background weights at 0 the edit without foreground pairs gets exactly zero gradients (the mean over nothing
    scatters nothing back), next to edits that have pairs."""
    name = "patch3_resized"
    case = variant_cases()[name]
    grid, shapes, lt, patch = case[:4]
    batch, singles = _run(dev, name, grid, shapes, lt, patch, [_edit_lists(name, case, k) for k in range(3)], 3,
                          bgw=[0.0] * len(shapes))
    _assert_bit_identical(batch, singles, name)
    assert all(not g[2].any() for g in batch[2]) and all(g[0].any() for g in batch[2])


# name -> (grid, layer shapes, background type, patch, binary lists)
_SHAPES = {
    "patch2_local": (64, [(3, 64, 64), (2, 32, 32)], "local_avg", 2, True),
    "patch3_global": (64, [(3, 64, 64), (2, 32, 32)], "global_avg", 3, False),
    "patch31_local": (64, [(3, 64, 64), (2, 32, 32)], "local_avg", 31, True),
    "patch31_global": (64, [(2, 64, 64)], "global_avg", 31, False),
    "down_to_4x4": (64, [(3, 4, 4), (2, 8, 8), (2, 16, 16), (2, 64, 64)], "global_avg", 1, False),
    "down_to_4x4_local": (64, [(3, 4, 4), (2, 64, 64)], "local_avg", 1, True),
    "odd_9x9": (64, [(4, 9, 9)], "global_avg", 1, True),
    "odd_63x63": (64, [(3, 63, 63), (2, 64, 64)], "local_avg", 1, False),
    "grid48_patch2": (48, [(4, 48, 48), (3, 24, 24)], "local_avg", 2, True),
    "grid48_odd": (48, [(3, 47, 47), (2, 5, 5)], "global_avg", 1, False),
    "sd2_local_patch1": (64, [(1280, 32, 32), (640, 64, 64), (320, 64, 64)], "local_avg", 1, True),
}


@gpu
@pytest.mark.parametrize("name", list(_SHAPES))
def test_patch_sizes_loss_types_and_shapes(dev, name):
    """Patch 2, 3 and 31, both background types, resized layers down to 4 x 4, odd map areas, grid 48, and the SD2 shapes with
    'local_avg' and patch 1 (the reference's local_avg sweep with all three layers evaluated), as batches of three."""
    grid, shapes, lt, patch, binary = _SHAPES[name]
    batch, singles = _run(dev, name, grid, shapes, lt, patch, _three(grid, binary, _lists(np.random.default_rng(7), grid, binary)), 3)
    _assert_bit_identical(batch, singles, name)


@gpu
@pytest.mark.parametrize("n_edits", [1, 2, 16, 20])
def test_patch_batch_sizes(dev, n_edits):
    """B = 1 (the single-edit kernels, no batch kernel), 2, 16 (one launch) and 20 (16 + 4), with per-edit identities."""
    name = "patch3_resized"
    case = variant_cases()[name]
    grid, shapes, lt, patch = case[:4]
    lists = [_edit_lists(name, case, k % 3) for k in range(n_edits)]
    batch, singles = _run(dev, name, grid, shapes, lt, patch, lists, n_edits, mode="stacked")
    _assert_bit_identical(batch, singles, n_edits)


@gpu
@pytest.mark.parametrize("mode", ["shared", "stacked", "list"])
def test_patch_batch_identity_forms(dev, mode):
    """Recorded activations shared by every edit (C,h,w), one per edit (B,C,h,w), or a per-edit list whose edits share
    tensors pairwise: all read in place, every edit its own bits."""
    name = "grid63_patch3"
    case = variant_cases()[name]
    grid, shapes, lt, patch = case[:4]
    batch, singles = _run(dev, name, grid, shapes, lt, patch, [_edit_lists(name, case, k % 3) for k in range(5)], 5, mode=mode)
    _assert_bit_identical(batch, singles, mode)


@gpu
def test_two_calls_on_one_workspace(dev):
    """ProcessedCorrespondences cache their plans, so two batched calls in a row use one cached runner and one workspace, and
    give the same bits as each other and as the single-edit calls between them."""
    from diffusionhandles_b200 import losses
    from diffusionhandles_b200.guided_stable_diffuser import ProcessedCorrespondences
    name = "patch3_native"
    case = variant_cases()[name]
    grid, shapes, lt, patch = case[:4]
    curs, origs, fgw, bgw = _inputs(name, shapes)
    gen = torch.Generator().manual_seed(9)
    cur_b = [torch.stack([c, torch.randn(c.shape, generator=gen), -c]).to(dev) for c in curs]
    org = [o.to(dev) for o in origs]
    pcs = []
    for k in range(3):
        pc = ProcessedCorrespondences(_pc(*_edit_lists(name, case, k), grid))
        pc.grid, pc.device_lists = grid, losses._lists(dict(pc), grid, dev)
        pcs.append(pc)
    kw = dict(bg_loss_type=lt, activations_size=(grid, grid), patch_size=patch)
    first = _to_np(losses.guidance_loss_and_grad_batch(cur_b, org, pcs, fgw, bgw, **kw))
    plan0 = losses._plan_for(pcs[0], grid, dev)
    runners = [r for k, r in plan0._runners.items() if k[0] == "batch"]
    assert len(runners) == 1
    ws = runners[0][3]
    singles = [_to_np(losses.guidance_loss_and_grad([c[e] for c in cur_b], org, pcs[e], fgw, bgw, **kw)) for e in range(3)]
    second = _to_np(losses.guidance_loss_and_grad_batch(cur_b, org, pcs, fgw, bgw, **kw))
    assert [r for k, r in plan0._runners.items() if k[0] == "batch"] == runners and runners[0][3] is ws
    for what, res in (("first", first), ("second", second)):
        _assert_bit_identical(res, singles, what)


@gpu
def test_guided_denoise_batch_local_avg_all_layers(dev, golden_pc, monkeypatch):
    """The reference's 'local_avg' schedule evaluated faithfully (skip_zero_weight_layers=False, the resized layer included):
    every guided iteration of guided_denoise_batch is one batch launch, and each edit follows its own guided_denoise run."""
    from diffusionhandles_b200 import guided_loop
    from diffusionhandles_b200.guided_loop import DDIMSchedule, guided_denoise, guided_denoise_batch
    meta, g = golden_pc
    T, B = 3, 3
    conf, unet, gsd, gen, latents0, depth, cond, uncond = _tiny(dev, T)
    acts_orig = [torch.randn((T, c, s, s), generator=gen, device=dev) for c, s in ((6, 32), (5, 64), (4, 64))]
    corr = torch.from_numpy(g["cfg1/corr"].astype(np.int64))
    corrs = [corr, corr.flip(0)[: len(corr) // 2], torch.cat([corr[:, :2], corr[:, :2]], 1)]
    pcs = [gsd.process_correspondences(c, 512) for c in corrs]
    d64 = gsd.init_depth(depth)
    lat_b = torch.cat([latents0, latents0 * 0.9, latents0 + 0.1])
    ddim = DDIMSchedule()
    ddim.set_timesteps(T)
    ts = ddim.timesteps

    def mk(Bn):
        # TinyUNet run sample by sample (see test_loss_batch_gpu): the batched loop must reproduce every single-edit run
        def unet_fn(x, t):
            outs = [unet(torch.cat([x[i:i + 1], d64], 1), t, encoder_hidden_states=cond) for i in range(Bn)]
            o = [torch.cat([q[k] for q in outs]) for k in (0, 4, 5, 6)]
            return o[0], o[1:]

        def cfg_pair(x, t, t_idx):
            o = unet_fn(x, t)[0]
            return o * 0.5, o
        return unet_fn, cfg_pair
    kw = dict(fg_weight=1.5, bg_weight=1.25, num_optsteps=2, guidance_max_step=2, ddim=ddim,
              bg_loss_type="local_avg", skip_zero_weight_layers=False)
    calls = {"loss": 0}
    real = guided_loop.guidance_loss_and_grad_batch
    monkeypatch.setattr(guided_loop, "guidance_loss_and_grad_batch",
                        lambda *a, **k: (calls.__setitem__("loss", calls["loss"] + 1), real(*a, **k))[1])
    ufn, cp = mk(B)
    res = {}
    ran, _ = _patch_launches(lambda: res.setdefault("out", guided_denoise_batch(lat_b.clone(), ts, ufn, None, acts_orig, pcs,
                                                                                cfg_pair=cp, **kw)))
    out = res["out"]
    assert calls["loss"] == 2 * 2, calls
    assert ran == Counter({"loss_patch_batch_kernel": 4, "loss_patch_finish_batch_kernel": 4}), ran
    ufn1, cp1 = mk(1)
    for e in range(B):
        ref = guided_denoise(lat_b[e:e + 1].clone(), ts, ufn1, None, acts_orig, pcs[e], cfg_pair=cp1, **kw)
        assert torch.allclose(out[e:e + 1], ref, rtol=1e-5, atol=1e-5 * float(ref.abs().max())), (e, float((out[e] - ref[0]).abs().max()))
