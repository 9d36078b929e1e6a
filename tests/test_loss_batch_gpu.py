"""GPU (``-m gpu``): batched guidance losses (``dh_guidance_loss_batch`` / ``losses.guidance_loss_and_grad_batch``) and the
batched guided loop and facade built on them.  Every edit of a batch must give the bits the single-edit launch gives."""
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.dirname(os.path.abspath(__file__))):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from test_loss_plan_and_variants_gpu import (FUSED_VARIANTS, _check_against_oracle, _inputs, _lists, _pc,  # noqa: E402
                                             kernels_of, variant_cases)

gpu = pytest.mark.gpu
_B = "loss_fused_batch_kernel<{}>"


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _batch_kernels(fn):
    """{'loss_fused_batch_kernel<kG, kBinary, kMem, kGroups>': {groups}} and the single-edit kernels that ran inside fn()."""
    import json
    import re
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
    found = {}
    for e in events:
        if e.get("cat") != "kernel":
            continue
        m = re.search(r"loss_fused_batch_kernel<(\d+), ?(true|false|\(bool\)[01]), ?(\d+), ?(\d+)>", e["name"])
        if not m:
            continue
        b = {"(bool)1": "true", "(bool)0": "false"}.get(m.group(2), m.group(2))
        found.setdefault(_B.format(f"{m.group(1)}, {b}, {m.group(3)}, {m.group(4)}"), []).append(e["args"]["block"][0] // 256)
    return found


def _twin(single):
    return single.replace("loss_fused_kernel", "loss_fused_batch_kernel")


def _edit_lists(name, case, k):
    """Edit 0: the case's own lists; edit 1: lists of another seed; edit 2: no foreground pair at all."""
    grid, lists = case[0], case[5]
    binary = "bin" in name
    if k == 0:
        return lists
    other = _lists(np.random.default_rng(100 + k), grid, binary)
    if k == 1:
        return other
    e = np.zeros(0, np.int64)
    return (e, e) + tuple(other[2:])


def _single(dev, acts, origs, pc, fgw, bgw, lt, grid):
    from diffusionhandles_b200 import losses
    t, p, g = losses.guidance_loss_and_grad(acts, origs, pc, fgw, bgw, bg_loss_type=lt, activations_size=(grid, grid))
    return t.cpu().numpy(), p.cpu().numpy(), [x.cpu().numpy() for x in g]


def _run_batch(dev, name, case, n_edits, shared_orig=True, seeds=None):
    """A batch of n_edits edits of one variant case; returns (batch results, per-edit single results)."""
    from diffusionhandles_b200 import losses
    grid, shapes, lt = case[0], case[1], case[2]
    curs, origs, fgw, bgw = _inputs(name, shapes)
    gen = torch.Generator().manual_seed(7)
    cur_b = [torch.stack([c] + [torch.randn(c.shape, generator=gen) for _ in range(n_edits - 1)]).to(dev) for c in curs]
    org_b = [o.to(dev) if shared_orig else torch.stack([o] + [torch.randn(o.shape, generator=gen) for _ in range(n_edits - 1)]).to(dev)
             for o in origs]
    pcs = [_pc(*_edit_lists(name, case, k if seeds is None else seeds[k]), grid) for k in range(n_edits)]
    res = {}

    def run():
        t, p, g = losses.guidance_loss_and_grad_batch(cur_b, org_b, pcs, fgw, bgw, bg_loss_type=lt, activations_size=(grid, grid))
        res["b"] = (t.cpu().numpy(), p.cpu().numpy(), [x.cpu().numpy() for x in g])
    ran = _batch_kernels(run)
    singles = [_single(dev, [c[e] for c in cur_b], [o if shared_orig else o[e] for o in org_b], pcs[e], fgw, bgw, lt, grid)
               for e in range(n_edits)]
    return res["b"], singles, ran


def _assert_bit_identical(batch, singles, what):
    t, p, g = batch
    for e, (ts, ps, gs) in enumerate(singles):
        assert np.array_equal(t[e], ts, equal_nan=True), (what, e, t[e], ts)
        assert np.array_equal(p[e], ps, equal_nan=True), (what, e)
        for l, gl in enumerate(gs):
            assert np.array_equal(g[l][e], gl), (what, e, l)


_FUSED = [n for n, c in variant_cases().items() if c[4] != "loss_patch_kernel"]


@gpu
@pytest.mark.parametrize("name", _FUSED)
def test_every_batch_instantiation_is_bit_identical(dev, name):
    """A batch of three edits (the case's lists, another seed's, an empty foreground list) runs as ONE batch launch of the
    instantiation the case's single edit runs, and every edit's value, parts and gradients are that edit's own bits."""
    case = variant_cases()[name]
    batch, singles, ran = _run_batch(dev, name, case, 3)
    assert list(ran) == [_twin(case[4])] and len(ran[_twin(case[4])]) == 1, (name, ran)
    _assert_bit_identical(batch, singles, name)
    assert np.isnan(batch[1][2][0::2]).all() and not np.isnan(batch[1][2][1::2]).any()     # empty foreground list: NaN fg terms
    if name == "flat64_bin":
        _check_against_oracle(name, case, float(batch[0][0]), batch[1][0], [g[0] for g in batch[2]])


def test_every_batch_instantiation_is_selected():
    assert {_twin(variant_cases()[n][4]) for n in _FUSED} == {_twin(v) for v in FUSED_VARIANTS}


@gpu
def test_mixed_batch(dev):
    """A count plan next to binary plans runs the count instantiation (kBinary needs every plan binary); per-edit recorded
    activations next to a shared one; results are every edit's own bits."""
    name = "flat64_bin"
    case = variant_cases()[name]
    from diffusionhandles_b200 import losses
    grid, shapes, lt = case[0], case[1], case[2]
    curs, origs, fgw, bgw = _inputs(name, shapes)
    cur_b = [torch.stack([c, c * 0.5 - 0.25, -c]).to(dev) for c in curs]
    org_b = [torch.stack([o, o + 0.5, o * 2]).to(dev) for o in origs]
    pcs = [_pc(*case[5], grid), _pc(*_lists(np.random.default_rng(5), grid, False), grid), _pc(*_lists(np.random.default_rng(6), grid, True), grid)]
    res = {}
    ran = _batch_kernels(lambda: res.setdefault("b", losses.guidance_loss_and_grad_batch(cur_b, org_b, pcs, fgw, bgw, bg_loss_type=lt)))
    assert list(ran) == [_B.format("64, false, 1, 4")], ran
    t, p, g = res["b"]
    singles = [_single(dev, [c[e] for c in cur_b], [o[e] for o in org_b], pcs[e], fgw, bgw, lt, grid) for e in range(3)]
    _assert_bit_identical((t.cpu().numpy(), p.cpu().numpy(), [x.cpu().numpy() for x in g]), singles, "mixed")


@gpu
@pytest.mark.parametrize("name,groups", [("flat64_many_cnt", 4), ("one_resized_many_cnt", 3), ("grid48_many_cnt", 3)])
def test_many_cases_at_two_edits(dev, name, groups):
    """Two edits of 640 (320) work items each: 1280 (640) items in all, so no group sits idle (148 * (groups - 1) < items) and
    the launch keeps the group count the preference gives the single edit: 4 for the flat build, 3 otherwise."""
    case = variant_cases()[name]
    batch, singles, ran = _run_batch(dev, name, case, 2, seeds=[0, 1])
    assert ran == {_twin(case[4]): [groups]}, (name, ran)
    _assert_bit_identical(batch, singles, name)


@gpu
@pytest.mark.parametrize("n_edits", [1, 16, 20])
def test_batch_limits(dev, n_edits):
    """B = 1 (the single-edit launch), the 16 edits of one launch, and B = 20, which runs as 16 + 4."""
    name = "one_resized_bin"
    case = variant_cases()[name]
    batch, singles, ran = _run_batch(dev, name, case, n_edits, shared_orig=False, seeds=[k % 2 for k in range(n_edits)])
    # one edit takes the single-edit launch (cheaper than a batch of one); 20 edits run as 16 + 4
    assert (not ran) if n_edits == 1 else (list(ran) == [_twin(case[4])] and len(ran[_twin(case[4])]) == (1 if n_edits <= 16 else 2)), ran
    _assert_bit_identical(batch, singles, n_edits)
    if n_edits == 1:
        _check_against_oracle(name, case, float(batch[0][0]), batch[1][0], [g[0] for g in batch[2]])


@gpu
def test_general_path_loops_the_single_launch(dev):
    """Inputs that go to the general patch kernel (patch 3) run one launch per edit with the same results."""
    from diffusionhandles_b200 import losses
    grid, shapes = 64, [(3, 64, 64), (2, 32, 32)]
    curs, origs, fgw, bgw = _inputs("general", shapes)
    cur_b = [torch.stack([c, c + 1.0]).to(dev) for c in curs]
    pcs = [_pc(*_lists(np.random.default_rng(s), grid, True), grid) for s in (1, 2)]
    t, p, g = losses.guidance_loss_and_grad_batch(cur_b, [o.to(dev) for o in origs], pcs, fgw, bgw, bg_loss_type="local_avg", patch_size=3)
    for e in range(2):
        ts, ps, gs = losses.guidance_loss_and_grad([c[e] for c in cur_b], [o.to(dev) for o in origs], pcs[e], fgw, bgw,
                                                   bg_loss_type="local_avg", patch_size=3)
        assert torch.equal(t[e], ts) and torch.equal(p[e], ps) and all(torch.equal(a[e], b) for a, b in zip(g, gs))


@gpu
def test_repeated_calls_rearm_the_counters(dev):
    """The same plans and the same cached runner (one workspace, zeroed once) serve every call: two consecutive batched calls,
    then single-edit calls on the same plans, then a batched call again, all give the same bits (each launch re-arms every
    edit's queue counter and finish ticket)."""
    from diffusionhandles_b200 import losses
    from diffusionhandles_b200.guided_stable_diffuser import ProcessedCorrespondences
    name = "one_resized_cnt"
    case = variant_cases()[name]
    grid, shapes, lt = case[0], case[1], case[2]
    curs, origs, fgw, bgw = _inputs(name, shapes)
    gen = torch.Generator().manual_seed(9)
    cur_b = [torch.stack([c, torch.randn(c.shape, generator=gen), -c]).to(dev) for c in curs]
    org = [o.to(dev) for o in origs]
    pcs = []
    for k in range(3):      # ProcessedCorrespondences cache their plan: every call below reuses the same three plans
        pc = ProcessedCorrespondences(_pc(*_edit_lists(name, case, k), grid))
        pc.grid, pc.device_lists = grid, losses._lists(dict(pc), grid, dev)
        pcs.append(pc)

    def batch():
        t, p, g = losses.guidance_loss_and_grad_batch(cur_b, org, pcs, fgw, bgw, bg_loss_type=lt, activations_size=(grid, grid))
        return t.cpu().numpy(), p.cpu().numpy(), [x.cpu().numpy() for x in g]
    first = batch()
    plan0 = losses._plan_for(pcs[0], grid, dev)
    runners = [r for k, r in plan0._runners.items() if k[0] == "batch"]
    assert len(runners) == 1
    ws = runners[0][3]
    second = batch()
    singles = [_single(dev, [c[e] for c in cur_b], org, pcs[e], fgw, bgw, lt, grid) for e in range(3)]
    third = batch()
    assert [r for k, r in plan0._runners.items() if k[0] == "batch"] == runners and runners[0][3] is ws      # one runner, one workspace
    assert all(losses._plan_for(pc, grid, dev) is p for pc, p in zip(pcs, runners[0][0]))
    for what, res in (("first", first), ("second", second), ("after singles", third)):
        _assert_bit_identical(res, singles, what)


@gpu
def test_shared_and_per_edit_recorded_layers_in_one_call(dev):
    """Recorded activations shared by every edit (C,h,w) next to per-edit ones (B,C,h,w) in the same call, on a resized and a
    flat layer each."""
    from diffusionhandles_b200 import losses
    name = "two_resized_cnt"
    case = variant_cases()[name]
    grid, shapes, lt = case[0], case[1], case[2]
    curs, origs, fgw, bgw = _inputs(name, shapes)
    gen = torch.Generator().manual_seed(10)
    cur_b = [torch.stack([c, torch.randn(c.shape, generator=gen), c * 0.5]).to(dev) for c in curs]
    org = [origs[0].to(dev), torch.stack([origs[1], torch.randn(origs[1].shape, generator=gen), -origs[1]]).to(dev),
           torch.stack([origs[2], origs[2] + 1.0, torch.randn(origs[2].shape, generator=gen)]).to(dev)]
    # layer 0 (resized) shared; layers 1 (resized) and 2 (flat) per edit; then layer 2 shared too
    org_shared2 = [org[0], org[1], origs[2].to(dev)]      # layer 2 shared as well
    pcs = [_pc(*_edit_lists(name, case, k), grid) for k in range(3)]
    for origs_b in (org, org_shared2):
        res = {}
        ran = _batch_kernels(lambda: res.setdefault("b", losses.guidance_loss_and_grad_batch(cur_b, origs_b, pcs, fgw, bgw, bg_loss_type=lt)))
        assert list(ran) == [_twin(case[4])], ran
        t, p, g = res["b"]
        singles = [_single(dev, [c[e] for c in cur_b], [o if o.dim() == 3 else o[e] for o in origs_b], pcs[e], fgw, bgw, lt, grid)
                   for e in range(3)]
        _assert_bit_identical((t.cpu().numpy(), p.cpu().numpy(), [x.cpu().numpy() for x in g]), singles, "shared+per-edit")


def _child_main(out_path):
    dev = torch.device("cuda:0")
    saved = {}
    for name in ("flat64_cnt", "one_resized_bin", "two_resized_cnt", "grid48_bin"):
        (t, p, g), _, ran = _run_batch(dev, name, variant_cases()[name], 3)
        saved[f"{name}/t"], saved[f"{name}/p"] = t, p
        for i, x in enumerate(g):
            saved[f"{name}/g{i}"] = x
        saved[f"{name}/k"] = np.array(sorted(ran))
    np.savez(out_path, **saved)


@gpu
def test_knobs_give_bit_identical_batches(dev, tmp_path):
    """DH_LOSS_MEM=0 DH_LOSS_GROUPS=1 (read once per process: a child process) gives the default launch's bits."""
    out = tmp_path / "child.npz"
    env = {k: v for k, v in os.environ.items() if k not in ("DH_LOSS_NO_FOUR_GROUPS", "DH_LOSS_DEBUG_BUF")}
    env.update(DH_LOSS_MEM="0", DH_LOSS_GROUPS="1")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", str(out)], env=env, cwd=ROOT, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    child = np.load(out)
    for name in ("flat64_cnt", "one_resized_bin", "two_resized_cnt", "grid48_bin"):
        (t, p, g), _, ran = _run_batch(dev, name, variant_cases()[name], 3)
        assert np.array_equal(child[f"{name}/t"], t, equal_nan=True) and np.array_equal(child[f"{name}/p"], p, equal_nan=True), name
        assert all(np.array_equal(child[f"{name}/g{i}"], x) for i, x in enumerate(g)), name
        assert all(k.endswith(", 0, 3>") for k in child[f"{name}/k"]), (name, child[f"{name}/k"])


# ------------------------------------------------------------------------------------------------
# the batched loop and facade
# ------------------------------------------------------------------------------------------------
def _tiny(dev, T):
    from test_guided_step_gpu import _setup
    return _setup(dev, T)


class _PerSample(torch.nn.Module):
    """A U-Net run one sample at a time (each with its own condition row): it mixes no samples, and its arithmetic does not
    depend on the batch size (at batch 3 cuDNN may pick another algorithm, and TinyUNet's mean over the whole condition rounds
    differently), so a batched run must reproduce every single-edit run."""

    def __init__(self, unet):
        super().__init__()
        self.unet, self.config = unet, unet.config

    def forward(self, x, t, encoder_hidden_states=None, cross_attention_kwargs=None, return_dict=False):
        outs = [self.unet(x[i:i + 1], t, encoder_hidden_states=encoder_hidden_states[i:i + 1]) for i in range(x.shape[0])]
        return tuple(None if outs[0][k] is None else torch.cat([o[k] for o in outs]) for k in range(len(outs[0])))


@gpu
def test_guided_denoise_batch_matches_per_edit_runs(dev, golden_pc, monkeypatch):
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
        # TinyUNet run sample by sample with the condition repeated per edit: a stub that mixes no samples and whose per-sample
        # arithmetic does not depend on the batch size (cuDNN may pick another algorithm at batch 3, and TinyUNet's mean over
        # the whole condition rounds differently), so the batched loop must reproduce every single-edit run
        def unet_fn(x, t):
            outs = [unet(torch.cat([x[i:i + 1], d64], 1), t, encoder_hidden_states=cond) for i in range(Bn)]
            o = [torch.cat([q[k] for q in outs]) for k in (0, 4, 5, 6)]
            return o[0], o[1:]

        def cfg_pair(x, t, t_idx):
            o = unet_fn(x, t)[0]
            return o * 0.5, o
        return unet_fn, cfg_pair
    kw = dict(fg_weight=1.5, bg_weight=1.25, num_optsteps=2, guidance_max_step=2, ddim=ddim, skip_zero_weight_layers=True)
    calls = {"loss": 0, "lat": 0, "ddim": 0}
    real = (guided_loop.guidance_loss_and_grad_batch, guided_loop.latent_step, guided_loop.cfg_ddim_step)

    def count(k, f):
        return lambda *a, **k2: (calls.__setitem__(k, calls[k] + 1), f(*a, **k2))[1]
    monkeypatch.setattr(guided_loop, "guidance_loss_and_grad_batch", count("loss", real[0]))
    monkeypatch.setattr(guided_loop, "latent_step", count("lat", real[1]))
    monkeypatch.setattr(guided_loop, "cfg_ddim_step", count("ddim", real[2]))
    ufn, cp = mk(B)
    out = guided_denoise_batch(lat_b.clone(), ts, ufn, None, acts_orig, pcs, cfg_pair=cp, **kw)
    assert calls == {"loss": 2 * 2, "lat": 2 * 2, "ddim": T}, calls
    ufn1, cp1 = mk(1)
    for e in range(B):
        ref = guided_denoise(lat_b[e:e + 1].clone(), ts, ufn1, None, acts_orig, pcs[e], cfg_pair=cp1, **kw)
        assert torch.allclose(out[e:e + 1], ref, rtol=1e-5, atol=1e-5 * float(ref.abs().max())), (e, float((out[e] - ref[0]).abs().max()))
    # one identity per edit gives the same as the shared one when the identities are equal (the loss bits are the same; cuDNN's
    # backward is not bit-reproducible from run to run)
    out2 = guided_denoise_batch(lat_b.clone(), ts, ufn, None, [acts_orig] * B, pcs, cfg_pair=cp, **kw)
    assert torch.allclose(out, out2, rtol=1e-5, atol=1e-5 * float(out.abs().max()))
    with pytest.raises(NotImplementedError):
        guided_denoise_batch(lat_b.clone(), ts, ufn, None, acts_orig, pcs, cfg_pair=cp, bg_loss_type="local_avg", bg_patch_size=3, **kw)


@gpu
def test_transform_foreground_batch(dev, golden_pc):
    from diffusionhandles_b200 import DiffusionHandles
    from diffusionhandles_b200.depth_transform import transform_depth
    from oracle import dh_oracle as O
    meta, g = golden_pc
    m = meta["cfg1"]
    T = 3
    conf, unet, gsd, gen, latents0, _, cond, uncond = _tiny(dev, T)
    conf.save_denoising_steps = False
    gsd.unet = _PerSample(unet)
    dh = DiffusionHandles(SimpleNamespace(guided_diffuser=conf, depth_transform_mode='pc'), diffuser=gsd).to(dev)
    depth, bg, mask = O.synthetic_scene(**m["scene"])
    td, tb, tm = (torch.from_numpy(a).to(dev)[None, None] for a in (depth, bg, mask))
    acts = [torch.randn((T, c, s, s), generator=gen, device=dev) for c, s in ((6, 32), (5, 64), (4, 64))]
    angles = [m["angle"], m["angle"] * 0.5, 10.0]
    axes = [torch.tensor(m["axis"]), torch.tensor(m["axis"]), torch.tensor([1.0, 0.0, 0.0])]
    shifts = [torch.tensor(m["translation"]), torch.zeros(3), torch.tensor(m["translation"]) * 0.5]
    images, disp = dh.transform_foreground_batch(td, cond, tm, tb, uncond, latents0, acts, angles, axes, shifts)
    assert disp.shape == (3, 1, 512, 512) and images.shape == (3, 4, 64, 64)
    K = gsd.get_depth_intrinsics(device=dev)
    _, corrs = dh.edit_geometry_batch(td, tm, tb, angles, axes, shifts)
    for e in range(3):
        d1, c1 = transform_depth(td, tb, tm, K, angles[e], axes[e], shifts[e])
        assert torch.equal(disp[e:e + 1], d1) and torch.equal(corrs[e], c1), e
        img, d2 = dh.transform_foreground(td, cond, tm, tb, uncond, latents0, acts, rot_angle=angles[e], rot_axis=axes[e],
                                          translation=shifts[e])
        assert torch.allclose(images[e:e + 1], img, rtol=1e-5, atol=1e-5 * float(img.abs().max())), (e, float((images[e] - img[0]).abs().max()))
    assert np.array_equal(corrs[0].numpy(), g["cfg1/corr"].astype(np.int64))         # the reference's correspondences


if __name__ == "__main__" and len(sys.argv) == 3 and sys.argv[1] == "--child":
    _child_main(sys.argv[2])
