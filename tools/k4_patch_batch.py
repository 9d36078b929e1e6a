"""Batched general-patch guidance losses (dh_guidance_loss_patch_batch, through guidance_loss_and_grad_batch) against B
back-to-back single-edit patch launches (guidance_loss_and_grad per edit).

    python tools/k4_patch_batch.py --out profiles/k4_patch_batch.json [--reps 5]

Edits: the config-1 scene (synthetic_scene(512, 0)) with the B first transforms of the config-4 recipe, B in 1, 2, 4, 8, 16.
Shapes: config 3 ((1280, 32^2), (640, 64^2), (320, 64^2)), every layer evaluated with the weights 1.5 / 1.25.  Loss settings:
(a) 'local_avg' with patch 1, which needs the general kernel because layer 0 is smaller than the loss grid, and (b) patch 3
('global_avg').  Current activations differ per edit; one recorded identity of T timesteps is shared by every edit.  One timed
pass walks R sets of current activations x T timesteps: R * T evaluations of B edits, i.e. R * T batched calls or R * T * B
single-edit calls, captured in one CUDA graph per mode and timed with CUDA events; the modes alternate, ``--reps`` times.
After timing, every evaluation of the pass runs once more in each mode and the two modes' totals, parts and gradients are
compared bit for bit.  A torch.profiler run of one evaluation per mode gives the device time of the main patch kernels alone.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(1280, 32), (640, 64), (320, 64)]
T = 4           # recorded timesteps walked by one timed pass
R = 2           # sets of current activations (B edits each) walked by one timed pass
BATCHES = (1, 2, 4, 8, 16)
SETTINGS = {"local_avg_patch1": ("local_avg", 1), "global_avg_patch3": ("global_avg", 3)}
FGW, BGW = [1.5, 1.5, 1.5], [1.25, 1.25, 1.25]


def _setup(n_edits, dev):
    import numpy as np
    import torch
    from diffusionhandles_b200.engine import EditEngine, make_rigid
    from diffusionhandles_b200.guided_stable_diffuser import GuidedStableDiffuser
    from diffusionhandles_b200.synthetic import synthetic_scene
    K = GuidedStableDiffuser.get_depth_intrinsics()
    depth, bg, mask = synthetic_scene(512, 0)
    angles = np.linspace(-90.0, 90.0, 16)
    rigids = [make_rigid(float(angles[k]), [0.0, 1.0, 0.0], [0.1 * k - 0.8, 0.0, 0.05 * k]) for k in range(n_edits)]
    eng = EditEngine(dev, n_edits, 512, 512)
    res = eng.run(*(torch.from_numpy(a).to(dev)[None].expand(n_edits, 512, 512).contiguous() for a in (depth, bg, mask)), K, rigids,
                  poisson=False)
    gsd = GuidedStableDiffuser()
    pcs = [gsd.process_correspondences(res.correspondences(e), 512, 0) for e in range(n_edits)]
    g = torch.Generator(device=dev).manual_seed(4)
    origs = [torch.randn((T, c, s, s), generator=g, device=dev) for c, s in SHAPES]
    curs = [[torch.randn((n_edits, c, s, s), generator=g, device=dev) for c, s in SHAPES] for _ in range(R)]
    return pcs, origs, curs


def _graph_timer(fn, dev, reps_inner=3):
    """fn captured in a CUDA graph; returns a closure giving ms per replay.  Relaxed capture: the patch entries set a kernel
    attribute on every call, which is not a stream operation."""
    import torch
    fn()
    torch.cuda.synchronize(dev)
    gr, side = torch.cuda.CUDAGraph(), torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        fn()
        side.synchronize()
        with torch.cuda.graph(gr, stream=side, capture_error_mode="relaxed"):
            fn()
    torch.cuda.current_stream(dev).wait_stream(side)
    gr.replay()
    torch.cuda.synchronize(dev)

    def timed():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps_inner):
            gr.replay()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / reps_inner
    return timed


def _kernel_us(fn):
    """Device µs of the main patch kernels (single and batch, finish kernels excluded) launched by fn(), from torch.profiler."""
    import tempfile
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    return sum(float(e["dur"]) for e in events
               if e.get("cat") == "kernel" and re.search(r"\bloss_patch(_batch)?_kernel\b", e.get("name", "")))


def _measure(n_edits, setting, reps, dev):
    import torch
    from diffusionhandles_b200 import losses
    lt, patch = SETTINGS[setting]
    pcs, origs, curs = _setup(n_edits, dev)
    kw = dict(bg_loss_type=lt, patch_size=patch)

    def batch_eval(r, t):
        return losses.guidance_loss_and_grad_batch(curs[r], [o[t] for o in origs], pcs, FGW, BGW, **kw)

    def single_eval(r, t, e):
        return losses.guidance_loss_and_grad([c[e] for c in curs[r]], [o[t] for o in origs], pcs[e], FGW, BGW, **kw)

    def batch():
        for r in range(R):
            for t in range(T):
                batch_eval(r, t)

    def single():
        for r in range(R):
            for t in range(T):
                for e in range(n_edits):
                    single_eval(r, t, e)
    timers = {"batch": _graph_timer(batch, dev), "single": _graph_timer(single, dev)}
    samples = {"batch": [], "single": []}
    for _ in range(reps):               # alternate the two modes
        for k in ("batch", "single"):
            samples[k].append(timers[k]() / (R * T * n_edits) * 1e3)      # µs per edit-evaluation
    # both modes' outputs, bit for bit, for every evaluation of the pass
    identical = True
    for r in range(R):
        for t in range(T):
            tb, pb, gb = batch_eval(r, t)
            for e in range(n_edits):
                ts, ps, gs = single_eval(r, t, e)
                identical &= bool(torch.equal(tb[e], ts) and torch.equal(pb[e], ps) and all(torch.equal(a[e], b) for a, b in zip(gb, gs)))
    kernel = {"batch": _kernel_us(lambda: batch_eval(0, 0)) / n_edits,
              "single": _kernel_us(lambda: [single_eval(0, 0, e) for e in range(n_edits)]) / n_edits}
    out = {k: {"median_us": sorted(v)[len(v) // 2], "min_us": min(v), "max_us": max(v)} for k, v in samples.items()}
    out["main_kernel_us_per_edit"] = kernel
    out["bit_identical"] = identical
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    import torch
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    plane_bytes = sum(c * s * s for c, s in SHAPES) * 4
    result = {"gpu": smi[0] if smi else torch.cuda.get_device_name(dev), "shapes": SHAPES, "timesteps_per_pass": T,
              "current_sets_per_pass": R, "l2_bytes": torch.cuda.get_device_properties(dev).L2_cache_size,
              "working_set_bytes_per_edit": 2 * R * plane_bytes,
              "note": "µs of device time per edit-evaluation: the batched call (one patch launch + one finish launch per 16 edits) "
                      "against B single-edit calls (two launches each), both captured in CUDA graphs; median and [min, max] of "
                      "alternating passes; main_kernel_us_per_edit: the main patch kernels alone (torch.profiler, one evaluation)",
              "settings": {k: {"bg_loss_type": v[0], "patch_size": v[1]} for k, v in SETTINGS.items()}, "batches": {}}
    for setting in SETTINGS:
        for B in BATCHES:
            res = _measure(B, setting, args.reps, dev)
            result["batches"][f"{setting}/B{B}"] = res
            print(setting, B, res, flush=True)
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    differ = [k for k, v in result["batches"].items() if not v["bit_identical"]]
    if differ:
        raise SystemExit(f"the batched results differ from the single-edit results: {differ}")


if __name__ == "__main__":
    main()
