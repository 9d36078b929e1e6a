"""Batched guidance losses (dh_guidance_loss_batch) against back-to-back single-edit launches, and the single-edit config-3
launch of this tree against another build of the project (``--baseline-tree``, e.g. an export of main with its library built).

    python tools/k4_batch.py --out profiles/k4_batch.json [--baseline-tree build/main_tree] [--reps 5]

Edits: the config-1 scene (synthetic_scene(512, 0)) with the B first transforms of the config-4 recipe, B in 1, 2, 4, 8, 16.
Shapes: config 3 ((1280, 32^2), (640, 64^2), (320, 64^2)).  Current activations differ per edit; one recorded identity of
T timesteps is shared by every edit.  One timed pass walks R sets of current activations x T timesteps: R * T evaluations of
B edits each, i.e. R * T batched launches or R * T * B single-edit launches, captured in one CUDA graph per mode and timed with
CUDA events; the modes alternate, ``--reps`` times.  The pass reads R * B * 21 MB of current activations, T * 21 MB of recorded
ones and writes R * B * 21 MB of gradients; the result records that working set against the 126 MB L2 (``l2_cold``).  Within
one timestep the shared recorded planes are read B times back to back (once per edit, in both modes), so after the first
edit they come from L2.  Weight sets: (a) all three layers, (b) the reference schedule, which gives layer 0 (the resized 32^2
layer) the weight 0 (guided_inference skips it).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(1280, 32), (640, 64), (320, 64)]
T = 12          # recorded timesteps walked by one timed pass
R = 2           # sets of current activations (B edits each) walked by one timed pass
BATCHES = (1, 2, 4, 8, 16)


def _setup(root, n_edits, dev):
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


def _graph_ms(fn, dev, reps_inner=3):
    import torch
    fn()
    torch.cuda.synchronize(dev)
    gr, side = torch.cuda.CUDAGraph(), torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        fn()
        side.synchronize()
        with torch.cuda.graph(gr, stream=side):
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


WEIGHTS = {"all_layers": ([1.5, 1.5, 1.5], [1.25, 1.25, 1.25]), "reference_schedule": ([0.0, 1.5, 1.5], [0.0, 1.25, 1.25])}


def _modes(root, n_edits, weights, dev):
    """Timed closures: 'batch' (one batched launch per evaluation of n_edits edits) and 'single' (n_edits single launches)."""
    sys.path.insert(0, root)
    from diffusionhandles_b200 import losses
    pcs, origs, curs = _setup(root, n_edits, dev)
    fgw, bgw = WEIGHTS[weights]
    keep = [i for i in range(3) if fgw[i] or bgw[i]]
    sel = lambda xs: [xs[i] for i in keep]       # noqa: E731
    out = {}

    def single():
        for r in range(R):
            for t in range(T):
                for e in range(n_edits):
                    losses.guidance_loss_and_grad([c[e] for c in sel(curs[r])], [o[t] for o in sel(origs)], pcs[e], sel(fgw), sel(bgw))
    out["single"] = _graph_ms(single, dev)
    if hasattr(losses, "guidance_loss_and_grad_batch"):
        def batch():
            for r in range(R):
                for t in range(T):
                    losses.guidance_loss_and_grad_batch(sel(curs[r]), [o[t] for o in sel(origs)], pcs, sel(fgw), sel(bgw))
        out["batch"] = _graph_ms(batch, dev)
    return out


def child_single(root, reps):
    """Single-edit config-3 evaluation (B = 1, all layers) of the build in `root`: ms per evaluation, `reps` samples."""
    import torch
    dev = torch.device("cuda:0")
    timed = _modes(root, 1, "all_layers", dev)["single"]
    return [timed() / (R * T) for _ in range(reps)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--baseline-tree", default=None)
    ap.add_argument("--child-single", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child_single:
        print(json.dumps(child_single(args.child_single, args.reps)))
        return
    import torch
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    plane_bytes = sum(c * s * s for c, s in SHAPES) * 4          # one edit's activations of the three layers
    l2_bytes = torch.cuda.get_device_properties(dev).L2_cache_size
    result = {"gpu": smi[0] if smi else torch.cuda.get_device_name(dev), "shapes": SHAPES, "timesteps_per_pass": T,
              "current_sets_per_pass": R, "l2_bytes": l2_bytes,
              "note": "per edit-evaluation times; within a timestep the shared recorded planes are re-read once per edit (L2-warm "
                      "after the first edit) in both modes", "batches": {}}
    for w in WEIGHTS:
        for B in BATCHES:
            modes = _modes(ROOT, B, w, dev)
            samples = {"batch": [], "single": []}
            for _ in range(args.reps):          # alternate the two modes
                for k in ("batch", "single"):
                    samples[k].append(modes[k]() / (R * T * B) * 1e3)      # us per edit-evaluation
            result["batches"][f"{w}/B{B}"] = {k: {"median_us": sorted(v)[len(v) // 2], "min_us": min(v), "max_us": max(v)}
                                             for k, v in samples.items()}
            ws = (2 * R * B + T) * plane_bytes          # current + gradient of every edit of the pass, the recorded stacks
            result["batches"][f"{w}/B{B}"].update(working_set_bytes=ws, l2_cold=ws > 4 * l2_bytes)
            print(w, B, result["batches"][f"{w}/B{B}"], flush=True)
            torch.cuda.empty_cache()
    if args.baseline_tree:
        # the single-edit config-3 launch of this tree and of the baseline build, alternating child processes
        runs = {"this_tree": [], "baseline": []}
        base = os.path.abspath(args.baseline_tree)
        for _ in range(3):
            for k, root in (("this_tree", ROOT), ("baseline", base)):
                env = dict(os.environ, DH_B200_LIB=os.path.join(root, "diffusionhandles_b200", "lib", "libdiffhandles_b200.so"))
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child-single", root, "--reps", str(args.reps)],
                                   env=env, capture_output=True, text=True, timeout=900, cwd=root)
                if r.returncode != 0:
                    raise RuntimeError(r.stderr[-3000:])
                runs[k] += [v * 1e3 for v in json.loads(r.stdout.strip().splitlines()[-1])]
        result["single_edit_config3_us"] = {k: {"median": sorted(v)[len(v) // 2], "min": min(v), "max": max(v), "samples": v}
                                            for k, v in runs.items()}
        print(result["single_edit_config3_us"], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
