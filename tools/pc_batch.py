"""'pc' edits of one scene: B single-edit ``transform_depth_pc`` calls against one ``transform_depth_pc_batch`` call.

    python tools/pc_batch.py --out profiles/pc_batch.json [--reps 7]

Edits: the config-1 scene (synthetic_scene(512, 0)) with the B first transforms of the config-4 recipe (as tools/mesh_batch.py
builds them), B in 1, 2, 4, 8, 16.  Reported per B: wall time per edit of both arms, each ending with the correspondences on the
CPU as the API returns them (host clock around the call, which ends in device-to-host copies and a synchronise); the two arms
alternate, ``--reps`` passes, medians with [min, max].  Both arms' outputs (disparities bit for bit, correspondences values and
order) are compared in the same run; the result records the GPU's name, power limit and maximum SM clock.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
BATCHES = (1, 2, 4, 8, 16)


def _stats(v):
    s = sorted(v)
    return {"median": s[len(s) // 2], "min": s[0], "max": s[-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    if args.reps < 5:
        raise SystemExit("--reps must be at least 5")
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    from diffusionhandles_b200 import depth_transform as dt
    from diffusionhandles_b200.guided_stable_diffuser import GuidedStableDiffuser
    from diffusionhandles_b200.synthetic import synthetic_scene
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    K = GuidedStableDiffuser.get_depth_intrinsics(device=dev)
    td, tb, tm = (torch.from_numpy(a).to(dev)[None, None] for a in synthetic_scene(512, 0))
    angle = np.linspace(-90.0, 90.0, 16)
    result = {"gpu": smi[0] if smi else torch.cuda.get_device_name(dev), "scene": "synthetic_scene(512, 0)",
              "transforms": "config-4 recipe: angle linspace(-90, 90, 16)[k] about +y, translation (0.1 k - 0.8, 0, 0.05 k)",
              "reps": args.reps, "note": "wall_ms_per_edit: host clock per edit, each arm ending with CPU correspondences", "batches": {}}
    for B in BATCHES:
        angles = [float(angle[k]) for k in range(B)]
        axes = [torch.tensor([0.0, 1.0, 0.0]) for _ in range(B)]
        shifts = [torch.tensor([0.1 * k - 0.8, 0.0, 0.05 * k]) for k in range(B)]

        def loop_arm():
            outs = [dt.transform_depth_pc(td, tb, tm, K, a, ax, t) for a, ax, t in zip(angles, axes, shifts)]
            torch.cuda.synchronize(dev)
            return outs

        def batch_arm():
            out = dt.transform_depth_pc_batch(td, tb, tm, K, angles, axes, shifts)
            torch.cuda.synchronize(dev)
            return out
        singles = loop_arm()
        disp, corrs = batch_arm()
        equal = all(torch.equal(disp[b:b + 1].view(torch.int32), d.view(torch.int32)) and torch.equal(corrs[b], c)
                    for b, (d, c) in enumerate(singles))
        if not equal:
            raise SystemExit(f"B={B}: the batch differs from the single-edit calls")
        samples = {"loop": [], "batch": []}
        for _ in range(args.reps):
            for k, fn in (("loop", loop_arm), ("batch", batch_arm)):
                t0 = time.perf_counter()
                fn()
                samples[k].append((time.perf_counter() - t0) * 1e3 / B)
        row = {"outputs_equal": equal, "n_corr": [int(c.shape[0]) for c in corrs],
               "wall_ms_per_edit": {k: _stats(v) for k, v in samples.items()}}
        result["batches"][f"B{B}"] = row
        print(B, json.dumps(row), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
