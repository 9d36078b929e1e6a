"""Multi-object 'pc' edits: device time of one K-object edit against the single-object edit of the union, and geometry throughput
at batch 256.

    python tools/objects_edit.py --out profiles/objects_edit.json [--reps 30]

Scene: the config-1 scene (synthetic_scene(512, 0)) with its disc split into K = 1, 2, 4, 8 angular sectors; object k takes
transform k of the config-4 recipe, the union edit takes transform 0.  Device time: CUDA events around the engine call (splat,
mask cleaning, correspondences, disparity, hole fill; no count read-back), the two arms alternating on one card, ``--reps``
passes, medians with [min, max].  Throughput: one engine call of 256 edits (K = 1 and K = 4 against the single-object batch of
``transform_depth_pc_batch``), edits per second of device time.  Both arms' outputs are checked against each other for K = 1.
The GPU's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def _stats(v):
    s = sorted(v)
    return {"median": s[len(s) // 2], "min": s[0], "max": s[-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU")
    from objects_oracle import sector_masks
    from diffusionhandles_b200.engine import get_engine, make_rigid
    from diffusionhandles_b200.guided_stable_diffuser import GuidedStableDiffuser
    from diffusionhandles_b200.synthetic import synthetic_scene
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    Kc = GuidedStableDiffuser.get_depth_intrinsics(device=dev)
    depth, bg, mask = synthetic_scene(512, 0)
    S = 512
    angle = np.linspace(-90.0, 90.0, 16)

    def rigid(k):
        return make_rigid(float(angle[k]), [0.0, 1.0, 0.0], [0.1 * k - 0.8, 0.0, 0.05 * k])

    def planes(B, n_obj):
        masks = sector_masks(mask, n_obj)
        labels = np.zeros((S, S), np.uint8)
        for k in range(n_obj):
            labels[masks[k] != 0] = k + 1
        union = (labels > 0).astype(np.float32)
        return [torch.from_numpy(a).to(dev)[None].expand(B, S, S).contiguous() for a in (depth, bg, union, labels)]

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize(dev)
        return a.elapsed_time(b)

    result = {"gpu": smi[0] if smi else torch.cuda.get_device_name(dev), "scene": "synthetic_scene(512, 0), disc split into K sectors",
              "transforms": "object k: config-4 recipe k (angle linspace(-90, 90, 16)[k] about +y, translation (0.1 k - 0.8, 0, 0.05 k))",
              "reps": args.reps, "note": "device ms from CUDA events around one engine call; arms alternate", "single_edit": {},
              "batch256": {}}
    eng1 = get_engine(dev, 1, S, S)
    for n_obj in (1, 2, 4, 8):
        d, b, m, lab = planes(1, n_obj)
        rig = [rigid(k) for k in range(n_obj)]
        arms = {"objects": lambda: eng1.run_objects(d, b, m, lab, n_obj, Kc, rig, sync_counts=False),
                "union": lambda: eng1.run(d, b, m, Kc, [rig[0]], sync_counts=False)}
        for fn in arms.values():
            fn()
        if n_obj == 1:
            r1 = eng1.run(d, b, m, Kc, [rig[0]])
            ref = (r1.disparity.clone(), r1.correspondences(0).clone())
            r2 = eng1.run_objects(d, b, m, lab, 1, Kc, rig)
            assert torch.equal(r2.disparity.view(torch.int32), ref[0].view(torch.int32)) and torch.equal(r2.correspondences(0), ref[1])
        samples = {k: [] for k in arms}
        for _ in range(args.reps):
            for k, fn in arms.items():
                samples[k].append(timed(fn))
        row = {k: _stats(v) for k, v in samples.items()}
        result["single_edit"][f"K{n_obj}"] = row
        print("single", n_obj, json.dumps(row), flush=True)
    B = 256
    engB = get_engine(dev, B, S, S)
    for n_obj in (1, 4):
        d, b, m, lab = planes(B, n_obj)
        rig = [rigid((e + k) % 16) for e in range(B) for k in range(n_obj)]
        rig1 = [rigid(e % 16) for e in range(B)]
        arms = {"objects": lambda: engB.run_objects(d, b, m, lab, n_obj, Kc, rig, sync_counts=False),
                "single_object_batch": lambda: engB.run(d, b, m, Kc, rig1, sync_counts=False)}
        for fn in arms.values():
            fn()
        samples = {k: [] for k in arms}
        for _ in range(max(args.reps // 3, 5)):
            for k, fn in arms.items():
                samples[k].append(timed(fn))
        row = {k: dict(_stats(v), edits_per_s=B / (_stats(v)["median"] * 1e-3)) for k, v in samples.items()}
        result["batch256"][f"K{n_obj}"] = row
        print("batch256", n_obj, json.dumps(row), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
