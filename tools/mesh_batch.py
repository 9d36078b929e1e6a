"""Mesh-mode edits of one scene: B single-edit ``transform_depth_mesh`` calls against one ``transform_depth_mesh_batch`` call.

    python tools/mesh_batch.py --out profiles/mesh_batch.json [--reps 7]

Edits: the config-1 scene (synthetic_scene(512, 0)) with the B first transforms of the config-4 recipe (as tools/k4_batch.py
builds them), B in 1, 2, 4, 8, 16.  Reported per B:
  (a) wall time per edit of both arms, each ending with the correspondences on the CPU as the API returns them (host clock
      around the call, which ends in device-to-host copies and a synchronise); the two arms alternate, ``--reps`` passes;
  (b) device time of the dh_edit_mesh_batch call alone (CUDA events around ``INNER`` back-to-back calls on prepared meshes).
Medians with [min, max].  Both arms' outputs (disparities bit for bit, correspondences values and order) are compared in the
same run; the result records the GPU's name, power limit and maximum SM clock.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
BATCHES = (1, 2, 4, 8, 16)
INNER = 10          # native calls per device-time sample


def _edits(n):
    import numpy as np
    import torch
    angles = np.linspace(-90.0, 90.0, 16)
    return ([float(angles[k]) for k in range(n)], [torch.tensor([0.0, 1.0, 0.0]) for _ in range(n)],
            [torch.tensor([0.1 * k - 0.8, 0.0, 0.05 * k]) for k in range(n)])


def _stats(v):
    s = sorted(v)
    return {"median": s[len(s) // 2], "min": s[0], "max": s[-1]}


def _native_timer(td, tb, tm, K, angles, axes, shifts, dev):
    """CUDA-event timer of the dh_edit_mesh_batch call alone, on the meshes and arguments transform_depth_mesh_batch prepares"""
    import torch
    from diffusionhandles_b200 import _native as N
    from diffusionhandles_b200.depth_transform import depth_to_mesh
    from diffusionhandles_b200.renderer import MeshRenderer, fov_scales
    lib = N.load()
    B, (H, W) = len(angles), td.shape[-2:]
    bg, fg = depth_to_mesh(tb, K), depth_to_mesh(td, K, mask=tm[0, 0] > 0.5)
    bv, bf = bg.verts.contiguous(), bg.faces.to(torch.int32).contiguous()
    fv, fc, ff = fg.verts.contiguous(), fg.vert_attributes["color"].contiguous(), fg.faces.to(torch.int32).contiguous()
    sx, sy = fov_scales(K[1, 1], H, W, MeshRenderer.z_near)
    ang = (C.c_float * B)(*[float(torch.tensor(a, dtype=torch.float32)) for a in angles])
    axs = (C.c_float * (3 * B))(*[float(v) for a in axes for v in a])
    trs = (C.c_float * (3 * B))(*[float(v) for t in shifts for v in t])
    R, T = (C.c_float * 9)(1, 0, 0, 0, 1, 0, 0, 0, 1), (C.c_float * 3)(0, 0, 0)
    z = torch.empty((B, H, W), dtype=torch.float32, device=dev)
    corr = torch.empty((B, H * W, 4), dtype=torch.int64, device=dev)
    n = torch.empty(B, dtype=torch.int32, device=dev)
    ws_bytes = int(lib.dh_edit_mesh_batch_workspace_bytes(B, bv.shape[0], fv.shape[0], H, W))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    st = N.stream_handle(dev)

    def call():
        N.check(lib.dh_edit_mesh_batch(N.ptr(bv), bv.shape[0], N.ptr(bf), bf.shape[0], N.ptr(fv), N.ptr(fc), fv.shape[0], N.ptr(ff),
                                       ff.shape[0], B, ang, axs, trs, H, W, R, T, sx, sy, 1e-5, 1, 1, 1, N.ptr(z), N.ptr(corr), N.ptr(n),
                                       None, N.ptr(ws), ws_bytes, st), "dh_edit_mesh_batch")
    call()
    torch.cuda.synchronize(dev)

    def timed():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(INNER):
            call()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) / INNER
    return timed, {"V_bg": bv.shape[0], "F_bg": bf.shape[0], "V_fg": fv.shape[0], "F_fg": ff.shape[0]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    if args.reps < 5:
        raise SystemExit("--reps must be at least 5")
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
    depth, bg, mask = synthetic_scene(512, 0)
    td, tb, tm = (torch.from_numpy(a).to(dev)[None, None] for a in (depth, bg, mask))
    result = {"gpu": smi[0] if smi else torch.cuda.get_device_name(dev), "scene": "synthetic_scene(512, 0)",
              "transforms": "config-4 recipe: angle linspace(-90, 90, 16)[k] about +y, translation (0.1 k - 0.8, 0, 0.05 k)",
              "reps": args.reps, "native_calls_per_sample": INNER,
              "note": "wall_ms_per_edit: host clock per edit, each arm ending with CPU correspondences; device_ms: CUDA events around "
                      "the dh_edit_mesh_batch call alone (per call, not per edit)", "batches": {}}

    def loop_arm(angles, axes, shifts):
        outs = [dt.transform_depth_mesh(td, tb, tm, K, a, ax, t) for a, ax, t in zip(angles, axes, shifts)]
        torch.cuda.synchronize(dev)
        return outs

    def batch_arm(angles, axes, shifts):
        out = dt.transform_depth_mesh_batch(td, tb, tm, K, angles, axes, shifts)
        torch.cuda.synchronize(dev)
        return out

    for B in BATCHES:
        angles, axes, shifts = _edits(B)
        singles = loop_arm(angles, axes, shifts)                  # warm-up of both arms, and the equality check
        disp, corrs = batch_arm(angles, axes, shifts)
        equal = all(torch.equal(disp[b:b + 1].view(torch.int32), d.view(torch.int32)) and torch.equal(corrs[b], c)
                    for b, (d, c) in enumerate(singles))
        if not equal:
            raise SystemExit(f"B={B}: the batch differs from the single-edit calls")
        samples = {"loop": [], "batch": []}
        for _ in range(args.reps):                                # alternate the two arms
            for k, fn in (("loop", loop_arm), ("batch", batch_arm)):
                t0 = time.perf_counter()
                fn(angles, axes, shifts)
                samples[k].append((time.perf_counter() - t0) * 1e3 / B)
        timed, sizes = _native_timer(td, tb, tm, K, angles, axes, shifts, dev)
        dev_ms = [timed() for _ in range(args.reps)]
        row = {"outputs_equal": equal, "n_corr": [int(c.shape[0]) for c in corrs], **sizes,
               "wall_ms_per_edit": {k: _stats(v) for k, v in samples.items()}, "device_ms": _stats(dev_ms)}
        row["wall_speedup_median"] = row["wall_ms_per_edit"]["loop"]["median"] / row["wall_ms_per_edit"]["batch"]["median"]
        result["batches"][f"B{B}"] = row
        print(B, json.dumps(row), flush=True)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
