"""Edits of many scenes: per-scene batch calls against one scene-table call, in both depth transform modes.

    python tools/edit_scenes.py --out profiles/edit_scenes.json [--reps 7]

Workload: the reference's 20 photogen scenes with their 90 edits (tests/golden/photogen_inputs.npz; the background is the
scene's own bg_depth).  For each mode ('pc', 'mesh') two arms:
  (a) 20 calls of transform_depth_{mode}_batch, one per scene with that scene's edits;
  (b) ONE transform_depth_{mode}_scenes call with all 90 edits.
Reported per mode and arm, medians with [min, max] over ``--reps`` alternating passes:
  wall_ms_per_edit  host clock around the arm, which ends with every edit's correspondences on the CPU (as the API returns them);
  device_ms         CUDA events around the native work of the arm alone, on inputs prepared outside the timed window: 'mesh'
                    the dh_edit_mesh_batch calls (a) or the dh_edit_mesh_scenes call (b) on prepared meshes; 'pc' the
                    EditEngine runs (a) or the plane gather + one EditEngine run (b), without the count read-back.
Both arms' outputs (disparities bit for bit, correspondences values and order) are compared in the same run; the result records
the GPU's name, power limit and maximum SM clock, read in the same command.
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
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
INNER = 5           # native arm repetitions per device-time sample


def _stats(v):
    s = sorted(v)
    return {"median": s[len(s) // 2], "min": s[0], "max": s[-1]}


def _workload(dev):
    import numpy as np
    import torch
    from helpers import load_photogen
    meta, get = load_photogen()
    scenes = sorted(meta)
    planes = [[], [], []]
    index, angles, axes, shifts = [], [], [], []
    for s, scene in enumerate(scenes):
        for k, a in enumerate(get(scene)):
            planes[k].append(a)
        for e in meta[scene]["edits"].values():
            index.append(s)
            angles.append(e["rotation_angle"])
            axes.append(torch.tensor(e["rotation_axis"]))
            shifts.append(torch.tensor(e["translation"]))
    d, b, m = (torch.from_numpy(np.stack(p)).to(dev)[:, None] for p in planes)
    return scenes, (d, b, m), (index, angles, axes, shifts)


def _per_scene(index, S):
    return [[e for e, s in enumerate(index) if s == k] for k in range(S)]


def _mesh_native_timers(dev, K, planes, edits):
    """CUDA-event timers of arm (a) (one dh_edit_mesh_batch per scene) and arm (b) (one dh_edit_mesh_scenes) on prepared meshes"""
    import torch
    from diffusionhandles_b200 import _native as N
    from diffusionhandles_b200.depth_transform import depth_to_mesh
    from diffusionhandles_b200.renderer import MeshRenderer, fov_scales
    lib = N.load()
    d, b, m = planes
    index, angles, axes, shifts = edits
    S, H, W = d.shape[0], d.shape[-2], d.shape[-1]
    f32, i32 = torch.float32, torch.int32
    meshes = []
    for s in range(S):
        bg, fg = depth_to_mesh(b[s:s + 1], K), depth_to_mesh(d[s:s + 1], K, mask=m[s, 0] > 0.5)
        meshes.append((bg.verts.to(f32).contiguous(), bg.faces.to(i32).contiguous(), fg.verts.to(f32).contiguous(),
                       fg.vert_attributes["color"].to(f32).contiguous(), fg.faces.to(i32).contiguous()))
    sx, sy = fov_scales(K[1, 1], H, W, MeshRenderer.z_near)
    R, T = (C.c_float * 9)(1, 0, 0, 0, 1, 0, 0, 0, 1), (C.c_float * 3)(0, 0, 0)
    st = N.stream_handle(dev)

    def host_edits(es):
        n = len(es)
        return ((C.c_float * n)(*[float(torch.tensor(angles[e], dtype=f32)) for e in es]),
                (C.c_float * (3 * n))(*[float(v) for e in es for v in axes[e]]), (C.c_float * (3 * n))(*[float(v) for e in es for v in shifts[e]]))
    B = len(index)
    z = torch.empty((B, H, W), dtype=f32, device=dev)
    corr = torch.empty((B, H * W, 4), dtype=torch.int64, device=dev)
    n = torch.empty(B, dtype=i32, device=dev)
    groups = _per_scene(index, S)
    calls_a = []
    for s, es in enumerate(groups):
        bv, bf, fv, fc, ff = meshes[s]
        ws_bytes = int(lib.dh_edit_mesh_batch_workspace_bytes(len(es), bv.shape[0], fv.shape[0], H, W))
        calls_a.append((s, es, host_edits(es), torch.empty(ws_bytes, dtype=torch.uint8, device=dev), ws_bytes))

    def arm_a():
        for s, es, (ang, axs, trs), ws, ws_bytes in calls_a:
            bv, bf, fv, fc, ff = meshes[s]
            N.check(lib.dh_edit_mesh_batch(N.ptr(bv), bv.shape[0], N.ptr(bf), bf.shape[0], N.ptr(fv), N.ptr(fc), fv.shape[0], N.ptr(ff),
                                           ff.shape[0], len(es), ang, axs, trs, H, W, R, T, sx, sy, 1e-5, 1, 1, 1, N.ptr(z), N.ptr(corr),
                                           N.ptr(n), None, N.ptr(ws), ws_bytes, st), "dh_edit_mesh_batch")
    cat = [torch.cat([mm[k] for mm in meshes]).contiguous() for k in range(5)]
    counts = [(C.c_int32 * S)(*[mm[k].shape[0] for mm in meshes]) for k in (0, 1, 2, 4)]
    idx = (C.c_int32 * B)(*index)
    ang, axs, trs = host_edits(list(range(B)))
    ws_b_bytes = int(lib.dh_edit_mesh_scenes_workspace_bytes(S, *counts, B, idx, H, W))
    ws_b = torch.empty(ws_b_bytes, dtype=torch.uint8, device=dev)

    def arm_b():
        N.check(lib.dh_edit_mesh_scenes(S, N.ptr(cat[0]), N.ptr(cat[1]), counts[0], counts[1], N.ptr(cat[2]), N.ptr(cat[3]), N.ptr(cat[4]),
                                        counts[2], counts[3], B, idx, ang, axs, trs, H, W, R, T, sx, sy, 1e-5, 1, 1, 1, N.ptr(z), N.ptr(corr),
                                        N.ptr(n), None, N.ptr(ws_b), ws_b_bytes, st), "dh_edit_mesh_scenes")
    return arm_a, arm_b


def _pc_native_timers(dev, K, planes, edits):
    """CUDA-event timers of arm (a) (one EditEngine run per scene) and arm (b) (the plane gather and one EditEngine run)"""
    import torch
    from diffusionhandles_b200.engine import get_engine, make_rigid
    d, b, m = planes
    index, angles, axes, shifts = edits
    S, H, W = d.shape[0], d.shape[-2], d.shape[-1]
    rigids = [make_rigid(a, ax, t) for a, ax, t in zip(angles, axes, shifts)]
    groups = _per_scene(index, S)
    runs_a = [(get_engine(dev, len(es), H, W), tuple(x[s].expand(len(es), H, W).contiguous() for x in (d[:, 0], b[:, 0], m[:, 0])),
               [rigids[e] for e in es]) for s, es in enumerate(groups)]
    eng_b = get_engine(dev, len(index), H, W)
    gather = torch.tensor(index, device=dev)

    def arm_a():
        for eng, (dd, bb, mm), rg in runs_a:
            eng.run(dd, bb, mm, K, rg, poisson=True, sync_counts=False)

    def arm_b():
        dd, bb, mm = (x.reshape(-1, H, W).index_select(0, gather).contiguous() for x in (d, b, m))
        eng_b.run(dd, bb, mm, K, rigids, poisson=True, sync_counts=False)
    return arm_a, arm_b


def _event_ms(fn):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(INNER):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / INNER


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
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    K = GuidedStableDiffuser.get_depth_intrinsics(device=dev)
    scenes, planes, edits = _workload(dev)
    d, b, m = planes
    index, angles, axes, shifts = edits
    B, S = len(index), len(scenes)
    groups = _per_scene(index, S)
    result = {"gpu": smi[0] if smi else torch.cuda.get_device_name(dev), "workload": f"{S} photogen scenes, {B} edits (transforms.json)",
              "reps": args.reps, "native_arm_repetitions_per_sample": INNER,
              "note": "wall_ms_per_edit: host clock per edit, each arm ending with CPU correspondences; device_ms: CUDA events around the "
                      "native work of one arm (per arm, not per edit): (a) 20 per-scene batch calls, (b) one scenes call", "modes": {}}
    for mode in ("pc", "mesh"):
        batch = dt.transform_depth_pc_batch if mode == "pc" else dt.transform_depth_mesh_batch
        scenes_call = dt.transform_depth_pc_scenes if mode == "pc" else dt.transform_depth_mesh_scenes

        def arm_a():
            out = [batch(d[s:s + 1], b[s:s + 1], m[s:s + 1], K, [angles[e] for e in es], [axes[e] for e in es], [shifts[e] for e in es])
                   for s, es in enumerate(groups)]
            torch.cuda.synchronize(dev)
            return out

        def arm_b():
            out = scenes_call(d, b, m, K, index, angles, axes, shifts)
            torch.cuda.synchronize(dev)
            return out
        per_scene = arm_a()                                     # warm-up of both arms, and the equality check
        disp, corrs = arm_b()
        equal = True
        for s, es in enumerate(groups):
            ds, cs = per_scene[s]
            for k, e in enumerate(es):
                equal &= torch.equal(disp[e:e + 1].view(torch.int32), ds[k:k + 1].view(torch.int32)) and torch.equal(corrs[e], cs[k])
        if not equal:
            raise SystemExit(f"{mode}: the scenes call differs from the per-scene batch calls")
        samples = {"per_scene_batches": [], "scenes_call": []}
        for _ in range(args.reps):                              # alternate the two arms
            for k, fn in (("per_scene_batches", arm_a), ("scenes_call", arm_b)):
                t0 = time.perf_counter()
                fn()
                samples[k].append((time.perf_counter() - t0) * 1e3 / B)
        native = (_pc_native_timers if mode == "pc" else _mesh_native_timers)(dev, K, planes, edits)
        for fn in native:
            fn()
        torch.cuda.synchronize(dev)
        dev_ms = {"per_scene_batches": [], "scenes_call": []}
        for _ in range(args.reps):
            for k, fn in zip(dev_ms, native):
                dev_ms[k].append(_event_ms(fn))
        row = {"outputs_equal": equal, "n_corr_total": int(sum(c.shape[0] for c in corrs)),
               "wall_ms_per_edit": {k: _stats(v) for k, v in samples.items()}, "device_ms": {k: _stats(v) for k, v in dev_ms.items()}}
        row["wall_speedup_median"] = row["wall_ms_per_edit"]["per_scene_batches"]["median"] / row["wall_ms_per_edit"]["scenes_call"]["median"]
        row["device_speedup_median"] = row["device_ms"]["per_scene_batches"]["median"] / row["device_ms"]["scenes_call"]["median"]
        result["modes"][mode] = row
        print(mode, json.dumps(row), flush=True)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
