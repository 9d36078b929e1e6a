"""Randomised sweep of multi-object 'pc' edits against the oracle: random scenes, K in 1..16, masks split into angular sectors,
a random transform per object (some off-screen, some objects empty); bit-exact comparison of centroids, object ids, foreground
points, winners, depth maps, masks, correspondences and raw disparity.  python tests/fuzz/fuzz_objects.py [n_cases] [seed]"""
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import dh_oracle as O                                        # noqa: E402
from objects_oracle import sector_masks, transform_depth_pc_objects     # noqa: E402
from test_objects_gpu import _assert_matches_oracle, _run_objects, _snapshot   # noqa: E402
from diffusionhandles_b200.guided_stable_diffuser import GuidedStableDiffuser   # noqa: E402


def run(n_cases: int, seed: int, verbose: bool = True) -> int:
    """Returns the number of mismatching cases."""
    rng = np.random.default_rng(seed)
    dev = torch.device("cuda:0")
    K = GuidedStableDiffuser.get_depth_intrinsics(device=dev)
    bad = 0
    for case in range(n_cases):
        S = int(rng.choice([64, 96, 128, 160, 256]))
        depth, bg, mask = O.synthetic_scene(S, int(rng.integers(0, 10_000)), cx=float(rng.uniform(0.2, 0.8) * S),
                                            cy=float(rng.uniform(0.2, 0.8) * S), radius=float(rng.uniform(0.05, 0.45) * S),
                                            quantize=float(rng.choice([0.0, 0.1])) or None)
        n_obj = int(rng.integers(1, 17))
        masks = sector_masks(mask, n_obj, cx=float(rng.uniform(0, S)), cy=float(rng.uniform(0, S)))
        transforms = []
        for _ in range(int(rng.integers(1, 4))):
            tr = []
            for _ in range(n_obj):
                axis = [(0.0, 1.0, 0.0), (1.0, 0.0, 0.0), tuple(rng.normal(size=3).tolist())][int(rng.integers(0, 3))]
                big = rng.random() < 0.2
                t = tuple(float(np.float32(v)) for v in rng.normal(size=3) * (2.5 if big else 0.3))
                tr.append((float(rng.uniform(-180, 180)), axis, t))
            transforms.append(tr)
        try:
            eng, res = _run_objects(dev, K, depth, bg, masks, transforms)
            snaps = _snapshot(eng, res)
            for e, tr in enumerate(transforms):
                o = transform_depth_pc_objects(depth, bg, masks, O.get_depth_intrinsics(), [a for a, _, _ in tr], [x for _, x, _ in tr],
                                               [t for _, _, t in tr], poisson=False)
                _assert_matches_oracle(snaps[e], o, S, (case, e))
        except AssertionError as err:
            bad += 1
            if verbose:
                print(f"case {case}: S={S} K={n_obj} MISMATCH {err}", flush=True)
    return bad


if __name__ == "__main__":
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 50
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    t0 = time.time()
    bad = run(n, seed)
    print(f"{n} cases, seed {seed}: {bad} mismatching, {time.time() - t0:.1f} s")
    sys.exit(1 if bad else 0)
