#!/usr/bin/env python
"""Mesh export timing: NeRF.extract_mesh on the synthetic unit sphere at 256^3 and 512^3 -- the density grid (the fused
bf16 forward, one ray per lattice column), the marching-tetrahedra isosurface, and the per-vertex colour query.  The
model is trained first (600 steps on whole 128 x 128 views, as tests/test_gpu_mesh.py does) so that the surface is the
one a user would export, not the noise of random weights.  Every stage ends with a device synchronise; each resolution
is run once to warm up, then `reps` times; the median is reported.  Prints one JSON line.
usage: python benchmarks/mesh.py [reps=3] [threshold=1.0]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                            "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except Exception as e:  # pragma: no cover
        return f"nvidia-smi unavailable: {e}"


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    thr = float(sys.argv[2]) if len(sys.argv) > 2 else 1.0
    from keras_nerf_b200 import NeRF
    from keras_nerf_b200.data.synthetic import SyntheticScene
    from keras_nerf_b200.model.nerf import mlp as mlp_mod
    dev = torch.device("cuda", 0)
    R = 128 * 128
    mlp_mod.set_seed(42)
    m = NeRF(precision="bf16", device=dev)
    m.compile(optimizer="adam", loss="mse", batch_size=1, image_height=128, image_width=128, ray_chunks=R,
              white_background=True)
    scene = SyntheticScene(128, 64, n_views=40, device=dev)
    for step in range(600):
        img, rays = scene.ray_batch((step * 7) % 40, R, seed=step)
        m.accumulate_gradients(img, rays, seed=10_000 + step, want_images=False)
        m.apply_gradients()
        m._losses.zero_()
    torch.cuda.synchronize()
    out = {"gpu_before": _gpu_info(), "precision": m.precision, "threshold": thr, "bound": 1.5, "reps": reps}
    for res in (256, 512):
        runs = []
        for _ in range(reps + 1):
            mesh = m.extract_mesh(resolution=res, threshold=thr, bound=1.5)
            runs.append(mesh["seconds"])
        sec = {k: float(np.median([r[k] for r in runs[1:]])) for k in runs[0]}
        v = mesh["vertices"]
        n_pts = (res + 2) ** 3                                   # close=True pads one layer
        out[str(res)] = {
            "grid_s": round(sec["grid"], 4), "grid_ns_per_sample": round(sec["grid"] / res ** 3 * 1e9, 3),
            "isosurface_s": round(sec["isosurface"], 4),
            # the field is read by both passes; 5 B per point of workspace written by the count pass, read by emit
            "isosurface_field_GBps": round(2 * 4 * n_pts / sec["isosurface"] / 1e9, 1),
            "colors_s": round(sec["colors"], 4), "V": int(v.shape[0]), "T": int(mesh["faces"].shape[0]),
            "median_abs_radius_error": round(float(torch.median((torch.linalg.norm(v, dim=1) - 1).abs())), 5),
        }
        del mesh
    out["gpu_after"] = _gpu_info()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
