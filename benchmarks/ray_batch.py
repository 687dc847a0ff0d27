#!/usr/bin/env python
"""Random ray batches drawn across all training views (knerf_generate_ray_batch, data.loader.RayBatchDataset).

  kernel       ns/ray and GB/s of knerf_generate_ray_batch for 1,048,576 rays x 64 samples from a cache of 100 views
               of 400 x 400 (256 MB, twice the L2), against knerf_generate_rays on 1024 x 1024 rays; CUDA events over
               `launches` launches after warm-up, three alternating rounds, median.
  step         bf16 training step (fp8 records) at 32,768 rays: random ray batches against the contiguous single-view
               windows of benchmarks/records_convergence.py.  Batches are generated before the timed loop, so only the
               step is timed; the two arms alternate, `runs` runs of `steps` steps each.
  convergence  two identically seeded bf16 models on the synthetic scene, same steps and rays: whole 200 x 200 views
               (batch_size 1, 40,000 rays) against --ray_batch 40000 over the same 100 views, validation PSNR on 4
               held-out poses (halfway between training poses) every `every` steps; a third run repeats the whole-view
               arm with other draws as the run-to-run yardstick (constant-learning-rate trajectories are chaotic).
usage: python benchmarks/ray_batch.py kernel [launches=200]
       python benchmarks/ray_batch.py step [runs=5] [steps=30]
       python benchmarks/ray_batch.py convergence [steps=2000] [every=200]
Prints one JSON line."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def scene_cache(scene, n_views):
    imgs = torch.stack([scene.view(k, seed=k)[0] for k in range(n_views)]).contiguous()
    poses = torch.tensor(np.stack([scene.pose(k) for k in range(n_views)]), dtype=torch.float32,
                         device=imgs.device)
    return imgs, poses


def kernel(launches=200):
    from keras_nerf_b200 import _lib, pose_spherical
    dev = torch.device("cuda", 0)
    n_img, HW, R, N = 100, 400, 1 << 20, 64
    P = n_img * HW * HW
    g = torch.Generator(device=dev).manual_seed(0)
    images = torch.rand((n_img, HW, HW, 4), generator=g, device=dev)
    poses = torch.tensor(np.stack([pose_spherical(3.6 * k, -30.0, 4.0) for k in range(n_img)]), dtype=torch.float32,
                         device=dev)
    mk = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)  # noqa: E731
    o, d, t, tgt = mk(R, 3), mk(R, 3), mk(R, N), mk(R, 3)
    c2w = np.asarray(pose_spherical(10.0, -30.0, 4.0), dtype=np.float32)
    st = _lib.stream()
    windows = P // R

    def batch(i):
        _lib.call("knerf_generate_ray_batch", images.data_ptr(), n_img, HW, HW, 4, poses.data_ptr(), 400.0, 2.0, 6.0,
                  N, 42, i // windows, (i % windows) * R, R, None, 1000 + i, o.data_ptr(), d.data_ptr(),
                  t.data_ptr(), tgt.data_ptr(), None, st)

    def rays(i):
        _lib.call("knerf_generate_rays", c2w.ctypes.data, 1024, 1024, 400.0, 2.0, 6.0, N, None, 1000 + i,
                  o.data_ptr(), d.data_ptr(), t.data_ptr(), st)

    def time(fn):
        for i in range(10):
            fn(i)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(launches):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e6 / (launches * R)          # ns per ray

    res = {"ray_batch": [], "rays": []}
    for _ in range(3):
        res["ray_batch"].append(time(batch))
        res["rays"].append(time(rays))
    # bytes the algorithm needs per ray: writes o, d (24), t (4N), target (12); one 16-byte read of the cached pixel
    need = {"ray_batch": 24 + 4 * N + 12 + 16, "rays": 24 + 4 * N}
    out = {"mode": "kernel", "card": card(), "rays": R, "n_samples": N, "cache_views": n_img, "view_wh": HW,
           "launches": launches}
    for k, v in res.items():
        ns = float(np.median(v))
        out[k] = {"ns_per_ray": round(ns, 4), "runs_ns_per_ray": [round(x, 4) for x in v],
                  "bytes_per_ray": need[k], "GB_per_s": round(need[k] / ns, 1)}
    print(json.dumps(out))


def _model(R, ray_chunks, **kw):
    from keras_nerf_b200 import NeRF
    from keras_nerf_b200.model.nerf import mlp as mlp_mod
    mlp_mod.set_seed(42)
    torch.manual_seed(0)
    m = NeRF(precision="bf16", records="fp8", device=torch.device("cuda", 0))
    m.compile(optimizer="adam", loss="mse", ray_chunks=ray_chunks, white_background=True, **kw)
    return m


def step(runs=5, steps=30):
    from keras_nerf_b200.data.loader import RayBatchDataset
    from keras_nerf_b200.data.synthetic import SyntheticScene
    dev = torch.device("cuda", 0)
    R = 32768
    scene = SyntheticScene(400, 64, n_views=100, device=dev)
    imgs, poses = scene_cache(scene, 100)
    ds = RayBatchDataset(imgs, poses, scene.focal, 2.0, 6.0, 64, R, perm_seed=1)
    rng = np.random.default_rng(0)
    window = [scene.ray_batch(int(rng.integers(0, 100)), R, offset=int(rng.integers(0, 400 * 400 - R)), seed=10 + i)
              for i in range(8)]
    random = [ds.batch(0, i, seed=10 + i) for i in range(8)]
    m_w = _model(R, R, batch_size=1, image_height=R // 256, image_width=256)
    m_r = _model(R, R, batch_size=1, image_height=R // 256, image_width=256, ray_batch=R)
    arms = {"window": (m_w, window), "random": (m_r, random)}
    times = {k: [] for k in arms}
    for m, batches in arms.values():                                 # warm-up
        for i in range(5):
            m.accumulate_gradients(*batches[i % 8], seed=7000 + i, want_images=False)
            m.apply_gradients()
    torch.cuda.synchronize()
    for _ in range(runs):
        for name, (m, batches) in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                m.accumulate_gradients(*batches[i % 8], seed=7000 + i, want_images=False)
                m.apply_gradients()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / steps)
    # what producing one batch costs each arm (the window arm generates the whole 400 x 400 view, then slices it)
    gen = {}
    for name, fn in (("window", lambda i: scene.ray_batch(i % 100, R, offset=i * 977, seed=i)),
                     ("random", lambda i: ds.batch(1, i, seed=i))):
        for i in range(3):
            fn(i)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(50):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        gen[name] = round(e0.elapsed_time(e1) / 50, 3)
    out = {"mode": "step", "card": card(), "rays_per_step": R, "runs": runs, "steps_per_run": steps,
           "batch_ms": gen}
    for k, v in times.items():
        out[k] = {"median_ms": round(float(np.median(v)), 3), "min_ms": round(min(v), 3), "max_ms": round(max(v), 3),
                  "runs_ms": [round(x, 3) for x in v]}
    print(json.dumps(out))


def convergence(steps=2000, every=200):
    from keras_nerf_b200.data.loader import RayBatchDataset
    from keras_nerf_b200.data.synthetic import SyntheticScene
    dev = torch.device("cuda", 0)
    WH, R = 200, 200 * 200
    scene = SyntheticScene(WH, 64, n_views=100, device=dev)
    imgs, poses = scene_cache(scene, 100)
    held_scene = SyntheticScene(WH, 64, n_views=200, device=dev)   # odd poses lie halfway between training poses
    held = [held_scene.view(2 * j * 25 + 1, seed=500 + j) for j in range(4)]

    def evaluate(m):
        mse = np.zeros(2)
        for img, (o, d, t) in held:
            res = m.predict_and_render_images((o[None], d[None], t[None]), seed=1)
            for j in range(2):
                mse[j] += float(((res[j]["image"][0] - img[..., :3]) ** 2).mean()) / len(held)
        return [round(float(-10 * np.log10(x)), 3) for x in mse]

    def run(arm, draws):
        m = _model(R, 8000, batch_size=1, image_height=WH, image_width=WH,
                   **({"ray_batch": R} if arm == "random" else {}))
        rng = np.random.default_rng(draws)
        ds = RayBatchDataset(imgs, poses, scene.focal, 2.0, 6.0, 64, R, perm_seed=draws)
        per_epoch = len(ds)
        curve = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            if arm == "random":
                batch = ds.batch(i // per_epoch, i % per_epoch, seed=draws * 100003 + i)
            else:
                k = int(rng.integers(0, 100))
                img, rays = scene.view(k, seed=draws * 100003 + i)
                batch = (img[None], tuple(x[None] for x in rays))
            m.train_step(batch, seed=draws * 7919 + 7000 + i)
            if (i + 1) % every == 0 or i + 1 == steps:
                c, f = evaluate(m)
                curve.append({"step": i + 1, "val_coarse_psnr": c, "val_fine_psnr": f})
        e1.record()
        torch.cuda.synchronize()
        return {"curve": curve, "seconds_incl_eval": round(e0.elapsed_time(e1) / 1e3, 2)}

    out = {"mode": "convergence", "card": card(), "steps": steps, "rays_per_step": R, "views": 100, "view_wh": WH,
           "held_out_views": len(held)}
    out["whole_views"] = run("views", 0)
    out["ray_batch"] = run("random", 0)
    out["whole_views_other_draws"] = run("views", 1)
    print(json.dumps(out))


if __name__ == "__main__":
    mode = sys.argv[1] if len(sys.argv) > 1 else "kernel"
    args = [int(a) for a in sys.argv[2:]]
    {"kernel": kernel, "step": step, "convergence": convergence}[mode](*args)
