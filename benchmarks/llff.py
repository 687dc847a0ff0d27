#!/usr/bin/env python
"""Forward-facing scenes: the NDC ray kernels and NDC against world-space sampling on an LLFF-layout scene.

  kernel       ns/ray and GB/s of knerf_generate_rays_ndc against knerf_generate_rays (1024 x 1024 rays x 64 samples,
               Philox jitter), and of knerf_generate_ray_batch_ndc against knerf_generate_ray_batch (1,048,576 rays
               from a cache of 100 views of 400 x 400, 256 MB, twice the L2); CUDA events over `launches` launches
               after warm-up, five rounds alternating the four kernels, median.
  convergence  the write_llff_like scene (20 views of 192 x 256, llffhold 8: 17 training and 3 held-out views), bf16
               with fp8 records, random ray batches of 4,096 rays, 64 + 128 samples per ray in both arms, for `steps`
               steps: NDC rays against world-space rays between the bounds (--no_ndc), two seeds per arm (model
               initialisation, permutation and jitter), fine and coarse PSNR on the held-out views every `every` steps.
usage: python benchmarks/llff.py kernel [launches=200]
       python benchmarks/llff.py convergence [steps=2000] [every=250]
Prints one JSON line.  Writes the scene to a temporary directory."""
import json
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from benchmarks.ray_batch import card  # noqa: E402


def kernel(launches=200):
    from keras_nerf_b200 import _lib
    dev = torch.device("cuda", 0)
    n_img, HW, R, N, focal = 100, 400, 1 << 20, 64, 400.0
    P = n_img * HW * HW
    g = torch.Generator(device=dev).manual_seed(0)
    images = torch.rand((n_img, HW, HW, 4), generator=g, device=dev)
    rng = np.random.default_rng(0)
    poses = np.tile(np.eye(4, dtype=np.float32), (n_img, 1, 1))
    poses[:, :3, 3] = rng.normal(size=(n_img, 3)) * 0.2          # forward-facing: every camera looks down -z
    poses = torch.from_numpy(poses).to(dev)
    mk = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)  # noqa: E731
    o, d, t, tgt = mk(R, 3), mk(R, 3), mk(R, N), mk(R, 3)
    c2w = poses[7].cpu().numpy()
    st = _lib.stream()
    windows = P // R
    out_ptrs = lambda: (o.data_ptr(), d.data_ptr(), t.data_ptr())  # noqa: E731

    def batch(i, ndc):
        head = (images.data_ptr(), n_img, HW, HW, 4, poses.data_ptr(), focal)
        tail = (N, 42, i // windows, (i % windows) * R, R, None, 1000 + i) + out_ptrs() + (tgt.data_ptr(), None, st)
        if ndc:
            _lib.call("knerf_generate_ray_batch_ndc", *head, *tail)
        else:
            _lib.call("knerf_generate_ray_batch", *head, 2.0, 6.0, *tail)

    def rays(i, ndc):
        if ndc:
            _lib.call("knerf_generate_rays_ndc", c2w.ctypes.data, 1024, 1024, focal, N, None, 1000 + i, *out_ptrs(), st)
        else:
            _lib.call("knerf_generate_rays", c2w.ctypes.data, 1024, 1024, focal, 2.0, 6.0, N, None, 1000 + i,
                      *out_ptrs(), st)

    arms = {"rays": (rays, False), "rays_ndc": (rays, True), "ray_batch": (batch, False),
            "ray_batch_ndc": (batch, True)}

    def time(fn, ndc):
        for i in range(10):
            fn(i, ndc)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(launches):
            fn(i, ndc)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e6 / (launches * R)          # ns per ray

    res = {k: [] for k in arms}
    for _ in range(5):
        for k, (fn, ndc) in arms.items():
            res[k].append(time(fn, ndc))
    # bytes the algorithm needs per ray: writes o, d (24), t (4N); the batch kernels also write target (12) and read
    # one 16-byte cached pixel
    need = {"rays": 24 + 4 * N, "rays_ndc": 24 + 4 * N, "ray_batch": 24 + 4 * N + 28, "ray_batch_ndc": 24 + 4 * N + 28}
    out = {"mode": "kernel", "card": card(), "rays": R, "n_samples": N, "cache_views": n_img, "view_wh": HW,
           "launches": launches}
    for k, v in res.items():
        ns = float(np.median(v))
        out[k] = {"ns_per_ray": round(ns, 4), "runs_ns_per_ray": [round(x, 4) for x in v],
                  "bytes_per_ray": need[k], "GB_per_s": round(need[k] / ns, 1)}
    print(json.dumps(out))


def convergence(steps=2000, every=250):
    from keras_nerf_b200 import NeRF
    from keras_nerf_b200.data.llff import LLFFDatasetLoader
    from keras_nerf_b200.data.synthetic import write_llff_like
    from keras_nerf_b200.model.nerf import mlp as mlp_mod
    dev = torch.device("cuda", 0)
    R = 4096
    tmp = tempfile.mkdtemp(prefix="knerf_llff_")
    write_llff_like(tmp, H=192, W=256, n_views=20)

    def run(ndc, draws):
        loader = LLFFDatasetLoader(tmp, factor=1, llffhold=8, ndc=ndc, device=dev)
        torch.manual_seed(draws)
        ds = loader.load_dataset(batch_size=1, n_sample=64, ray_batch=R)[0]
        ds.perm_seed = 1000 + draws
        gen = loader.rays_generator(64)
        held = [(loader.load_image(loader.image_paths[i]), gen(loader.poses[i], seed=500 + int(i)))
                for i in loader.i_test]
        mlp_mod.set_seed(42 + draws)
        m = NeRF(precision="bf16", records="fp8", device=dev)
        m.compile(optimizer="adam", loss="mse", batch_size=1, image_height=loader.H, image_width=loader.W,
                  ray_chunks=4096, white_background=False, ray_batch=R)

        def evaluate():
            mse = np.zeros(2)
            for img, (o, d, t) in held:
                res = m.predict_and_render_images((o[None], d[None], t[None]), seed=1)
                for j in range(2):
                    mse[j] += float(((res[j]["image"][0] - img[..., :3]) ** 2).mean()) / len(held)
            return [round(float(-10 * np.log10(x)), 3) for x in mse]

        per_epoch, curve = len(ds), []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            m.train_step(ds.batch(i // per_epoch, i % per_epoch, seed=draws * 100003 + i),
                         seed=draws * 7919 + 7000 + i)
            if (i + 1) % every == 0 or i + 1 == steps:
                c, f = evaluate()
                curve.append({"step": i + 1, "val_coarse_psnr": c, "val_fine_psnr": f})
        e1.record()
        torch.cuda.synchronize()
        last = [p["val_fine_psnr"] for p in curve if p["step"] > 0.7 * steps]
        return {"curve": curve, "fine_psnr_last_checkpoints_mean": round(float(np.mean(last)), 3),
                "near_far": [loader.near, loader.far], "seconds_incl_eval": round(e0.elapsed_time(e1) / 1e3, 2)}

    probe = LLFFDatasetLoader(tmp, factor=1, llffhold=8, ndc=False)
    out = {"mode": "convergence", "card": card(), "steps": steps, "rays_per_step": R, "samples": [64, 128],
           "H": probe.H, "W": probe.W, "views": len(probe.poses), "train_views": len(probe.i_train),
           "held_out_views": len(probe.i_test), "bounds_after_rescale": [float(probe.bds.min()), float(probe.bds.max())],
           "precision": "bf16 (fp8 records)"}
    for ndc in (True, False):
        for draws in (0, 1):
            out[f"{'ndc' if ndc else 'no_ndc'}_seed{draws}"] = run(ndc, draws)
    print(json.dumps(out))


if __name__ == "__main__":
    mode = sys.argv[1] if len(sys.argv) > 1 else "kernel"
    args = [int(a) for a in sys.argv[2:]]
    {"kernel": kernel, "convergence": convergence}[mode](*args)
