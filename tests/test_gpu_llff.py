"""GPU: knerf_generate_rays_ndc against an fp32 NumPy restatement in the kernel's op order (bit for bit) and against
vanilla NeRF's float64 ndc_rays, knerf_generate_ray_batch_ndc against the whole-view kernel, the LLFF loader on
write_llff_like directories, and train.py / inference.py --dataset_type llff end to end."""
import csv
import os

import numpy as np
import pytest
import torch

import llff_oracle as LO
import oracle as O
from ray_batch_oracle import permute

pytestmark = pytest.mark.gpu

f32 = np.float32


def _pose(seed):
    """a forward-facing camera: a few degrees of rotation, a small offset"""
    rng = np.random.default_rng(seed)
    k = rng.normal(size=3)
    k /= np.linalg.norm(k)
    a = np.radians(rng.uniform(2, 8))
    K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    c2w = np.eye(4)
    c2w[:3, :3] = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    c2w[:3, 3] = rng.normal(size=3) * 0.2
    return c2w.astype(np.float32)


def ndc_rays_fp32(c2w, H, W, focal, N, u):
    """knerf_generate_rays_ndc restated in fp32 NumPy, every operation rounded on its own in the kernel's order ->
    (o [HW,3], d [HW,3], t [HW,N], s [HW,N], |d_ndc| [HW])"""
    c2w, focal = np.asarray(c2w, f32), f32(focal)
    y, x = np.divmod(np.arange(H * W), W)
    xc = (x.astype(f32) - f32(W) * f32(0.5)) / focal
    yc = (y.astype(f32) - f32(H) * f32(0.5)) / focal
    R = c2w[:3, :3]
    w = np.stack([(xc * R[i, 0] + (-yc) * R[i, 1]) + (f32(-1) * R[i, 2]) for i in range(3)], -1)
    nrm = np.sqrt((w[:, 0] * w[:, 0] + w[:, 1] * w[:, 1]) + w[:, 2] * w[:, 2])
    w = w / nrm[:, None]
    o = np.broadcast_to(c2w[:3, 3], w.shape)
    sx, sy = (f32(-2) * focal) / f32(W), (f32(-2) * focal) / f32(H)
    tau = (-(f32(1) + o[:, 2])) / w[:, 2]
    op = o + tau[:, None] * w
    rx, ry, q = op[:, 0] / op[:, 2], op[:, 1] / op[:, 2], f32(2) / op[:, 2]
    o_ndc = np.stack([sx * rx, sy * ry, f32(1) + q], -1)
    dn = np.stack([sx * (w[:, 0] / w[:, 2] - rx), sy * (w[:, 1] / w[:, 2] - ry), -q], -1)
    dnorm = np.sqrt((dn[:, 0] * dn[:, 0] + dn[:, 1] * dn[:, 1]) + dn[:, 2] * dn[:, 2])
    # the stratified depths of knerf_generate_rays for near = 0, far = 1
    delta, interval = f32(1) / f32(N - 1) if N > 1 else f32(0), f32(1) / f32(N)
    i = np.arange(N)
    lin = delta * i.astype(f32)
    lin[N - 1], lin[0] = f32(1), f32(0)
    noise = np.asarray(u, f32).reshape(H * W, N) * interval - interval * f32(0.5)
    s = np.minimum(np.maximum(lin[None] + noise, f32(0)), f32(1))
    return o_ndc, dn / dnorm[:, None], dnorm[:, None] * s, s, dnorm


def _uniform(n, seed):
    from keras_nerf_b200 import _lib
    out = torch.empty(n, dtype=torch.float32, device="cuda")
    _lib.call("knerf_uniform", _lib.ptr(out), n, seed, 0, _lib.stream())
    return out.cpu().numpy()


@pytest.mark.parametrize("N", [64, 7])
@pytest.mark.parametrize("philox", [False, True])
def test_whole_view_kernel_bits_and_vanilla(N, philox):
    from keras_nerf_b200 import RaysGenerator
    H, W, focal = 29, 37, 33.5
    for seed in range(3):
        c2w = _pose(seed)
        gen = RaysGenerator(focal, W, H, 123.0, 456.0, N, ndc=True)      # near / far are not used with ndc
        if philox:
            o, d, t = gen(c2w, seed=1000 + seed)
            u = _uniform(H * W * N, 1000 + seed)
            o2, d2, t2 = gen(c2w, u=u.reshape(H, W, N))
            assert torch.equal(o, o2) and torch.equal(d, d2) and torch.equal(t, t2)
        else:
            u = O.uniform24(np.random.default_rng(seed), (H, W, N))
            o, d, t = gen(c2w, u=u)
        assert o.shape == (H, W, 3) and t.shape == (H, W, N)
        ro, rd, rt, s, dnorm = ndc_rays_fp32(c2w, H, W, focal, N, u)
        for got, want in ((o, ro), (d, rd), (t, rt)):
            np.testing.assert_array_equal(got.reshape(H * W, -1).cpu().numpy(), want)   # the same bits
        # vanilla NeRF in float64: ndc_rays(near = 1) of the unnormalised world rays
        wo, wd = LO.world_rays(c2w, H, W, focal)
        vo, vd = LO.ndc_rays(H, W, focal, 1.0, wo.reshape(-1, 3), wd.reshape(-1, 3))
        o64, d64, t64 = (x.reshape(H * W, -1).cpu().double().numpy() for x in (o, d, t))
        assert np.abs(o64 - vo).max() <= 1e-5
        assert np.abs(d64 - vd / np.linalg.norm(vd, axis=-1, keepdims=True)).max() <= 1e-5
        pts = o64[:, None] + d64[:, None] * t64[..., None]
        assert np.abs(pts - (vo[:, None] + s.astype(np.float64)[..., None] * vd[:, None])).max() <= 1e-5
        # the samples run from the near plane z = -1 to infinity, z = 1
        assert pts[..., 2].min() >= -1 - 1e-5 and pts[..., 2].max() <= 1 + 1e-5
        mid = gen(c2w, u=np.full((H, W, N), 0.5, np.float32))              # no jitter: the end points themselves
        z = (mid[0][..., 2:3] + mid[1][..., 2:3] * mid[2]).double()
        assert float((z[..., 0] + 1).abs().max()) <= 1e-5 and float((z[..., -1] - 1).abs().max()) <= 1e-5


@pytest.mark.parametrize("N", [64, 7])
def test_batch_kernel_is_the_whole_view_kernel(N):
    from keras_nerf_b200 import RaysGenerator
    from keras_nerf_b200.data.rays import generate_ray_batch
    n_img, H, W, focal = 3, 29, 37, 33.5
    P = n_img * H * W
    rng = np.random.default_rng(N)
    images = torch.from_numpy(rng.uniform(0, 1, (n_img, H, W, 4)).astype(np.float32)).cuda()
    poses = torch.from_numpy(np.stack([_pose(10 + k) for k in range(n_img)])).cuda()
    first, R = 211, 1500
    u = O.uniform24(np.random.default_rng(N + 1), (R, N))
    target, o, d, t, pixel = generate_ray_batch(images, poses, focal, 2.0, 6.0, N, 77, 2, first, R, u=u,
                                                with_pixel=True, ndc=True)
    pix = pixel.cpu().numpy()
    np.testing.assert_array_equal(pix, permute(np.arange(first, first + R), P, perm_seed=77, epoch=2))
    assert torch.equal(target, images.reshape(P, 4)[pixel, :3])
    gen = RaysGenerator(focal, W, H, 0.0, 1.0, N, ndc=True)
    seen = 0
    for v in range(n_img):
        rows = np.nonzero(pix // (H * W) == v)[0]
        q = torch.from_numpy(pix[rows] - v * H * W).cuda()
        u_full = np.zeros((H * W, N), np.float32)
        u_full[pix[rows] - v * H * W] = u[rows]
        ov, dv, tv = gen(poses[v].cpu().numpy(), u=u_full.reshape(H, W, N))
        r = torch.from_numpy(rows).cuda()
        for got, ref, k in ((o, ov, 3), (d, dv, 3), (t, tv, N)):
            assert torch.equal(got[r], ref.reshape(H * W, k)[q])
        seen += len(rows)
    assert seen == R
    # and the RayBatchDataset of the loader draws exactly these rays
    from keras_nerf_b200.data.loader import RayBatchDataset
    ds = RayBatchDataset(images, poses, focal, 0.0, 1.0, N, R, perm_seed=77, ndc=True)
    b = generate_ray_batch(images, poses, focal, 0.0, 1.0, N, 77, 0, 0, R, seed=5, ndc=True)
    got = ds.batch(0, 0, seed=5)
    assert torch.equal(got[0], b[0]) and all(torch.equal(x, y) for x, y in zip(got[1], b[1:]))


@pytest.mark.parametrize("prefactored", [True, False])
def test_loader_on_llff_like_directories(tmp_path, prefactored):
    from PIL import Image

    from keras_nerf_b200.data import llff as L
    from keras_nerf_b200.data.loader import RayBatchDataset
    from keras_nerf_b200.data.synthetic import write_llff_like
    d = write_llff_like(str(tmp_path / "s"), H=36, W=48, n_views=10, factors=(2,) if prefactored else ())
    loader = L.LLFFDatasetLoader(d, factor=2, llffhold=4)
    assert (loader.H, loader.W, loader.resize) == (18, 24, not prefactored)
    train, val, test = loader.load_dataset(batch_size=1, n_sample=16)
    assert (len(train), len(val), len(test)) == (7, 3, 3)
    assert [int(i) for i in loader.i_test] == [0, 4, 8]
    view = loader.load_image(loader.image_paths[5])
    assert view.shape == (18, 24, 4) and bool((view[..., 3] == 1).all())
    png = np.asarray(Image.open(loader.image_paths[5]).convert("RGB"), np.float32) / 255.0
    if prefactored:           # the PNG's pixel (y, x) is the view's (y, x)
        np.testing.assert_allclose(view[..., :3].cpu().numpy(), png, atol=1e-6)
    else:                     # the antialiased 2x reduction of the full-size PNG, in the same orientation
        ref = torch.nn.functional.interpolate(torch.from_numpy(png).permute(2, 0, 1)[None], size=(18, 24),
                                              mode="bilinear", antialias=True, align_corners=False)[0]
        err = (view[..., :3].cpu() - ref.permute(1, 2, 0)).abs()
        assert float(err.mean()) <= 0.02, float(err.mean())
    # poses: the Dataset's cameras are the loader's recentred poses, which match vanilla's float64 arithmetic
    ref = LO.load_poses(np.load(os.path.join(d, "poses_bounds.npy")))
    np.testing.assert_allclose(loader.poses[:, :3, :4], ref["recentred"][:, :, :4], atol=1e-6)
    assert [np.asarray(c, np.float32).tolist() for c in test.camera_params] == \
        [loader.poses[i].tolist() for i in (0, 4, 8)]
    images, rays = next(iter(test))
    assert images.shape == (1, 18, 24, 4) and rays[0].shape == (1, 18, 24, 3) and rays[2].shape == (1, 18, 24, 16)
    assert float(rays[0][..., 2].max()) <= -1 + 1e-4                       # NDC origins on the near plane z = -1
    rb = loader.load_dataset(batch_size=1, n_sample=16, ray_batch=512)[0]
    assert isinstance(rb, RayBatchDataset) and rb.ndc and rb.images.shape == (7, 18, 24, 4)
    np.testing.assert_array_equal(rb.poses.cpu().numpy(), loader.poses[loader.i_train])
    assert torch.equal(rb.images[4], loader.load_image(loader.image_paths[int(loader.i_train[4])]))


def test_train_and_inference_scripts_llff(tmp_path):
    import inference
    import train
    from PIL import Image

    from keras_nerf_b200 import NeRF
    from keras_nerf_b200.data.synthetic import write_llff_like
    # 45 x 63 views: no power of two divides them.  The scripts render in chunks of 945 (the largest divisor <= 1024)
    # while the 2,048-ray training batches keep chunks of 1,024
    d = write_llff_like(str(tmp_path / "scene"), H=90, W=126, n_views=10, factors=(2,))
    base = ["--data_dir", d, "--dataset_type", "llff", "--factor", "2", "--llffhold", "8", "--batch_size", "1",
            "--ray_chunks", "1024", "--log_freq", "1", "--precision", "bf16", "--num_epochs", "2"]
    for name, extra in (("views", []), ("rays", ["--ray_batch", "2048"])):
        logs, models = str(tmp_path / f"logs_{name}"), str(tmp_path / f"model_{name}")
        nerf = train.main(base + ["--name", name, "--log_dir", logs, "--model_dirs", models] + extra, multi_gpu=False)
        assert nerf.ray_chunks == 945
        if extra:
            assert nerf._train_ray_chunks * nerf._train_chunks == 2048 and nerf._train_ray_chunks % 1024 == 0
        run = os.path.join(logs, name)
        rows = list(csv.DictReader(open(os.path.join(run, "log.csv"))))
        assert [int(r["epoch"]) for r in rows] == [0, 1]
        assert float(rows[1]["fine_loss"]) < float(rows[0]["fine_loss"]), rows
        assert np.isfinite(float(rows[1]["val_fine_loss"]))
        assert NeRF.has_checkpoint(os.path.join(run, "model")) and NeRF.has_checkpoint(os.path.join(models, name))
    out = inference.main(["--model_dirs", os.path.join(models, "rays"), "--dataset_type", "llff", "--data_dir", d,
                          "--factor", "2", "--output_dir", str(tmp_path / "out"), "--precision", "bf16"])
    with Image.open(out) as gif:
        assert gif.size == (63, 45) and gif.n_frames == 120


def test_compile_llff_view_size_with_power_of_two_ray_batch():
    """378 x 504 (an LLFF scene at factor 8) with 4,096-ray batches: rendering and training keep chunks near the
    requested 1,024 instead of the 16 rays both sizes share"""
    from keras_nerf_b200 import NeRF
    from keras_nerf_b200.data.llff import ray_chunks_for
    render, train_rc = ray_chunks_for(378 * 504, 4096, 1024)
    m = NeRF(precision="bf16")
    m.compile(optimizer="adam", loss="mse", batch_size=1, image_height=378, image_width=504, ray_chunks=render,
              ray_batch=4096, train_ray_chunks=train_rc)
    assert (m.ray_chunks, m.sequential_chunks) == (1008, 189)
    assert m._train_ray_chunks * m._train_chunks == 4096 and m._train_ray_chunks % 1024 == 0
    m2 = NeRF(precision="bf16")
    m2.compile(optimizer="adam", loss="mse", batch_size=1, image_height=378, image_width=504, ray_chunks=render,
               ray_batch=4032)           # without train_ray_chunks the render chunk trains too, as before
    assert m2._train_ray_chunks * m2._train_chunks == 4032 and 4032 % m2._train_ray_chunks == 0
