"""GPU: knerf_generate_ray_batch against the NumPy permutation and knerf_generate_rays, RayBatchDataset rank slices,
the ray-batch training step against the whole-image one, and train.py --ray_batch end to end."""
import csv
import os

import numpy as np
import pytest
import torch

import oracle as O
from ray_batch_oracle import permute

pytestmark = pytest.mark.gpu

NEAR, FAR = 2.0, 6.0


def _cache(n_img, H, W, seed=0):
    from keras_nerf_b200 import pose_spherical
    rng = np.random.default_rng(seed)
    images = torch.from_numpy(rng.uniform(0, 1, (n_img, H, W, 4)).astype(np.float32)).cuda()
    poses = torch.tensor(np.stack([pose_spherical(360.0 * k / n_img + 11.0, -30.0 + 7 * k, 4.0)
                                   for k in range(n_img)]), dtype=torch.float32).cuda()
    return images, poses


def _batch(images, poses, focal, N, epoch, first, R, u=None, seed=0, perm_seed=77):
    from keras_nerf_b200.data.rays import generate_ray_batch
    return generate_ray_batch(images, poses, focal, NEAR, FAR, N, perm_seed, epoch, first, R, u=u, seed=seed,
                              with_pixel=True)


@pytest.mark.parametrize("N", [64, 7])
def test_batch_matches_permutation_and_per_view_rays(N):
    from keras_nerf_b200 import RaysGenerator
    n_img, H, W, focal = 3, 37, 29, 31.5
    P = n_img * H * W
    images, poses = _cache(n_img, H, W)
    first, R = 517, 1001
    u = O.uniform24(np.random.default_rng(N), (R, N))
    target, o, d, t, pixel = _batch(images, poses, focal, N, 3, first, R, u=u)
    want = permute(np.arange(first, first + R), P, perm_seed=77, epoch=3).astype(np.int64)
    pix = pixel.cpu().numpy()
    np.testing.assert_array_equal(pix, want)
    assert torch.equal(target, images.reshape(P, 4)[pixel, :3])
    gen = RaysGenerator(focal, W, H, NEAR, FAR, N)
    seen = 0
    for v in range(n_img):
        rows = np.nonzero(pix // (H * W) == v)[0]
        q = torch.from_numpy(pix[rows] - v * H * W).cuda()
        u_full = np.zeros((H * W, N), np.float32)
        u_full[pix[rows] - v * H * W] = u[rows]
        ov, dv, tv = gen(poses[v].cpu().numpy(), u=u_full.reshape(H, W, N))
        r = torch.from_numpy(rows).cuda()
        for got, ref, k in ((o, ov, 3), (d, dv, 3), (t, tv, N)):
            assert torch.equal(got[r], ref.reshape(H * W, k)[q])          # the same bits, not just close
        seen += len(rows)
    assert seen == R


def test_full_epoch_windows_and_repeat():
    n_img, H, W, N, focal = 3, 37, 29, 8, 31.5
    P = n_img * H * W
    images, poses = _cache(n_img, H, W, seed=1)
    u = O.uniform24(np.random.default_rng(5), (P, N))
    whole = _batch(images, poses, focal, N, 1, 0, P, u=u)
    assert torch.equal(torch.sort(whole[4]).values, torch.arange(P, device="cuda"))
    cuts = [0, 1, 33, 34, 1000, 2222, P]
    parts = [_batch(images, poses, focal, N, 1, a, b - a, u=u[a:b]) for a, b in zip(cuts[:-1], cuts[1:])]
    for k in range(5):
        assert torch.equal(torch.cat([p[k] for p in parts]), whole[k]), k
    again = _batch(images, poses, focal, N, 1, 0, P, u=u)
    assert all(torch.equal(a, b) for a, b in zip(again, whole))
    # Philox jitter: the same seed gives the same bytes, another epoch another order
    a = _batch(images, poses, focal, N, 2, 100, 500, seed=9)
    b = _batch(images, poses, focal, N, 2, 100, 500, seed=9)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert not torch.equal(_batch(images, poses, focal, N, 3, 100, 500, seed=9)[4], a[4])


def test_philox_depths_stay_in_their_strata():
    n_img, H, W, N, focal = 3, 37, 29, 64, 31.5
    images, poses = _cache(n_img, H, W, seed=2)
    t = _batch(images, poses, focal, N, 0, 0, 3000, seed=1234)[3].double()
    lin = torch.linspace(NEAR, FAR, N, dtype=torch.float64, device="cuda")
    half = (FAR - NEAR) / N / 2
    assert float((t - lin).abs().max()) <= half + 1e-5
    assert float(t.min()) >= NEAR and float(t.max()) <= FAR
    assert float(t.std(0).min()) > 0.1 * half            # actually jittered


def test_rank_slices_union_is_the_single_process_batch():
    from keras_nerf_b200.data.loader import RayBatchDataset
    images, poses = _cache(3, 37, 29, seed=3)
    N = 256
    mk = lambda n, r, w: RayBatchDataset(images, poses, 31.5, NEAR, FAR, 16, n, rank=r, world=w, perm_seed=5)  # noqa
    r0, r1, single = mk(N, 0, 2), mk(N, 1, 2), mk(2 * N, 0, 1)
    assert len(r0) == len(r1) == len(single)
    for step in (0, 3, len(single) - 1):
        a = r0.batch(4, step, seed=1, with_pixel=True)
        b = r1.batch(4, step, seed=1, with_pixel=True)
        s = single.batch(4, step, seed=1, with_pixel=True)
        assert not set(a[2].tolist()) & set(b[2].tolist())
        assert torch.equal(torch.cat([a[2], b[2]]), s[2])
        assert torch.equal(torch.cat([a[0], b[0]]), s[0])
        for k in range(2):
            assert torch.equal(torch.cat([a[1][k], b[1][k]]), s[1][k])


def test_train_step_on_a_ray_batch_is_the_image_step():
    """fp32: N flat rays train like the same rays laid out as a [1, N/w, w] image with the same fine draws, seed and
    chunking.  The forward is deterministic, so the rendered pixels are the same bits.  The fp32 weight-gradient
    kernels flush with atomics whose order differs run to run, so gradients agree to the fp32 summation order."""
    from keras_nerf_b200 import NeRF, RaysGenerator, pose_spherical
    from keras_nerf_b200.model.nerf import mlp as mlp_mod
    images, poses = _cache(4, 24, 20, seed=4)
    N, w = 512, 256
    target, o, d, t, _ = _batch(images, poses, 25.0, 64, 0, 960, N, seed=3)
    u_f = O.uniform24(np.random.default_rng(6), (N, 128))
    mlp_mod.set_seed(42)
    old = NeRF(precision="fp32")
    old.compile(optimizer="adam", loss="mse", batch_size=1, image_height=N // w, image_width=w, ray_chunks=w,
                white_background=True)
    mlp_mod.set_seed(42)
    new = NeRF(precision="fp32")
    new.compile(optimizer="adam", loss="mse", batch_size=1, image_height=16, image_width=16, ray_chunks=w,
                white_background=True, ray_batch=N)
    assert (new._train_ray_chunks, new._train_chunks) == (old._train_ray_chunks, old._train_chunks) == (w, 2)
    img = lambda x: x.reshape(1, N // w, w, x.shape[-1])  # noqa: E731
    ci_o, fi_o = old.accumulate_gradients(img(target), (img(o), img(d), img(t)), u_fine=u_f, seed=11)
    ci_n, fi_n = new.accumulate_gradients(target, (o, d, t), u_fine=u_f, seed=11)
    assert ci_n.shape == (N, 3)
    assert torch.equal(ci_n, ci_o.reshape(N, 3)) and torch.equal(fi_n, fi_o.reshape(N, 3))
    for a, b in ((old._grad_flat, new._grad_flat), (old._losses, new._losses)):
        assert float((a - b).abs().max()) <= 1e-5 * float(a.abs().max())
    old.apply_gradients()
    new.apply_gradients()
    new._losses.zero_()
    old._losses.zero_()
    logs = new.train_step((target, (o, d, t)), u_fine=u_f, seed=12)
    ref = old.train_step((img(target), (img(o), img(d), img(t))), u_fine=u_f, seed=12)
    assert set(logs) == set(ref) and np.isnan(logs["fine_ssim"]) and np.isnan(logs["coarse_ssim"])
    for k in ("coarse_loss", "fine_loss", "coarse_psnr", "fine_psnr"):       # the PSNR of the batch MSE
        assert abs(logs[k] - ref[k]) <= 1e-4 * max(1.0, abs(ref[k])), k
    # rendering still works at the compiled image shape
    ro, rd, rt = RaysGenerator(25.0, 16, 16, NEAR, FAR, 64)(pose_spherical(30.0, -30.0, 4.0), seed=2)
    c, f = new.predict_and_render_images((ro[None], rd[None], rt[None]), seed=1)
    assert f["image"].shape == (1, 16, 16, 3) and bool(torch.isfinite(f["image"]).all())
    for m in new.metrics:
        m.reset_state()
    logs = new.test_step((torch.rand(1, 16, 16, 4, device="cuda"), (ro[None], rd[None], rt[None])), seed=1)
    assert np.isfinite(logs["fine_psnr"]) and np.isfinite(logs["fine_ssim"])


def test_train_script_ray_batch(tmp_path):
    import train
    from keras_nerf_b200.data.synthetic import write_nerf_synthetic_like
    d = write_nerf_synthetic_like(str(tmp_path / "scene"), image_wh=64, n_train=8, n_val=1, n_test=1)
    logs, models = str(tmp_path / "logs"), str(tmp_path / "model")
    train.main(["--name", "ball", "--data_dir", d, "--img_wh", "64", "--white_bg", "--batch_size", "1",
                "--ray_chunks", "1024", "--log_dir", logs, "--model_dirs", models, "--log_freq", "1",
                "--precision", "bf16", "--ray_batch", "4096", "--num_epochs", "2"], multi_gpu=False)
    run = os.path.join(logs, "ball")
    rows = list(csv.DictReader(open(os.path.join(run, "log.csv"))))
    assert [int(r["epoch"]) for r in rows] == [0, 1]
    assert {"coarse_loss", "fine_loss", "fine_psnr", "fine_ssim", "val_fine_loss", "val_fine_ssim"} <= set(rows[0])
    assert np.isfinite(float(rows[1]["val_fine_ssim"]))
    assert float(rows[1]["fine_loss"]) < float(rows[0]["fine_loss"])
    from keras_nerf_b200 import NeRF
    assert NeRF.has_checkpoint(os.path.join(run, "model")) and NeRF.has_checkpoint(os.path.join(models, "ball"))
