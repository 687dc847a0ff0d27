#!/usr/bin/env python
"""Generate tests/golden/*.npz by EXECUTING THE REFERENCE'S OWN PYTHON (unmodified, imported from
/root/reference) over oracle/tfshim (a torch-CPU stand-in for the tf.* ops; TensorFlow itself is
not installable offline).  Run in the build container only:

    python tests/golden/make_golden.py

The fixtures are small (sub-sampled where the full tensor would be large) and committed; nothing at
test time reads /root/reference.  Random draws are pushed into the shim's tf.random.uniform queue so
the very same numbers can be fed to the oracle and to the CUDA path.
"""
import contextlib
import hashlib
import io
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("KNERF_REFERENCE", "/root/reference")
sys.path.insert(0, os.path.join(ROOT, "oracle", "tfshim"))
sys.path.insert(1, REF)
sys.path.insert(2, ROOT)

import tensorflow as tf  # noqa: E402  (the shim)
from keras_nerf.data.rays import RaysGenerator  # noqa: E402  (reference code)
from keras_nerf.data.utils import get_focal_from_fov, pose_spherical  # noqa: E402
from keras_nerf.model.nerf.mlp import NeRFMLP  # noqa: E402
from keras_nerf.model.nerf.nerf import NeRF  # noqa: E402
from keras_nerf.model.nerf.utils import NeRFUtils  # noqa: E402

assert tf.__file__.startswith(os.path.join(ROOT, "oracle", "tfshim")), tf.__file__

LEGO_POSE = np.array([  # tests/data/test_rays.py:21-47
    [-0.9999021887779236, 0.004192245192825794, -0.013345719315111637, -0.05379832163453102],
    [-0.013988681137561798, -0.2996590733528137, 0.95394366979599, 3.845470428466797],
    [-4.656612873077393e-10, 0.9540371894836426, 0.29968830943107605, 1.2080823183059692],
    [0.0, 0.0, 0.0, 1.0]], dtype=np.float32)


def uniform24(rng, shape):
    return (rng.integers(0, 1 << 24, size=shape, dtype=np.int64).astype(np.float32) * np.float32(2.0 ** -24))


def npy(x):
    if isinstance(x, tf.Variable):
        return x.numpy()
    return x.detach().numpy() if torch.is_tensor(x) else np.asarray(x)


def save(name, **arrs):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **{k: np.asarray(v) for k, v in arrs.items()})
    print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB")


def digest(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest()[:8], dtype=np.uint64)


def tensor_summary(flat_list):
    """per-tensor (sum, abs-sum, first 32 entries) -- small stand-in for 595,844-float tensors."""
    sums = np.array([float(np.sum(a, dtype=np.float64)) for a in flat_list])
    asum = np.array([float(np.sum(np.abs(a), dtype=np.float64)) for a in flat_list])
    head = np.stack([np.resize(a.reshape(-1)[:32], 32) if a.size >= 32
                     else np.pad(a.reshape(-1), (0, 32 - a.size)) for a in flat_list])
    return sums, asum, head.astype(np.float32)


def main():
    # a fixed thread count fixes the CPU summation order test_oracle_golden.py replays (golden_threads fixture)
    torch.set_num_threads(8)
    # ---- a1/a2: focal + orbit poses --------------------------------------------------------
    focal = float(get_focal_from_fov(0.6911112070083618, 100))
    thetas = np.array([0.0, 9.0, 45.0, 180.0, 351.0], dtype=np.float64)
    poses = np.stack([npy(pose_spherical(float(t), -30.0, 4.0)) for t in thetas])
    save("camera", focal=np.float64(focal), fov=np.float64(0.6911112070083618), width=np.int64(100),
         thetas=thetas, phi=np.float64(-30.0), radius=np.float64(4.0), poses=poses)

    # ---- a3: rays on the reference's own fixture -------------------------------------------
    H = W = 128
    N = 32
    rng = np.random.default_rng(1234)
    u = uniform24(rng, (H, W, N))
    gen = RaysGenerator(focal_length=138.88887889922103, image_width=W, image_height=H,
                        near=2.0, far=6.0, n_sample=N)
    tf.random.queue.append(u)
    o, d, t = (npy(x) for x in gen(tf.constant(LEGO_POSE, dtype=tf.float32)))
    rows = np.array([0, 1, 63, 64, 127])
    save("rays", pose=LEGO_POSE, focal=np.float64(138.88887889922103), H=np.int64(H), W=np.int64(W),
         N=np.int64(N), near=np.float64(2.0), far=np.float64(6.0), rows=rows,
         u_rows=u[rows], o_rows=o[rows], d=d, t_rows=t[rows], u_digest=digest(u), t_digest=digest(t))

    # ---- a4/a5: positional encoding ---------------------------------------------------------
    rng = np.random.default_rng(7)
    R, S = 64, 16
    utils = NeRFUtils(batch_size=1, image_height=8, image_width=8, ray_chunks=R, pos_emb_xyz=10,
                      pos_emb_dir=4, white_background=True)
    oo = rng.uniform(-4, 4, (R, 3)).astype(np.float32)
    dd = rng.normal(size=(R, 3)).astype(np.float32)
    dd /= np.linalg.norm(dd, axis=-1, keepdims=True)
    tt = np.sort(rng.uniform(2, 6, (R, S)).astype(np.float32), axis=-1)
    xyz, dirs = utils.encode_position_and_directions(tf.constant(oo), tf.constant(dd), tf.constant(tt))
    pe = utils.positional_encoding(tf.constant(oo), 10)
    save("posenc", o=oo, d=dd, t=tt, xyz=npy(xyz), dirs=npy(dirs), pe_o=npy(pe))

    # ---- a7: compositing (chunk form with white bg + clip; full-image form without) ---------
    for S in (32, 64, 192):
        hw = 16 if S == 32 else 8
        R = hw * hw
        rng = np.random.default_rng(100 + S)
        util_w = NeRFUtils(1, hw, hw, R, 10, 4, white_background=True)
        util_b = NeRFUtils(1, hw, hw, R, 10, 4, white_background=False)
        rgb = rng.uniform(0, 1, (R, S, 3)).astype(np.float32)
        scale = np.where(rng.uniform(size=(R, 1)) < 0.25, 400.0, 8.0).astype(np.float32)
        sigma = (rng.uniform(0, 1, (R, S, 1)) ** 3).astype(np.float32) * scale[..., None]
        sigma[rng.uniform(size=sigma.shape) < 0.3] = 0.0
        t = np.sort(rng.uniform(2, 6, (R, S)).astype(np.float32), axis=-1)
        iw, dw, ww = (npy(x) for x in util_w.render_image_depth_chunk(tf.constant(rgb), tf.constant(sigma), tf.constant(t)))
        ib, db, wb = (npy(x) for x in util_b.render_image_depth_chunk(tf.constant(rgb), tf.constant(sigma), tf.constant(t)))
        full = NeRFUtils(1, hw, hw, R, 10, 4)
        with contextlib.redirect_stdout(io.StringIO()):      # the reference has debug print()s here
            i4, d4, w4 = (npy(x) for x in full.render_image_depth(
                tf.constant(rgb.reshape(1, hw, hw, S, 3)), tf.constant(sigma.reshape(1, hw, hw, S, 1)),
                tf.constant(t.reshape(1, hw, hw, S))))
        save(f"composite_S{S}", rgb=rgb, sigma=sigma, t=t, image_white=iw, depth_white=dw, weights_white=ww,
             image_black=ib, depth_black=db, weights_black=wb, image_full=i4, depth_full=d4, weights_full=w4)

    # ---- a8: hierarchical sampling, recording the cdf / indices the reference computed ------
    rec = {}
    orig_ss = tf.searchsorted

    def recording_searchsorted(cdf, uu, side="left", **kw):
        out = orig_ss(cdf, uu, side=side, **kw)
        rec["cdf"], rec["idx"], rec["side"] = npy(cdf).copy(), npy(out).copy(), side
        return out

    tf.searchsorted = recording_searchsorted
    for (Nc, Nf, tag) in ((64, 128, "flagship"), (32, 64, "reftest")):
        R = 128
        rng = np.random.default_rng(200 + Nc)
        ut = NeRFUtils(1, 16, 8, R, 10, 4, True)
        t_c = np.sort(rng.uniform(2, 6, (R, Nc)).astype(np.float32), axis=-1)
        mid = (0.5 * (t_c[..., 1:] + t_c[..., :-1])).astype(np.float32)
        w = rng.uniform(0, 1, (R, Nc)).astype(np.float32)
        w[R // 2:] = (w[R // 2:] ** 8)                       # peaked rows
        w[R // 2:, :] *= (rng.uniform(size=(R - R // 2, Nc)) < 0.2)
        w[-1] = 0.0                                           # all-zero weights row
        uu = uniform24(rng, (R, Nf))
        uu[0, :4] = [0.0, 1.0 - 2.0 ** -24, 0.5, 2.0 ** -24]
        tf.random.queue.append(uu)
        tf.config.gather_oob = "zero"
        s = npy(ut.fine_hierarchical_sampling_chunk(tf.constant(mid), tf.constant(w), Nf))
        assert rec["side"] == "right"
        raised = False
        tf.random.queue.append(uu)
        tf.config.gather_oob = "raise"
        try:
            ut.fine_hierarchical_sampling_chunk(tf.constant(mid), tf.constant(w), Nf)
        except IndexError:
            raised = True
        tf.config.gather_oob = "zero"
        save(f"sampler_{tag}", t_c=t_c, mid=mid, weights=w, u=uu, samples=s, cdf=rec["cdf"],
             idx=rec["idx"].astype(np.int32), cpu_gather_raises=np.bool_(raised))
    tf.searchsorted = orig_ss

    # ---- a6: MLP (reference's own unit-test widths: 99/99, and the flagship 63/27) ----------
    for (dx, dd_, tag) in ((63, 27, "flagship"), (99, 99, "reftest")):
        tf.keras.init_rng = np.random.default_rng(42)
        mlp = NeRFMLP(n_layers=8, dense_units=256, skip_layer=4)
        rng = np.random.default_rng(300 + dx)
        R, S = 24, 16
        x = rng.uniform(-1, 1, (R, S, dx)).astype(np.float32)
        dr = rng.uniform(-1, 1, (R, S, dd_)).astype(np.float32)
        rgb, sig = mlp((tf.constant(x), tf.constant(dr)))
        flat = np.concatenate([v.numpy().reshape(-1) for v in mlp.trainable_variables])
        names = [v.name for v in mlp.trainable_variables]
        save(f"mlp_{tag}", x=x, dirs=dr, rgb=npy(rgb), sigma=npy(sig), weights_digest=digest(flat),
             n_params=np.int64(flat.size), var_names=np.array(names), init_seed=np.int64(42))

    # ---- a9/a10/a11/a13: whole model through NeRF.predict_and_render_images and train_step --
    H = W = 16
    B, chunks = 1, 128
    tf.keras.init_rng = np.random.default_rng(42)
    nerf = NeRF()                                             # 64 / 128 / 10 / 4 / 8 / 256 / 4
    nerf.compile(optimizer="adam", loss=tf.keras.losses.MeanSquaredError(), batch_size=B,
                 image_height=H, image_width=W, ray_chunks=chunks, white_background=True)
    # _build_model draws its dummy inputs from tf.random.uniform (generator fallback) -- harmless.
    w0_c = np.concatenate([v.numpy().reshape(-1) for v in nerf.coarse.trainable_variables])
    w0_f = np.concatenate([v.numpy().reshape(-1) for v in nerf.fine.trainable_variables])
    focal16 = float(get_focal_from_fov(0.6911112070083618, W))
    gen = RaysGenerator(focal16, W, H, 2.0, 6.0, nerf.n_coarse)
    rng = np.random.default_rng(1234)
    u_c = uniform24(rng, (H, W, 64))
    tf.random.queue.append(u_c)
    pose = npy(pose_spherical(45.0, -30.0, 4.0))
    o, d, t = gen(tf.constant(pose))
    rays = (o[None], d[None], t[None])
    rng = np.random.default_rng(5678)
    n_chunks = (B * H * W) // chunks
    u_f = uniform24(rng, (B * H * W, 128))
    for i in range(n_chunks):
        tf.random.queue.append(u_f[i * chunks:(i + 1) * chunks])
    coarse, fine = nerf.predict_and_render_images(rays)
    render = {f"{k}_{n}": npy(v) for n, r in (("coarse", coarse), ("fine", fine)) for k, v in r.items()}

    rng = np.random.default_rng(99)
    images = rng.uniform(0, 1, (B, H, W, 4)).astype(np.float32)
    grads_rec = []
    for opt in (nerf.coarse_optimizer, nerf.fine_optimizer):
        orig = opt.apply_gradients

        def wrapped(gv, _orig=orig):
            gv = list(gv)
            grads_rec.append([npy(g).copy() for g, _ in gv])
            return _orig(gv)
        opt.apply_gradients = wrapped
    step_out = {}
    for step in range(2):
        for i in range(n_chunks):
            tf.random.queue.append(u_f[i * chunks:(i + 1) * chunks])
        for m in nerf.metrics:
            m.reset_state()
        met = nerf.train_step((tf.constant(images), rays))
        for k, v in met.items():
            step_out[f"s{step}_{k}"] = np.float64(float(v))
        for name, g in (("coarse", grads_rec[-2]), ("fine", grads_rec[-1])):
            sm, asm, head = tensor_summary(g)
            step_out[f"s{step}_grad_{name}_sum"] = sm
            step_out[f"s{step}_grad_{name}_abssum"] = asm
            step_out[f"s{step}_grad_{name}_head"] = head
        for name, net in (("coarse", nerf.coarse), ("fine", nerf.fine)):
            sm, asm, head = tensor_summary([v.numpy() for v in net.trainable_variables])
            step_out[f"s{step}_param_{name}_sum"] = sm
            step_out[f"s{step}_param_{name}_abssum"] = asm
            step_out[f"s{step}_param_{name}_head"] = head
    assert not tf.random.queue
    save("model", pose=pose, focal=np.float64(focal16), H=np.int64(H), W=np.int64(W), B=np.int64(B),
         ray_chunks=np.int64(chunks), u_coarse=u_c, u_fine=u_f, images=images,
         o=npy(o), d=npy(d), t=npy(t), w0_coarse_digest=digest(w0_c), w0_fine_digest=digest(w0_f),
         init_seed=np.int64(42), **render, **step_out)


if __name__ == "__main__":
    main()
