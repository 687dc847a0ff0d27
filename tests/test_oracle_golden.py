"""CPU: the oracle restatement against fixtures produced by the reference's own Python
(tests/golden/make_golden.py) and against the reference's own tests' assertions."""
import numpy as np
import pytest
import torch

import oracle as O
from conftest import load_golden

T = torch.from_numpy


def close(a, b, atol, rtol=0.0):
    a = a.detach().numpy() if torch.is_tensor(a) else np.asarray(a)
    np.testing.assert_allclose(a, np.asarray(b), atol=atol, rtol=rtol)


def test_focal_known_answer():
    # reference tests/data/test_utils.py:5-10 (the only known-answer test in the reference)
    assert O.get_focal_from_fov(0.6911112070083618, 100) == pytest.approx(138.88887889922103)
    g = load_golden("camera")
    assert O.get_focal_from_fov(float(g["fov"]), int(g["width"])) == float(g["focal"])


def test_pose_spherical():
    g = load_golden("camera")
    for th, pose in zip(g["thetas"], g["poses"]):
        close(O.pose_spherical(float(th), float(g["phi"]), float(g["radius"])), pose, atol=0)


def test_rays_reference_fixture():
    g = load_golden("rays")
    H, W, N = int(g["H"]), int(g["W"]), int(g["N"])
    rng = np.random.default_rng(1234)
    u = O.uniform24(rng, (H, W, N))
    rows = g["rows"]
    np.testing.assert_array_equal(u[rows], g["u_rows"])
    o, d, t = O.generate_rays(g["pose"], H, W, float(g["focal"]), float(g["near"]), float(g["far"]), N, u)
    close(o[rows], g["o_rows"], atol=0)
    close(d, g["d"], atol=1e-7)
    close(t[rows], g["t_rows"], atol=0)
    # the reference's own asserts (tests/data/test_rays.py:59-78)
    assert o.shape == (128, 128, 3) and d.shape == (128, 128, 3) and t.shape == (128, 128, 32)
    assert not torch.isnan(t).any()
    assert float(t.min()) >= 2.0 - 4.0 / 32 and float(t.max()) <= 6.0 + 4.0 / 32
    assert bool((t[..., 1:] > t[..., :-1]).all())          # SURVEY App. A1.7: strictly increasing


def test_positional_encoding():
    g = load_golden("posenc")
    xyz, dirs = O.encode_position_and_directions(g["o"], g["d"], g["t"], 10, 4)
    assert xyz.shape[-1] == 63 and dirs.shape[-1] == 27
    close(xyz, g["xyz"], atol=0)
    close(dirs, g["dirs"], atol=0)
    close(O.positional_encoding(T(g["o"]), 10), g["pe_o"], atol=0)


@pytest.mark.parametrize("S", [32, 64, 192])
def test_composite(S):
    g = load_golden(f"composite_S{S}")
    rgb, sigma, t = T(g["rgb"]), T(g["sigma"]), T(g["t"])
    for white, tag in ((True, "white"), (False, "black")):
        img, dep, w = O.render_image_depth_chunk(rgb, sigma, t, white)
        close(img, g[f"image_{tag}"], atol=1e-6)
        close(dep, g[f"depth_{tag}"], atol=2e-6)
        close(w, g[f"weights_{tag}"], atol=1e-7)
    img, dep, w = O.render_image_depth_chunk(rgb, sigma, t, False, clip=False)
    close(img.reshape(g["image_full"].shape), g["image_full"], atol=1e-6)
    close(w.reshape(g["weights_full"].shape), g["weights_full"], atol=1e-7)


def test_composite_backward_formula_matches_autograd():
    g = load_golden("composite_S64")
    rgb = T(g["rgb"]).clone().requires_grad_(True)
    sigma = T(g["sigma"])[..., 0].clone().requires_grad_(True)
    t = T(g["t"])
    for white in (True, False):
        img, _, _ = O.render_image_depth_chunk(rgb, sigma, t, white)
        tgt = torch.rand(img.shape, generator=torch.Generator().manual_seed(1))
        dimg = 2.0 * (img.detach() - tgt) / img.numel()
        gr, gs = torch.autograd.grad(((img - tgt) ** 2).mean(), [rgb, sigma])
        ar, as_ = O.composite_backward_analytic(rgb.detach(), sigma.detach(), t, dimg, white)
        close(ar, gr, atol=1e-9, rtol=1e-5)
        scale = float(gs.abs().max())
        close(as_ / scale, gs / scale, atol=2e-5)


@pytest.mark.parametrize("tag", ["flagship", "reftest"])
def test_sampler(tag):
    g = load_golden(f"sampler_{tag}")
    s, idx, cdf = O.fine_hierarchical_sampling_chunk(g["mid"], g["weights"], g["u"])
    close(cdf, g["cdf"], atol=0)
    np.testing.assert_array_equal(idx.numpy(), g["idx"])          # bit-exact bins
    close(s, g["samples"], atol=0)
    # bins stay bit-exact when the reference's cdf is handed in
    s2, idx2, _ = O.fine_hierarchical_sampling_chunk(g["mid"], g["weights"], g["u"], cdf=T(g["cdf"]))
    np.testing.assert_array_equal(idx2.numpy(), g["idx"])
    # TF-CPU gather raises on the out-of-range mid-point index (SURVEY App. C-1)
    assert bool(g["cpu_gather_raises"])
    with pytest.raises(IndexError):
        O.fine_hierarchical_sampling_chunk(g["mid"], g["weights"], g["u"], oob_mode=O.OOB_RAISE)
    sc, _, _ = O.fine_hierarchical_sampling_chunk(g["mid"], g["weights"], g["u"], oob_mode=O.OOB_CLAMP)
    assert float(sc.min()) >= float(g["mid"].min()) - 1e-6


@pytest.mark.parametrize("tag,dx,dd", [("flagship", 63, 27), ("reftest", 99, 99)])
def test_mlp(tag, dx, dd):
    g = load_golden(f"mlp_{tag}")
    cfg = O.NerfConfig()
    params = O.init_params(cfg, np.random.default_rng(int(g["init_seed"])), dx, dd)
    flat = O.flatten_params(params).numpy()
    assert flat.size == int(g["n_params"]) == O.param_count(cfg, dx, dd)
    import hashlib
    dig = np.frombuffer(hashlib.sha256(flat.tobytes()).digest()[:8], dtype=np.uint64)
    np.testing.assert_array_equal(dig, g["weights_digest"])       # same init draws as the reference run
    rgb, sigma = O.mlp_forward(params, T(g["x"]), T(g["dirs"]), cfg)
    assert rgb.shape == g["rgb"].shape and sigma.shape == g["sigma"].shape
    close(rgb, g["rgb"], atol=1e-6)
    close(sigma, g["sigma"], atol=1e-6)
    if tag == "flagship":
        assert flat.size == 595844


def _model_setup():
    g = load_golden("model")
    cfg = O.NerfConfig()
    rng = np.random.default_rng(int(g["init_seed"]))
    pc = O.init_params(cfg, rng)
    pf = O.init_params(cfg, rng)
    return g, cfg, pc, pf


def test_model_render():
    g, cfg, pc, pf = _model_setup()
    H, W = int(g["H"]), int(g["W"])
    o, d, t = O.generate_rays(g["pose"], H, W, float(g["focal"]), 2.0, 6.0, cfg.n_coarse, g["u_coarse"])
    close(o, g["o"], atol=0); close(d, g["d"], atol=1e-7); close(t, g["t"], atol=0)
    rays = (T(g["o"])[None], T(g["d"])[None], T(g["t"])[None])
    c, f = O.predict_and_render_images(pc, pf, cfg, rays, g["u_fine"], int(g["ray_chunks"]), True)
    for k, tol in (("image", 2e-6), ("depth", 1e-5), ("weights", 1e-6)):
        close(c[k], g[f"{k}_coarse"], atol=tol)
        close(f[k], g[f"{k}_fine"], atol=tol)


@pytest.fixture
def golden_threads():
    """model.npz was generated with 8 intra-op threads (make_golden.py).  The thread count sets the CPU summation
    order, and step 1's fine loss inherits it through Adam's sign(g) steps on ~zero gradients and the ill-conditioned
    fine pass (test_illconditioning_cpu.py): 1 / 16 threads move it by 3.7e-5 / 1.7e-5 relative, 8 threads reproduce
    the fixture to 1.3e-7.  The oracle runs with the fixture's thread count whatever the host's core count."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def test_model_train_two_steps(golden_threads):
    g, cfg, pc, pf = _model_setup()
    rays = (T(g["o"])[None], T(g["d"])[None], T(g["t"])[None])
    ac, af = O.AdamState(), O.AdamState()
    for step in range(2):
        out = O.train_step(pc, pf, ac, af, cfg, g["images"], rays, g["u_fine"], int(g["ray_chunks"]), True)
        assert out["coarse_loss"] == pytest.approx(float(g[f"s{step}_coarse_loss"]), rel=1e-5)
        assert out["fine_loss"] == pytest.approx(float(g[f"s{step}_fine_loss"]), rel=1e-5)
        assert out["coarse_psnr"] == pytest.approx(float(g[f"s{step}_coarse_psnr"]), abs=1e-4)
        assert out["fine_psnr"] == pytest.approx(float(g[f"s{step}_fine_psnr"]), abs=1e-4)
        for name, gr, pr in (("coarse", out["grad_coarse"], out["params_coarse"]),
                             ("fine", out["grad_fine"], out["params_fine"])):
            shapes = O.layer_shapes(cfg)
            off = 0
            k = 0
            gmax = float(gr.abs().max())
            for _, fi, fo in shapes:
                for n in (fi * fo, fo):
                    seg = gr[off:off + n].numpy()
                    head = g[f"s{step}_grad_{name}_head"][k]
                    m = min(n, 32)
                    np.testing.assert_allclose(seg[:m], head[:m], atol=2e-5 * gmax)
                    assert float(np.abs(seg).sum(dtype=np.float64)) == pytest.approx(
                        float(g[f"s{step}_grad_{name}_abssum"][k]), rel=2e-4, abs=1e-9)
                    off += n
                    k += 1
            k = 0
            for W_, b_ in pr:
                for arr in (W_, b_):
                    head = g[f"s{step}_param_{name}_head"][k]
                    m = min(arr.numel(), 32)
                    # Adam's first steps move every weight by ~lr regardless of |g|: sign(g) noise
                    # on ~zero gradients is excluded by the 2*lr tolerance
                    np.testing.assert_allclose(arr.reshape(-1)[:m].numpy(), head[:m], atol=2.1e-3)
                    k += 1
        pc, pf = out["params_coarse"], out["params_fine"]
