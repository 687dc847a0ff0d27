"""GPU (-m gpu): mesh export -- the marching-tetrahedra kernel against its NumPy restatement (tests/mesh_oracle.py),
the density grid through the fused forward against the oracle MLP, and NeRF.extract_mesh / extract_mesh.py on a model
trained on the synthetic unit sphere."""
import ctypes as C

import numpy as np
import pytest
import torch

import mesh_oracle as M
import oracle as O

pytestmark = pytest.mark.gpu


def _kernel(field, iso, origin=(0, 0, 0), spacing=(1, 1, 1)):
    from keras_nerf_b200.utils.mesh import marching_tetrahedra
    v, n, f = marching_tetrahedra(torch.as_tensor(field, dtype=torch.float32).cuda(), iso, origin, spacing)
    return v.cpu().numpy(), n.cpu().numpy(), f.cpu().numpy()


def _cases():
    rng = np.random.default_rng(7)
    shape = (17, 23, 29)
    u = rng.random(shape, dtype=np.float32)
    eq = u.copy()
    eq[::3, ::2] = 0.5                                       # values exactly at iso (outside, t = 0 vertices)
    quant = (rng.integers(0, 4, shape) / 4.0).astype(np.float32)   # many equal neighbours and exact ties
    single = np.zeros(shape, np.float32)
    single[8, 11, 14] = 2.0
    faces = np.zeros(shape, np.float32)                      # inside points on every grid face and corner
    faces[0, :, 3:9] = faces[-1, 4:10, :] = faces[:, 0, -1] = faces[5:9, -1, :] = faces[0, 0, 0] = 1.0
    faces[:, 10:12, 0] = 1.0
    smooth = np.fromfunction(lambda i, j, k: np.sin(0.4 * i) * np.cos(0.3 * j) + 0.1 * k - 1.0, shape,
                             dtype=np.float32).astype(np.float32)
    return [("uniform", u, 0.5, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)),
            ("ties", eq, 0.5, (-1.0, 2.0, 0.5), (0.25, 0.5, 0.125)),
            ("quantised", quant, 0.5, (-1.5, -1.5, -1.5), (3 / 16, 3 / 22, 3 / 28)),
            ("single", single, 0.0, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)),
            ("faces", faces, 0.5, (0.0, 0.0, 0.0), (0.1, 0.2, 0.3)),
            ("smooth", smooth, 0.0, (-2.0, -3.0, -1.0), (0.2, 0.25, 0.1)),
            ("all_inside", np.ones(shape, np.float32), 0.5, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)),
            ("all_outside", np.full(shape, 0.5, np.float32), 0.5, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)),
            ("thin", rng.random((2, 3, 2), dtype=np.float32), 0.4, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0))]


@pytest.mark.parametrize("case", _cases(), ids=lambda c: c[0])
def test_kernel_matches_reference(case):
    """same vertex and triangle counts, the same order, the same index triples; positions and normals to 1e-6 of the
    grid's extent (the kernel rounds every fp32 operation like the reference: observed equal bits)"""
    _, f, iso, origin, spacing = case
    v, n, t = _kernel(f, iso, origin, spacing)
    rv, rn, rt = M.isosurface(f, iso, origin, spacing)
    assert v.shape == rv.shape and t.shape == rt.shape
    assert np.array_equal(t.astype(np.int64), rt)
    ext = max(1.0, float(np.abs(np.asarray(origin)).max() + np.max(np.asarray(spacing) * np.asarray(f.shape))))
    if len(v):
        assert np.abs(v - rv).max() <= 1e-6 * ext
        assert np.abs(n - rn).max() <= 1e-6
    if case[0] == "single":                                   # away from the faces: a closed surface
        assert M.edge_manifold(t) and M.euler_characteristic(len(v), t) == 2


def test_two_runs_identical_and_emit_respects_capacity():
    from keras_nerf_b200 import _lib
    rng = np.random.default_rng(3)
    f = torch.from_numpy(rng.random((33, 40, 27), dtype=np.float32)).cuda()
    a = _kernel(f, 0.5)
    b = _kernel(f, 0.5)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
    V, T = len(a[0]), len(a[2])
    L = _lib.load()
    nx, ny, nz = f.shape
    wsb = L.knerf_isosurface_workspace_bytes(nx, ny, nz)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    counts = torch.empty(2, dtype=torch.int64, device="cuda")
    _lib.call("knerf_isosurface_count", _lib.ptr(f), nx, ny, nz, 0.5, _lib.ptr(counts, torch.int64), ws.data_ptr(),
              wsb, _lib.stream())
    assert counts.tolist() == [V, T]
    G = 4096                                                  # guard band (floats / ints) either side of each output
    mv, mt = V // 3, T // 2
    vbuf = torch.full((3 * mv + 2 * G,), -7.0, device="cuda")
    nbuf = torch.full((3 * mv + 2 * G,), -7.0, device="cuda")
    tbuf = torch.full((3 * mt + 2 * G,), -7, dtype=torch.int32, device="cuda")
    org = (C.c_float * 3)(0, 0, 0)
    sp = (C.c_float * 3)(1, 1, 1)
    _lib.call("knerf_isosurface_emit", _lib.ptr(f), nx, ny, nz, 0.5, org, sp, vbuf[G:].data_ptr(),
              nbuf[G:].data_ptr(), tbuf[G:].data_ptr(), mv, mt, ws.data_ptr(), wsb, _lib.stream())
    vb, nb, tb = vbuf.cpu().numpy(), nbuf.cpu().numpy(), tbuf.cpu().numpy()
    for buf, m, ref in ((vb, mv, a[0]), (nb, mv, a[1]), (tb, mt, a[2])):
        assert (buf[:G] == -7).all() and (buf[G + 3 * m:] == -7).all()
        assert np.array_equal(buf[G:G + 3 * m].reshape(m, 3), ref[:m])
    # zero capacity: nothing written at all, null outputs accepted
    _lib.call("knerf_isosurface_emit", _lib.ptr(f), nx, ny, nz, 0.5, org, sp, None, None, None, 0, 0, ws.data_ptr(),
              wsb, _lib.stream())
    torch.cuda.synchronize()


def test_analytic_sphere_128():
    xyz, origin, spacing = M.grid(128, -1.3, 1.3)
    f = 1.0 - np.linalg.norm(xyz, axis=-1)
    v, n, t = _kernel(f, 0.0, origin, spacing)
    assert M.edge_manifold(t) and M.euler_characteristic(len(v), t) == 2
    vol = M.signed_volume(v, t)
    assert abs(vol / (4 * np.pi / 3) - 1) < 0.005, vol
    assert (np.einsum("ij,ij->i", M.face_normals(v, t), v[t].mean(1)) > 0).all()
    radial = v / np.linalg.norm(v, axis=1, keepdims=True)
    assert (np.einsum("ij,ij->i", n, radial) > 0.99).all()


# ---- density grid through the fused forward ---------------------------------------------------------------------------
def _model(precision, reproducible=False, seed=5):
    from keras_nerf_b200 import NeRF
    from keras_nerf_b200.model.nerf import mlp as mlp_mod
    mlp_mod.set_seed(seed)
    m = NeRF(precision=precision, reproducible=reproducible)
    m.compile(optimizer="adam", loss="mse", batch_size=1, image_height=1, image_width=1, ray_chunks=1,
              is_training=False)
    return m


def test_density_grid_fp32_matches_oracle_mlp():
    m = _model("fp32")
    res, bound = (9, 12, 14), ((-1.5, -1.0, -0.5), (1.5, 1.25, 1.0))
    grid = m.density_grid(res, bound, network="coarse").cpu()
    n, lo, h = m._grid_frame(res, bound)
    axes = [torch.from_numpy(lo[a:a + 1]) + torch.arange(int(n[a]), dtype=torch.float32) * torch.from_numpy(h[a:a + 1])
            for a in range(3)]
    pts = torch.stack(torch.meshgrid(*axes, indexing="ij"), -1).reshape(-1, 3)
    cfg = O.NerfConfig()
    params = O.unflatten_params(m.coarse.params.cpu(), cfg)
    xyz = O.positional_encoding(pts, cfg.pos_emb_xyz)
    dirs = O.positional_encoding(torch.tensor([[0.0, 0.0, 1.0]]).expand(len(pts), 3), cfg.pos_emb_dir)
    _, sigma = O.mlp_forward(params, xyz, dirs, cfg)
    ref = sigma.reshape(grid.shape)
    assert float(ref.max()) > 0 and float((ref > 0).float().mean()) > 0.05     # a field worth comparing
    assert float((grid - ref).abs().max()) <= 1e-5 * float(ref.max())


@pytest.mark.parametrize("precision,reproducible", [("fp32", False), ("bf16", True)])
def test_density_grid_slab_size_does_not_change_a_bit(precision, reproducible):
    m = _model(precision, reproducible)
    a = m.density_grid(24, 1.2, samples_per_call=24 * 7)        # 7 columns per call, ragged last call
    b = m.density_grid(24, 1.2, samples_per_call=24 * 24 * 5)
    c = m.density_grid(24, 1.2)                                 # everything in one call
    assert torch.equal(a, b) and torch.equal(a, c)


def test_density_grid_bf16_within_tolerance_of_fp32():
    """bf16 operands through eight layers: the sigma pre-activation moves by ~0.5 % (DESIGN.md section 2); bar 1 % of
    the grid's largest sigma"""
    m32, m16 = _model("fp32"), _model("bf16")
    g32, g16 = m32.density_grid(32, 1.5), m16.density_grid(32, 1.5)
    err = float((g16 - g32).abs().max()) / float(g32.max())
    print(f"bf16 vs fp32 density grid: max |diff| / max sigma = {err:.2e}")
    assert err <= 1e-2


# ---- end to end on the synthetic unit sphere -----------------------------------------------------------------------
@pytest.fixture(scope="module")
def trained_sphere(tmp_path_factory):
    """the bf16 flagship model after 600 steps on whole 128 x 128 views of the analytic unit sphere (white background)"""
    from keras_nerf_b200 import NeRF
    from keras_nerf_b200.data.synthetic import SyntheticScene
    from keras_nerf_b200.model.nerf import mlp as mlp_mod
    dev = torch.device("cuda")
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
    path = str(tmp_path_factory.mktemp("sphere") / "sphere")
    m.save_model(path)
    return m, path


# Fixed once from the trained grid of the fixture (128^3 over [-1.5, 1.5]^3): after 600 steps sigma is still small --
# 10th / 50th / 90th percentiles 2.2 / 2.8 / 3.7 for |x| < 0.8, exactly 0 for |x| > 1.05 -- so the default threshold of
# a converged model (50) lies above the whole field and gives an empty mesh.  1.0 sits between the empty outside and
# the interior's 10th percentile.  Measured median ||v| - 1| by threshold: 0.25: 0.014, 0.5: 0.012, 1.0: 0.0088,
# 1.5: 0.0081; from 2.0 on (0.074) the level set also wraps low-density pockets inside the ball.
SPHERE_THRESHOLD = 1.0


def test_trained_sphere_mesh(trained_sphere):
    m, _ = trained_sphere
    mesh = m.extract_mesh(resolution=128, threshold=SPHERE_THRESHOLD)
    v, f = mesh["vertices"].cpu().numpy(), mesh["faces"].cpu().numpy()
    assert len(f) > 0 and M.edge_manifold(f)
    err = float(np.median(np.abs(np.linalg.norm(v, axis=1) - 1)))
    print(f"trained sphere at threshold {SPHERE_THRESHOLD}: median ||v| - 1| = {err:.4f}, V={len(v)}, T={len(f)}, "
          f"seconds {mesh['seconds']}")
    assert err <= 0.03
    c = mesh["colors"]
    assert c.shape == (len(v), 3) and float(c.min()) >= 0 and float(c.max()) <= 1


def test_extract_mesh_script_writes_a_ply(trained_sphere, tmp_path):
    import extract_mesh
    from keras_nerf_b200.utils.mesh import read_ply
    _, path = trained_sphere
    out = extract_mesh.main(["--model_dirs", path, "--resolution", "64", "--threshold", str(SPHERE_THRESHOLD),
                             "--output_dir", str(tmp_path / "out")])
    assert out.endswith("sphere.ply")
    mesh = read_ply(out)
    assert len(mesh["faces"]) > 0 and mesh["colors"].dtype == np.uint8 and mesh["normals"].shape == mesh["vertices"].shape
    assert M.edge_manifold(mesh["faces"].astype(np.int64))
    with pytest.raises(FileNotFoundError):
        extract_mesh.main(["--model_dirs", str(tmp_path / "empty")])
