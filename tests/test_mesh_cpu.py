"""CPU (-m "not gpu"): the isosurface rules on analytic fields through their NumPy restatement (tests/mesh_oracle.py,
which the GPU tests hold the kernel to), PLY files, and the host-side checks of the isosurface entry points."""
import ctypes as C

import numpy as np
import pytest

import mesh_oracle as M


def _sphere(n=64, lo=-1.5, hi=1.5):
    xyz, origin, spacing = M.grid(n, lo, hi)
    return 1.0 - np.linalg.norm(xyz, axis=-1), origin, spacing


def test_sphere_is_closed_oriented_and_has_the_right_volume():
    f, origin, spacing = _sphere()
    v, n, t = M.isosurface(f, 0.0, origin, spacing)
    assert len(v) > 1000 and t.min() >= 0 and t.max() < len(v)
    assert M.edge_manifold(t)                               # every edge in two faces, once in each direction
    assert M.euler_characteristic(len(v), t) == 2
    vol = M.signed_volume(v, t)
    assert vol > 0 and abs(vol / (4 * np.pi / 3) - 1) < 0.01
    fn = M.face_normals(v, t)
    assert (np.einsum("ij,ij->i", fn, v[t].mean(1)) > 0).all()     # every face outward
    assert np.allclose(np.linalg.norm(n, axis=1), 1, atol=1e-5)
    assert (np.einsum("ij,ij->i", n, v / np.linalg.norm(v, axis=1, keepdims=True)) > 0.99).all()


def test_torus_genus_one():
    xyz, origin, spacing = M.grid(64, -1.5, 1.5)
    R, r = 0.8, 0.3
    f = r - np.sqrt((np.sqrt(xyz[..., 0] ** 2 + xyz[..., 1] ** 2) - R) ** 2 + xyz[..., 2] ** 2)
    v, _, t = M.isosurface(f, 0.0, origin, spacing)
    assert M.edge_manifold(t) and M.euler_characteristic(len(v), t) == 0
    assert M.signed_volume(v, t) > 0


def test_rules_on_small_cases():
    # one inside point in the middle of a 3^3 grid: the 14 edges through it carry a vertex (6 axis, 6 face-diagonal,
    # 2 body-diagonal neighbours of the Kuhn lattice), a closed octahedron-like surface around it
    f = np.zeros((3, 3, 3), np.float32)
    f[1, 1, 1] = 1.0
    v, n, t = M.isosurface(f, 0.5)
    assert len(v) == 14 and M.edge_manifold(t) and M.euler_characteristic(len(v), t) == 2
    assert np.allclose(np.abs(v - 1).max(1), 0.5)           # every vertex halfway along its edge
    assert M.signed_volume(v, t) > 0
    # f == iso is outside; t = 0 then puts the vertex on the point itself
    f[0, 1, 1] = 0.5
    v2, _, _ = M.isosurface(f, 0.5)
    assert ((v2 == [0, 1, 1]).all(1)).sum() >= 1
    # constant fields: nothing
    for c in (0.0, 1.0):
        v3, n3, t3 = M.isosurface(np.full((4, 5, 6), c, np.float32), 0.5)
        assert len(v3) == len(t3) == 0 and n3.shape == (0, 3)
    # the orientation rule never needs a tie-break: every table entry has a nonzero dot (asserted while building)
    assert sum(len(M.TABLE[tet][p]) for tet in range(6) for p in range(16)) == 6 * (8 * 1 + 6 * 2)


def test_ply_round_trip(tmp_path):
    from keras_nerf_b200.utils.mesh import read_ply, write_ply
    rng = np.random.default_rng(0)
    V, T = 37, 51
    v = rng.standard_normal((V, 3)).astype(np.float32)
    n = rng.standard_normal((V, 3)).astype(np.float32)
    c = rng.random((V, 3)).astype(np.float32)
    f = rng.integers(0, V, (T, 3)).astype(np.int32)
    p = write_ply(str(tmp_path / "m.ply"), v, f, normals=n, colors=c)
    raw = open(p, "rb").read()
    end = raw.index(b"end_header\n") + len(b"end_header\n")
    header = raw[:end].decode("ascii")
    assert header.startswith("ply\nformat binary_little_endian 1.0\nelement vertex 37\n")
    assert "property uchar red" in header and "element face 51\nproperty list uchar int vertex_indices\n" in header
    assert len(raw) - end == V * (12 + 12 + 3) + T * (1 + 12)     # payload byte count
    m = read_ply(p)
    assert np.array_equal(m["vertices"], v) and np.array_equal(m["normals"], n) and np.array_equal(m["faces"], f)
    assert np.array_equal(m["colors"], np.rint(c * 255).astype(np.uint8))
    # geometry only
    p2 = write_ply(str(tmp_path / "sub" / "g.ply"), v, f)
    m2 = read_ply(p2)
    assert m2["normals"] is None and m2["colors"] is None and np.array_equal(m2["vertices"], v)
    assert len(open(p2, "rb").read()) - open(p2, "rb").read().index(b"end_header\n") - 11 == V * 12 + T * 13
    # an empty mesh is a valid file
    m3 = read_ply(write_ply(str(tmp_path / "e.ply"), np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32)))
    assert m3["vertices"].shape == (0, 3) and m3["faces"].shape == (0, 3)


def test_isosurface_entry_points_validate_arguments():
    import __graft_entry__ as g
    g.build()
    from keras_nerf_b200 import _lib
    L = _lib.load()
    n = 17 * 23 * 29
    ws = L.knerf_isosurface_workspace_bytes(17, 23, 29)
    assert ws >= 5 * n and ws < 5 * n + 4096                 # mask + two uint16 prefixes per point, per-tile offsets
    assert L.knerf_isosurface_workspace_bytes(1, 23, 29) < 0 and b"need >= 2" in L.knerf_last_error()
    assert L.knerf_isosurface_workspace_bytes(512, 512, 512) < 1 << 30
    # argument validation happens before any CUDA call: safe without a GPU
    assert L.knerf_isosurface_count(None, 17, 23, 29, 0.5, None, None, 0, None) == -1
    assert L.knerf_isosurface_count(C.c_void_p(256), 17, 23, 29, 0.5, C.c_void_p(256), None, 0, None) == -4
    o3 = (C.c_float * 3)(0, 0, 0)
    assert L.knerf_isosurface_emit(C.c_void_p(256), 17, 23, 29, 0.5, o3, o3, None, None, None, 10, 0, None, 0,
                                   None) == -1
    assert L.knerf_isosurface_emit(C.c_void_p(256), 17, 23, 29, 0.5, o3, o3, C.c_void_p(256), None, C.c_void_p(256),
                                   1 << 31, 1, C.c_void_p(256), ws, None) == -3
    assert b"int32" in L.knerf_last_error()


def test_grid_frame_and_arguments():
    from keras_nerf_b200 import NeRF
    n, lo, h = NeRF._grid_frame(5, 1.0)
    assert n.tolist() == [5, 5, 5] and lo.tolist() == [-1, -1, -1] and h.tolist() == [0.5, 0.5, 0.5]
    n, lo, h = NeRF._grid_frame((3, 5, 9), ((0, -1, -2), (1, 1, 2)))
    assert n.tolist() == [3, 5, 9] and lo.tolist() == [0, -1, -2] and h.tolist() == [0.5, 0.5, 0.5]
    with pytest.raises(ValueError):
        NeRF._grid_frame(1, 1.0)
    with pytest.raises(ValueError):
        NeRF._grid_frame(4, ((0, 0, 0), (1, 0, 1)))
