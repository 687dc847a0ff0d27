"""CPU: the LLFF loader's pose arithmetic (keras_nerf_b200.data.llff) against the float64 restatement of vanilla NeRF's
load_llff.py in tests/llff_oracle.py, write_llff_like round trips, the NDC refusal, and the argument checks of the two
NDC entry points (no device needed)."""
import os

import numpy as np
import pytest

import llff_oracle as LO
from keras_nerf_b200.data import llff as L


def _rot(axis, deg):
    a = np.radians(deg)
    k = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K


def _random_rig(seed, n=None):
    """poses_bounds [n, 17] of a forward-facing rig in LLFF's axes under a random global rotation and offset"""
    rng = np.random.default_rng(seed)
    n = n or int(rng.integers(8, 30))
    g = _rot(rng.normal(size=3), rng.uniform(0, 180))
    off = rng.normal(size=3)      # the loader works in fp32, as vanilla: recentring cancels |off| * 6e-8 of rounding
    rows = []
    for _ in range(n):
        r = g @ _rot(rng.normal(size=3), rng.uniform(0, 6))
        c2w = np.concatenate([r, (g @ np.append(rng.normal(size=2) * 0.4, rng.normal() * 0.05) + off)[:, None]], 1)
        m = np.stack([-c2w[:, 1], c2w[:, 0], c2w[:, 2], c2w[:, 3], [378.0, 504.0, 407.5]], 1)
        rows.append(np.concatenate([m.reshape(-1), [rng.uniform(1.0, 3.0), rng.uniform(20.0, 100.0)]]))
    return np.stack(rows).astype(np.float32)


def _close(a, b, tol=1e-6):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape
    err = float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b))))
    assert err <= tol, err


@pytest.mark.parametrize("seed", range(5))
def test_pose_functions_match_vanilla(seed):
    pb = _random_rig(seed)
    ref = LO.load_poses(pb)
    raw, bds = L.parse_poses_bounds(pb)
    swapped = L.llff_to_opengl(raw)
    _close(swapped, ref["swapped"])
    scaled, bds, sc = L.rescale(swapped, bds)
    _close(scaled, ref["scaled"])
    _close(bds, ref["bds"])
    rec = L.recenter_poses(scaled)
    _close(rec, ref["recentred"])
    _close(L.spiral_poses(rec, bds)[:, :, :4], ref["spiral"])
    near, far = L.near_far(bds, ndc=False)
    _close([near, far], [ref["near"], ref["far"]])
    assert L.near_far(bds, ndc=True) == (0.0, 1.0)
    for hold in (8, 3, 1, 0):
        got = L.split_views(rec, hold)
        want = LO.split(ref["recentred"], hold)
        assert [[int(i) for i in x] for x in got] == list(want)
    assert len(L.split_views(rec, 0)[2]) == 1          # no llffhold: vanilla holds out the most central view


def test_recentred_average_pose_is_identity():
    for seed in range(3):
        raw, bds = L.parse_poses_bounds(_random_rig(seed + 10))
        rec = L.recenter_poses(L.rescale(L.llff_to_opengl(raw), bds)[0])
        avg = L.poses_avg(rec)
        np.testing.assert_allclose(avg[:3, :4], np.eye(3, 4), atol=1e-6)


def test_write_llff_like_round_trip(tmp_path):
    from PIL import Image

    from keras_nerf_b200.data.synthetic import llff_like_poses, write_llff_like
    d = write_llff_like(str(tmp_path / "s"), H=24, W=32, n_views=6, factors=(2,), seed=3)
    pb = np.load(os.path.join(d, "poses_bounds.npy"))
    assert pb.shape == (6, 17) and pb.dtype == np.float32
    raw, bds = L.parse_poses_bounds(pb)
    np.testing.assert_allclose(L.llff_to_opengl(raw)[:, :, :4], llff_like_poses(6, seed=3).numpy(), atol=1e-6)
    np.testing.assert_allclose(raw[:, :, 4], np.tile([24.0, 32.0, 0.9 * 32], (6, 1)), atol=1e-5)
    assert (bds[:, 0] > 1.5).all() and (bds[:, 1] / bds[:, 0] > 20).all()      # the depth range NDC is for
    assert len(os.listdir(os.path.join(d, "images"))) == len(os.listdir(os.path.join(d, "images_2"))) == 6
    with Image.open(os.path.join(d, "images", "view_000.png")) as im:
        assert im.size == (32, 24)
    loader = L.LLFFDatasetLoader(d, factor=2, llffhold=4)
    assert (loader.H, loader.W, loader.resize) == (12, 16, False) and loader.focal == pytest.approx(0.9 * 32 / 2)
    assert list(loader.i_test) == [0, 4] and list(loader.i_train) == [1, 2, 3, 5]
    assert loader.render_path().shape == (120, 4, 4)
    loader = L.LLFFDatasetLoader(d, factor=4)
    assert (loader.H, loader.W, loader.resize) == (6, 8, True) and loader.focal == pytest.approx(0.9 * 32 / 4)


def test_ndc_refusal(tmp_path):
    from keras_nerf_b200.data.synthetic import write_llff_like
    d = write_llff_like(str(tmp_path / "s"), H=12, W=16, n_views=5)
    L.LLFFDatasetLoader(d, factor=1)
    pb = np.load(os.path.join(d, "poses_bounds.npy"))
    m = pb[2, :15].reshape(3, 5).astype(np.float64)
    m[:, :3] = _rot([0, 1, 0], 100) @ m[:, :3]             # one camera turned sideways: its frame reaches w_z >= 0
    pb[2, :15] = m.reshape(-1)
    np.save(os.path.join(d, "poses_bounds.npy"), pb)
    with pytest.raises(ValueError, match="w_z >= 0"):
        L.LLFFDatasetLoader(d, factor=1)
    loader = L.LLFFDatasetLoader(d, factor=1, ndc=False)
    assert loader.near < loader.far and loader.near == pytest.approx(0.9 * loader.bds.min())
    # the corners bound the frame: a pose turned just past the point where its x = 0 column looks along the image
    # plane is refused, one turned just short of it is not
    H, W, f = 10, 20, 10.0
    pose = np.eye(4, dtype=np.float32)
    L.check_ndc_views(pose[None], H, W, f)
    edge = np.degrees(np.arctan(f / (W * 0.5)))
    tilt = np.eye(4)
    tilt[:3, :3] = _rot([0, 1, 0], edge - 0.01)
    L.check_ndc_views(tilt[None], H, W, f)
    tilt[:3, :3] = _rot([0, 1, 0], edge + 0.01)
    with pytest.raises(ValueError):
        L.check_ndc_views(tilt[None], H, W, f)


def test_image_count_must_match_poses(tmp_path):
    from keras_nerf_b200.data.synthetic import write_llff_like
    d = write_llff_like(str(tmp_path / "s"), H=12, W=16, n_views=4)
    os.remove(os.path.join(d, "images", "view_001.png"))
    with pytest.raises(ValueError, match="3 images for 4 poses"):
        L.LLFFDatasetLoader(d, factor=1)


def test_ray_chunks_stay_near_the_requested_size():
    # (render chunk, training chunk): the LLFF view sizes at factors 8, 16 and 4 with vanilla's N_rand values
    assert L.ray_chunks_for(378 * 504, 4096, 1024) == (1008, 1024)
    assert L.ray_chunks_for(378 * 504, 1024, 1024) == (1008, 1024)
    assert L.ray_chunks_for(189 * 252, 4096, 1024) == (972, 1024)
    assert L.ray_chunks_for(756 * 1008, 4096, 1024) == (1008, 1024)
    assert L.ray_chunks_for(378 * 504, 4096, 4096) == (3969, 4096)
    assert L.ray_chunks_for(378 * 504, 0, 1024) == (1008, 1008)     # whole views: one chunk for both
    assert L.ray_chunks_for(45 * 63, 2048, 1024) == (945, 1024)
    assert L.ray_chunks_for(378 * 504, 1000, 1024) == (1008, 1000)
    assert L.ray_chunks_for(100, 0, 4096) == (100, 100)
    for hw in (378 * 504, 189 * 252, 756 * 1008, 45 * 63):
        for n in (1024, 2048, 4096, 32768):
            r, t = L.ray_chunks_for(hw, n, 1024)
            assert hw % r == 0 and n % t == 0 and r >= 900 and t == 1024


def test_spiral_is_checked_where_it_is_rendered(tmp_path):
    from keras_nerf_b200.data.synthetic import write_llff_like
    d = write_llff_like(str(tmp_path / "s"), H=12, W=16, n_views=5)
    loader = L.LLFFDatasetLoader(d, factor=1)
    loader.render_poses[3, :3, :3] = _rot([0, 1, 0], 100).astype(np.float32)   # a spiral pose that looks sideways
    with pytest.raises(ValueError, match="spiral poses \\[3\\]"):
        loader.render_path()
    loader.ndc = False
    assert loader.render_path().shape == (120, 4, 4)               # world-space rays have no such restriction


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from keras_nerf_b200 import _lib
    return _lib


def test_ndc_entry_points_validate_arguments(lib):
    Lb = lib.load()
    assert Lb.knerf_generate_rays_ndc(None, 4, 4, 1.0, 8, None, 0, None, None, None, None) == -1
    assert b"null" in Lb.knerf_last_error() and b"knerf_generate_rays_ndc" in Lb.knerf_last_error()
    assert Lb.knerf_generate_ray_batch_ndc(None, 1, 4, 4, 4, None, 1.0, 8, 0, 0, 0, 16, None, 0, None, None, None,
                                           None, None, None) == -1
    assert b"null" in Lb.knerf_last_error() and b"knerf_generate_ray_batch_ndc" in Lb.knerf_last_error()
    c2w = np.eye(4, dtype=np.float32)
    dummy = 16   # never dereferenced: the shape checks fail first
    assert Lb.knerf_generate_rays_ndc(c2w.ctypes.data, 0, 4, 1.0, 8, None, 0, dummy, dummy, dummy, None) == -1
    assert b"bad shape" in Lb.knerf_last_error()
    assert Lb.knerf_generate_ray_batch_ndc(dummy, 1, 4, 4, 4, dummy, 1.0, 8, 0, 0, 10, 16, None, 0, dummy, dummy,
                                           dummy, dummy, None, None) == -1
    assert b"outside" in Lb.knerf_last_error()
