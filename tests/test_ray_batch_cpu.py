"""CPU (-m "not gpu"): the epoch permutation of knerf_generate_ray_batch (NumPy restatement), the call's argument
checks, and the batch arithmetic of RayBatchDataset."""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy import stats

from ray_batch_oracle import half_bits, permute


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from keras_nerf_b200 import _lib
    return _lib


@pytest.mark.parametrize("P", [1, 2, 3, 5, 2 ** 10 - 1, 2 ** 10, 2 ** 10 + 1, 2 ** 13 - 1, 2 ** 13 + 1, 999983])
def test_permutation_is_a_bijection(P):
    for epoch in (0, 1, 7):
        pi = permute(np.arange(P), P, perm_seed=1234, epoch=epoch)
        assert pi.max() < P
        assert np.array_equal(np.sort(pi), np.arange(P, dtype=np.uint64)), (P, epoch)


def test_bit_width_is_the_smallest_even_one():
    assert [2 * half_bits(P) for P in (1, 2, 4, 5, 16, 17, 2 ** 20, 2 ** 20 + 1)] == [2, 2, 2, 4, 4, 6, 20, 22]


def test_epochs_and_seeds_give_different_orders():
    P = 100_003
    orders = [permute(np.arange(P), P, perm_seed=s, epoch=e) for s, e in ((5, 0), (5, 1), (5, 2), (6, 0))]
    for i in range(len(orders)):
        for j in range(i + 1, len(orders)):
            # two independent orders agree in about one position
            assert (orders[i] == orders[j]).sum() < 20, (i, j)


def test_rays_per_view_pass_chi_square():
    n_img, H, W, N = 100, 40, 40, 4096
    P = n_img * H * W
    for epoch in (0, 1, 2):
        for first in (0, 50 * N, P - N):
            pix = permute(np.arange(first, first + N), P, perm_seed=42, epoch=epoch)
            counts = np.bincount((pix // (H * W)).astype(np.int64), minlength=n_img)
            p = stats.chisquare(counts).pvalue
            assert p > 1e-3, (epoch, first, p)


def test_generate_ray_batch_rejects_bad_arguments(lib):
    """argument checks come before any device work, so they run here without a GPU"""
    L = lib.load()
    buf = (C.c_float * 64)()
    p = C.cast(buf, C.c_void_p)
    pix = C.cast((C.c_int64 * 8)(), C.c_void_p)
    good = dict(images=p, n_img=2, H=4, W=4, C=4, c2w=p, focal=3.0, near=2.0, far=6.0, N=8, perm_seed=1, epoch=0,
                first=0, R=8, u=None, seed=0, o=p, d=p, t=p, target=p, pixel=pix)

    def call(**kw):
        a = {**good, **kw}
        return L.knerf_generate_ray_batch(*a.values(), None)

    bad = [dict(images=None), dict(c2w=None), dict(o=None), dict(d=None), dict(t=None), dict(target=None),
           dict(n_img=0), dict(H=0), dict(W=-1), dict(N=0), dict(C=2), dict(first=-1), dict(first=25, R=8),
           dict(first=0, R=33), dict(R=-1)]
    for kw in bad:
        assert call(**kw) == -1, kw
    assert b"null" in (call(t=None), L.knerf_last_error())[1]
    assert b"C=2" in (call(C=2), L.knerf_last_error())[1]
    assert b"outside [0, 32)" in (call(first=25, R=8), L.knerf_last_error())[1]


def _dataset(n_img=3, H=5, W=7, N=4, rank=0, world=1, **kw):
    from keras_nerf_b200.data.loader import RayBatchDataset
    return RayBatchDataset(torch.zeros(n_img, H, W, 4), torch.eye(4).expand(n_img, 4, 4), 1.0, 2.0, 6.0, 8, N,
                           rank=rank, world=world, perm_seed=9, **kw)


def test_ray_batch_dataset_arithmetic():
    P = 3 * 5 * 7
    assert len(_dataset(N=4)) == P // 4 == 26
    assert len(_dataset(N=4, world=3)) == P // 12 == 8
    assert len(_dataset(N=105)) == 1 and len(_dataset(N=106)) == 0
    assert len(_dataset(N=4).take(5)) == 5 and len(_dataset(N=4).take(100)) == 26
    # rank windows: disjoint, and step s of all ranks together is the world=1 batch of N*world rays at step s
    world, N = 3, 4
    covered = []
    for r in range(world):
        ds = _dataset(N=N, rank=r, world=world)
        covered += [range(ds.window(s), ds.window(s) + N) for s in range(len(ds))]
    flat = sorted(i for w in covered for i in w)
    assert flat == list(range(len(_dataset(N=N, world=world)) * world * N))
    single = _dataset(N=N * world)
    for s in range(len(single)):
        assert set(range(single.window(s), single.window(s) + N * world)) == \
            {i for r in range(world) for i in range(_dataset(N=N, rank=r, world=world).window(s),
                                                     _dataset(N=N, rank=r, world=world).window(s) + N)}
    with pytest.raises(ValueError):
        _dataset(rank=2, world=2)


def test_ray_batch_dataset_epochs_and_resume():
    ds = _dataset()
    assert ds.epoch == 0
    iter(ds)
    iter(ds)
    assert ds.epoch == 2                          # one new epoch key per pass
    ds.epoch = 5                                  # a run resumed after epoch 4 continues with epoch 5
    iter(ds)
    assert ds.epoch == 6
    t = ds.take(2)
    assert t.epoch == 6 and t.images is ds.images and t.perm_seed == ds.perm_seed


def test_permutation_key_ignores_rank(monkeypatch):
    from keras_nerf_b200.data.loader import permutation_seed
    torch.manual_seed(42)
    monkeypatch.setenv("RANK", "0")
    a = permutation_seed()
    monkeypatch.setenv("RANK", "3")
    assert permutation_seed() == a
    torch.manual_seed(43)
    assert permutation_seed() != a
