"""RaysGenerator (reference: keras_nerf/data/rays.py) on the GPU via libknerf."""
from __future__ import annotations

import itertools

import numpy as np
import torch

from .. import _lib

_seed_counter = _lib.seed_stream(0x5EED0000)


class RaysGenerator:
    """Same constructor and call signature as keras_nerf/data/rays.py:5-27,69-130.

    `__call__(camera_params)` -> (ray_origin[H,W,3], ray_direction[H,W,3], sample_points[H,W,N]) as CUDA
    tensors.  The reference draws fresh `tf.random.uniform` jitter on every call; here the draws come
    from the library's Philox stream (a new seed per call) unless `u` [H,W,N] is passed explicitly.

    `ndc=True` (forward-facing scenes, vanilla NeRF's `ndc_rays` with near plane 1): `knerf_generate_rays_ndc` writes
    the rays in normalized device coordinates, o = o_ndc, d = normalize(d_ndc), t = |d_ndc| * s with s stratified on
    [0, 1]; `near` and `far` are not used.
    """

    def __init__(self, focal_length: float, image_width: int, image_height: int, near: float, far: float,
                 n_sample: int, device=None, ndc: bool = False, **kwargs):
        self.focal_length = float(focal_length)
        self.image_width = int(image_width)
        self.image_height = int(image_height)
        self.near = float(near)
        self.far = float(far)
        self.n_sample = int(n_sample)
        self.device = torch.device(device) if device is not None else None
        self.ndc = bool(ndc)

    def __call__(self, camera_params, u=None, seed=None):
        device = self.device or _lib.default_device()
        if torch.is_tensor(camera_params):
            camera_params = camera_params.detach().cpu().numpy()
        c2w = np.ascontiguousarray(np.asarray(camera_params, dtype=np.float32).reshape(4, 4))
        H, W, N = self.image_height, self.image_width, self.n_sample
        with torch.cuda.device(device):
            o = torch.empty((H, W, 3), dtype=torch.float32, device=device)
            d = torch.empty((H, W, 3), dtype=torch.float32, device=device)
            t = torch.empty((H, W, N), dtype=torch.float32, device=device)
            if u is not None:
                u = _lib.dev(u, device).reshape(H, W, N)
            if seed is None:
                seed = next(_seed_counter)
            if self.ndc:
                _lib.call("knerf_generate_rays_ndc", c2w.ctypes.data, H, W, self.focal_length, N, _lib.ptr(u),
                          int(seed), _lib.ptr(o), _lib.ptr(d), _lib.ptr(t), _lib.stream())
            else:
                _lib.call("knerf_generate_rays", c2w.ctypes.data, H, W, self.focal_length, self.near, self.far, N,
                          _lib.ptr(u), int(seed), _lib.ptr(o), _lib.ptr(d), _lib.ptr(t), _lib.stream())
        return o, d, t


def generate_ray_batch(images, poses, focal, near, far, n_sample, perm_seed, epoch, first, n_rays, u=None, seed=None,
                       with_pixel=False, ndc=False):
    """`knerf_generate_ray_batch`: rays first .. first+n_rays-1 of epoch `epoch` of the permutation keyed by
    `perm_seed` over every pixel of the view cache `images` [n_img, H, W, C] (CUDA fp32, C >= 3) with poses
    [n_img, 4, 4].  Returns (target[n,3], o[n,3], d[n,3], t[n,N]) (+ pixel[n] int64, id (img*H + y)*W + x, when
    `with_pixel`).  The jitter comes from Philox(seed), a new seed per call unless given, or from `u` [n, N].
    `ndc=True`: `knerf_generate_ray_batch_ndc`, the rays of RaysGenerator(..., ndc=True); near and far are not used."""
    n_img, H, W, C = images.shape
    device = images.device
    N = int(n_sample)
    with torch.cuda.device(device):
        mk = lambda *s: torch.empty(s, dtype=torch.float32, device=device)  # noqa: E731
        target, o, d, t = mk(n_rays, 3), mk(n_rays, 3), mk(n_rays, 3), mk(n_rays, N)
        pixel = torch.empty(n_rays, dtype=torch.int64, device=device) if with_pixel else None
        if u is not None:
            u = _lib.dev(u, device).reshape(n_rays, N)
        if seed is None:
            seed = next(_seed_counter)
        head = (_lib.ptr(images), n_img, H, W, C, _lib.ptr(poses), float(focal))
        tail = (N, int(perm_seed) & 0xFFFFFFFFFFFFFFFF, int(epoch) & 0xFFFFFFFFFFFFFFFF, int(first), int(n_rays),
                _lib.ptr(u), int(seed), _lib.ptr(o), _lib.ptr(d), _lib.ptr(t), _lib.ptr(target),
                None if pixel is None else pixel.data_ptr(), _lib.stream())
        if ndc:
            _lib.call("knerf_generate_ray_batch_ndc", *head, *tail)
        else:
            _lib.call("knerf_generate_ray_batch", *head, float(near), float(far), *tail)
    return (target, o, d, t, pixel) if with_pixel else (target, o, d, t)
