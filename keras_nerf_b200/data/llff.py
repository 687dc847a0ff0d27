"""LLFF datasets (forward-facing captures: COLMAP + LLFF's imgs2poses.py -> `poses_bounds.npy` + `images/`), vanilla
NeRF's `--dataset_type llff`.

The pose arithmetic is vanilla NeRF's load_llff.py and run_nerf.py restated in NumPy fp32 as pure functions (no GPU):
parse `poses_bounds.npy`, swap the axes from [down, right, back] to [right, up, back], rescale translations and bounds
by 1 / (0.75 * min bound), recentre on the average pose, hold out every `llffhold`-th view, and build the spiral render
path.  `LLFFDatasetLoader` does all of that in its constructor; `load_dataset` decodes and prepares the images on the
GPU and returns the same [train, val, test] as `DatasetLoader`.  With `ndc=True` (the default, as in vanilla) the rays
are generated in normalized device coordinates (`RaysGenerator(..., ndc=True)`).

Not covered: `spherify` (360-degree captures), `lindisp`, principal points and lens distortion."""
from __future__ import annotations

import logging
import os

import numpy as np
import torch

from .image import prepare_image
from .loader import Dataset, RayBatchDataset
from .rays import RaysGenerator

IMAGE_EXTENSIONS = (".png", ".jpg", ".JPG")
BD_FACTOR = 0.75


def parse_poses_bounds(arr) -> tuple:
    """poses_bounds.npy [N, 17] -> (poses [N, 3, 5] in LLFF's own axes [down, right, back, t, hwf], bounds [N, 2])"""
    arr = np.asarray(arr, dtype=np.float32)
    if arr.ndim != 2 or arr.shape[1] != 17:
        raise ValueError(f"poses_bounds.npy must be [N, 17], got {arr.shape}")
    return arr[:, :15].reshape(-1, 3, 5).copy(), arr[:, 15:17].copy()


def llff_to_opengl(poses) -> np.ndarray:
    """load_llff.py: columns [down, right, back, t, hwf] -> [right, up, back, t, hwf]"""
    p = np.asarray(poses, dtype=np.float32)
    return np.concatenate([p[:, :, 1:2], -p[:, :, 0:1], p[:, :, 2:]], 2)


def rescale(poses, bds, bd_factor: float = BD_FACTOR) -> tuple:
    """load_llff.py: translations and bounds times sc = 1 / (min bound * bd_factor) -> (poses, bds, sc)"""
    poses = np.array(poses, dtype=np.float32)
    bds = np.array(bds, dtype=np.float32)
    sc = np.float32(1.0 / (float(bds.min()) * bd_factor))
    poses[:, :3, 3] *= sc
    bds *= sc
    return poses, bds, sc


def normalize(x) -> np.ndarray:
    return x / np.linalg.norm(x)


def viewmatrix(z, up, pos) -> np.ndarray:
    """[3, 4] camera-to-world with back axis z, up-ish `up`, centre pos"""
    vec2 = normalize(z)
    vec0 = normalize(np.cross(up, vec2))
    vec1 = normalize(np.cross(vec2, vec0))
    return np.stack([vec0, vec1, vec2, pos], 1)


def poses_avg(poses) -> np.ndarray:
    """[3, 5]: mean centre, normalised summed back axis, summed up axis; hwf of the first view"""
    hwf = poses[0, :3, -1:]
    center = poses[:, :3, 3].mean(0)
    vec2 = normalize(poses[:, :3, 2].sum(0))
    up = poses[:, :3, 1].sum(0)
    return np.concatenate([viewmatrix(vec2, up, center), hwf], 1)


def recenter_poses(poses) -> np.ndarray:
    """load_llff.py: every pose premultiplied by the inverse of the average pose (hwf column kept)"""
    out = np.array(poses, dtype=np.float32)
    bottom = np.array([[0, 0, 0, 1.0]])                  # float64, as in load_llff.py: the product is taken in float64
    c2w = np.concatenate([poses_avg(out)[:3, :4], bottom], 0)
    full = np.concatenate([out[:, :3, :4], np.tile(bottom[None], (out.shape[0], 1, 1))], 1)
    out[:, :3, :4] = (np.linalg.inv(c2w) @ full)[:, :3, :4]
    return out


def closest_to_average(poses) -> int:
    """load_llff.py's i_test: the view whose centre is closest to the average pose's"""
    center = poses_avg(poses)[:3, 3]
    return int(np.argmin(np.sum(np.square(center - poses[:, :3, 3]), -1)))


def split_views(poses, llffhold: int) -> tuple:
    """run_nerf.py: test = val = every llffhold-th view, train = the rest -> (i_train, i_val, i_test).  With
    llffhold <= 0, test = val = the one view closest to the average pose (`closest_to_average`), as in vanilla."""
    n = len(poses)
    i_test = np.arange(n)[::llffhold] if llffhold > 0 else np.array([closest_to_average(poses)], np.int64)
    i_train = np.array([i for i in range(n) if i not in set(i_test.tolist())], dtype=np.int64)
    return i_train, i_test.copy(), i_test


def near_far(bds, ndc: bool) -> tuple:
    """run_nerf.py: (0, 1) in NDC (the depths then run over [0, |d_ndc|]), else (0.9 * min bound, max bound)"""
    if ndc:
        return 0.0, 1.0
    return float(np.float32(bds.min()) * np.float32(0.9)), float(np.float32(bds.max()) * np.float32(1.0))


def render_path_spiral(c2w, up, rads, focal, zrate, rots, n) -> np.ndarray:
    """load_llff.py: n poses [n, 3, 5] on a spiral of radii `rads` around c2w, looking at depth `focal`"""
    rads = np.array(list(rads) + [1.0])
    hwf = c2w[:, 4:5]
    out = []
    for theta in np.linspace(0.0, 2.0 * np.pi * rots, n + 1)[:-1]:
        c = np.dot(c2w[:3, :4], np.array([np.cos(theta), -np.sin(theta), -np.sin(theta * zrate), 1.0]) * rads)
        z = normalize(c - np.dot(c2w[:3, :4], np.array([0, 0, -focal, 1.0])))
        out.append(np.concatenate([viewmatrix(z, up, c), hwf], 1))
    return np.array(out).astype(np.float32)


def spiral_poses(poses, bds, n_views: int = 120, n_rots: int = 2, zrate: float = 0.5) -> np.ndarray:
    """load_llff.py (no spherify, no path_zflat): the render path [n_views, 3, 5] of the recentred, rescaled poses;
    focus depth 1 / ((1 - 0.75) / close + 0.75 / inf) with close = 0.9 * min bound, inf = 5 * max bound, radii the
    90th percentile of |translation|.  Computed in float64 (returned as fp32): the path is a smooth function of the
    poses, and fp32 intermediates would add ~1e-6 of noise to it."""
    poses, bds = np.asarray(poses, np.float64), np.asarray(bds, np.float64)
    c2w = poses_avg(poses)
    up = normalize(poses[:, :3, 1].sum(0))
    close_depth, inf_depth = bds.min() * 0.9, bds.max() * 5.0
    dt = 0.75
    focal = 1.0 / ((1.0 - dt) / close_depth + dt / inf_depth)
    rads = np.percentile(np.abs(poses[:, :3, 3]), 90, 0)
    return render_path_spiral(c2w, up, rads, focal, zrate=zrate, rots=n_rots, n=n_views)


def to_c2w(poses) -> np.ndarray:
    """[N, 3, >=4] -> [N, 4, 4] fp32 camera-to-world matrices (hwf column dropped)"""
    poses = np.asarray(poses, dtype=np.float32)
    out = np.zeros((poses.shape[0], 4, 4), np.float32)
    out[:, :3, :4] = poses[:, :3, :4]
    out[:, 3, 3] = 1.0
    return out


def check_ndc_views(poses, H: int, W: int, focal: float, what: str = "view") -> None:
    """ValueError unless every ray of every view looks down -z (w_z < 0), which NDC needs.  The direction is affine in
    the pixel coordinates (cam = ((x - W/2)/f, -(y - H/2)/f, -1), knerf_generate_rays), so the four corner pixels
    bound the whole frame."""
    poses = np.asarray(poses, dtype=np.float64)
    xs, ys = np.array([0, W - 1, 0, W - 1], np.float64), np.array([0, 0, H - 1, H - 1], np.float64)
    cam = np.stack([(xs - W * 0.5) / focal, -(ys - H * 0.5) / focal, -np.ones(4)], -1)    # [4, 3]
    wz = np.einsum("nj,cj->nc", poses[:, 2, :3], cam)                                     # [N, 4]
    bad = np.nonzero((wz >= 0).any(1))[0]
    if len(bad):
        raise ValueError(f"{what} {bad.tolist()} see rays with w_z >= 0 in the recentred frame: no NDC image "
                         "(not a forward-facing capture; use ndc=False / --no_ndc)")


def largest_divisor(n: int, limit: int) -> int:
    """the largest divisor of n that is <= limit (n itself when n <= limit)"""
    return max(c for c in range(1, min(limit, n) + 1) if n % c == 0)


def ray_chunks_for(image_rays: int, ray_batch: int, requested: int) -> tuple:
    """(render chunk, training chunk) for NeRF.compile(ray_chunks=, train_ray_chunks=): the largest divisors, up to
    `requested`, of the rays of an image batch and of the ray batch (of the image batch without one).  LLFF image sizes
    are rarely multiples of the scripts' chunk sizes: at 378 x 504 and --ray_batch 4096 with 1,024 requested the
    chunks are 1,008 and 1,024, where one chunk dividing both could be no more than 16."""
    render = largest_divisor(image_rays, requested)
    return render, (largest_divisor(ray_batch, requested) if ray_batch else render)


def image_paths(folder: str) -> list:
    return sorted(os.path.join(folder, f) for f in os.listdir(folder) if f.endswith(IMAGE_EXTENSIONS))


class LLFFDatasetLoader:
    """An LLFF scene directory -> [train, val, test] datasets like `DatasetLoader.load_dataset`.

    The constructor reads `poses_bounds.npy` and the image sizes only (host, no GPU) and computes `poses` ([N, 4, 4],
    recentred), `bds`, `H`, `W`, `focal`, `near`, `far`, the split (`i_train`, `i_val`, `i_test`) and the spiral
    `render_poses` ([120, 4, 4]).  Images come from `images_{factor}/` when it exists (H, W from the files), else from
    `images/`, resized on the GPU to (H0 // factor, W0 // factor) by `knerf_image_prepare` (antialiased).  Focal is the
    hwf focal / factor either way.  With `ndc=True`, a dataset view with a corner ray of w_z >= 0 raises ValueError in
    the constructor; the spiral is checked the same way only where it is rendered (`render_path`), so such a spiral
    does not stop training."""

    def __init__(self, data_dir: str, factor: int = 8, llffhold: int = 8, ndc: bool = True, device=None, **kwargs):
        self.data_dir, self.factor, self.llffhold, self.ndc, self.device = data_dir, int(factor), int(llffhold), \
            bool(ndc), device
        raw, bds = parse_poses_bounds(np.load(os.path.join(data_dir, "poses_bounds.npy")))
        folder = os.path.join(data_dir, f"images_{self.factor}")
        self.resize = not os.path.isdir(folder)
        if self.resize:
            folder = os.path.join(data_dir, "images")
        self.image_paths = image_paths(folder)
        if len(self.image_paths) != raw.shape[0]:
            raise ValueError(f"{folder}: {len(self.image_paths)} images for {raw.shape[0]} poses")
        from PIL import Image
        with Image.open(self.image_paths[0]) as im:
            w0, h0 = im.size
        self.H, self.W = (h0 // self.factor, w0 // self.factor) if self.resize else (h0, w0)
        if self.H <= 0 or self.W <= 0:
            raise ValueError(f"factor {self.factor} leaves no pixels of {h0} x {w0} images")
        self.focal = float(raw[0, 2, 4]) / self.factor
        poses = llff_to_opengl(raw)
        poses, self.bds, self.scale = rescale(poses, bds)
        poses = recenter_poses(poses)
        self.render_poses = to_c2w(spiral_poses(poses, self.bds))
        self.poses = to_c2w(poses)
        self.i_train, self.i_val, self.i_test = split_views(poses, self.llffhold)
        self.near, self.far = near_far(self.bds, self.ndc)
        if self.ndc:
            check_ndc_views(self.poses, self.H, self.W, self.focal, "views")

    def render_path(self) -> np.ndarray:
        """the spiral render poses [120, 4, 4]; with NDC, ValueError if one of them has a corner ray of w_z >= 0"""
        if self.ndc:
            check_ndc_views(self.render_poses, self.H, self.W, self.focal, "spiral poses")
        return self.render_poses

    def load_image(self, path) -> torch.Tensor:
        """one view as a float32 CUDA tensor [H, W, 4] (opaque alpha for JPEGs)"""
        return prepare_image(path, self.H, self.W, white_background=False, device=self.device)

    def rays_generator(self, n_sample: int) -> RaysGenerator:
        return RaysGenerator(self.focal, self.W, self.H, self.near, self.far, n_sample, device=self.device,
                             ndc=self.ndc)

    def load_dataset(self, batch_size: int, n_sample: int, ray_batch: int = 0, rank: int = 0, world: int = 1,
                     **kwargs) -> list:
        """[train, val, test] as `DatasetLoader.load_dataset`: whole-view `Dataset`s of `batch_size` views, or with
        `ray_batch` = N > 0 a `RayBatchDataset` training split of N rays per step for rank `rank` of `world`."""
        datasets = []
        for subset, idx in (("train", self.i_train), ("val", self.i_val), ("test", self.i_test)):
            paths = [self.image_paths[i] for i in idx]
            poses = [self.poses[i] for i in idx]
            if subset == "train" and ray_batch:
                images = None
                for k, path in enumerate(paths):
                    img = self.load_image(path)
                    if images is None:
                        images = torch.empty((len(paths),) + tuple(img.shape), dtype=img.dtype, device=img.device)
                    images[k] = img
                datasets.append(RayBatchDataset(images, np.stack(poses), self.focal, self.near, self.far, n_sample,
                                                ray_batch, rank=rank, world=world, ndc=self.ndc))
                logging.info(f"Loaded LLFF {subset} dataset. {len(paths)} images of {self.H} x {self.W}, "
                             f"{ray_batch} rays per step, ndc={self.ndc}.")
                continue
            datasets.append(Dataset(paths, [p.tolist() for p in poses], self.load_image,
                                    self.rays_generator(n_sample), batch_size))
            logging.info(f"Loaded LLFF {subset} dataset. {len(paths)} images of {self.H} x {self.W}, ndc={self.ndc}.")
        return datasets
