"""DatasetLoader (reference: keras_nerf/data/loader.py) -- nerf_synthetic-style directories
(`transforms_{train,val,test}.json` + PNG frames) -> three batched datasets of (images, rays), or, with
`ray_batch`, a training set of random ray batches drawn across all training views."""
from __future__ import annotations

import json
import logging
import os
import random

import torch

from .image import ImageLoader
from .. import _lib
from .rays import RaysGenerator, generate_ray_batch
from .utils import get_focal_from_fov


class _Iterator:
    """What `iter(tf.data.Dataset)` gives the callback (callback.py:56-57, 177): next() and get_next()."""

    def __init__(self, gen):
        self._gen = gen

    def __iter__(self):
        return self

    def __next__(self):
        return next(self._gen)

    def get_next(self):
        try:
            return next(self._gen)
        except StopIteration:
            raise IndexError("End of sequence") from None   # tf.errors.OutOfRangeError


class Dataset:
    """The slice of tf.data.Dataset the reference uses on `zip((images, rays)).shuffle(B).batch(B,
    drop_remainder=True).prefetch(AUTOTUNE)` (loader.py:99-107): re-iterable, reshuffled on every pass with a
    buffer of `shuffle_buffer` elements, `take(n)`, `len()`.

    Every pass re-runs the rays map, so the stratified jitter is fresh each epoch as in the reference (its
    `map(rays_generator)` is not cached).  Prepared images ARE cached on the GPU after the first pass (decode +
    resize are deterministic), which is what `prefetch` hides in the reference."""

    def __init__(self, image_paths, camera_params, image_loader, rays_generator, batch_size, shuffle_buffer=None,
                 limit=None, seed=None):
        self.image_paths, self.camera_params = list(image_paths), list(camera_params)
        self.image_loader, self.rays_generator = image_loader, rays_generator
        self.batch_size = int(batch_size)
        self.shuffle_buffer = self.batch_size if shuffle_buffer is None else int(shuffle_buffer)
        self.limit = limit
        self._rng = random.Random(seed)
        self._cache = {}

    def _element(self, i):
        if i not in self._cache:
            self._cache[i] = self.image_loader(self.image_paths[i])
        return self._cache[i], self.rays_generator(self.camera_params[i])

    def _shuffled_indices(self):
        # tf.data shuffle(buffer): fill a buffer, emit a uniformly chosen slot, refill it from the stream
        buf, out = [], []
        for i in range(len(self.image_paths)):
            buf.append(i)
            if len(buf) > max(self.shuffle_buffer, 1) - 1:
                out.append(buf.pop(self._rng.randrange(len(buf))))
        while buf:
            out.append(buf.pop(self._rng.randrange(len(buf))))
        return out

    def _batches(self):
        order, B = self._shuffled_indices(), self.batch_size
        n = len(order) // B                                # drop_remainder=True
        if self.limit is not None:
            n = min(n, self.limit)
        for b in range(n):
            elems = [self._element(i) for i in order[b * B:(b + 1) * B]]
            images = torch.stack([e[0] for e in elems])
            rays = tuple(torch.stack([e[1][k] for e in elems]) for k in range(3))
            yield images, rays

    def __iter__(self):
        return _Iterator(self._batches())

    def __len__(self):
        n = len(self.image_paths) // self.batch_size
        return n if self.limit is None else min(n, self.limit)

    def take(self, count):
        return Dataset(self.image_paths, self.camera_params, self.image_loader, self.rays_generator,
                       self.batch_size, self.shuffle_buffer, limit=count, seed=self._rng.random())


def permutation_seed() -> int:
    """Key of the epoch permutations of a RayBatchDataset: from the torch seed (torch.manual_seed, the scripts'
    tf.random.set_seed) and NOT the rank, so that every rank of a data-parallel run walks the same order."""
    return ((torch.initial_seed() & 0xFFFFFFFF) * 0x9E3779B1 + 0x52A7BA7C) & 0xFFFFFFFFFFFFFFFF


class RayBatchDataset:
    """Training rays drawn at random from the pixels of ALL training views (vanilla NeRF's `N_rand`) instead of whole
    views: every pass is one epoch that visits each of the P = n_img*H*W pixels exactly once, in the order of a
    permutation computed inside `knerf_generate_ray_batch` (one new key per pass, nothing stored per epoch).

    Yields (targets[N,3], (o[N,3], d[N,3], t[N,Nc])) for `NeRF.compile(..., ray_batch=N)`.  `len()` is
    floor(P / (N*world)) steps (the remainder is dropped, like `drop_remainder=True`).  Rank r of `world` takes
    positions [(step*world + r)*N, +N) of the epoch's order, so the ranks' batches of a step together are exactly the
    single-process batch of N*world rays.  The permutation key (`perm_seed`, default `permutation_seed()`) must be
    the same on every rank; the stratified jitter is rank-keyed like every other draw (`_lib.seed_stream`).

    `images` [n_img, H, W, C] (CUDA fp32, C >= 3) is the prepared view cache (n*H*W*16 bytes for RGBA: 256 MB for 100
    views of 400 x 400), `poses` [n_img, 4, 4].  `epoch` is the epoch the next pass walks; each pass advances it, and a
    resumed run sets it to the first epoch it trains."""

    def __init__(self, images, poses, focal, near, far, n_sample, ray_batch, rank=0, world=1, perm_seed=None,
                 epoch=0, limit=None):
        self.images = torch.as_tensor(images).contiguous()        # the kernel refuses anything but CUDA fp32
        self.poses = torch.as_tensor(poses, dtype=torch.float32, device=self.images.device).reshape(-1, 4, 4)
        self.poses = self.poses.contiguous()
        n_img, H, W, C = self.images.shape
        if self.poses.shape[0] != n_img or C < 3:
            raise ValueError(f"need images [n,H,W,C>=3] and poses [n,4,4], got {tuple(self.images.shape)} and "
                             f"{tuple(self.poses.shape)}")
        self.focal, self.near, self.far, self.n_sample = float(focal), float(near), float(far), int(n_sample)
        self.ray_batch, self.rank, self.world = int(ray_batch), int(rank), int(world)
        if self.ray_batch <= 0 or not 0 <= self.rank < self.world:
            raise ValueError(f"ray_batch must be > 0 and 0 <= rank < world (got {ray_batch}, {rank}, {world})")
        self.n_pixels = n_img * H * W
        self.perm_seed = permutation_seed() if perm_seed is None else int(perm_seed)
        self.epoch = int(epoch)
        self.limit = limit

    def window(self, step):
        """first position of this rank's batch `step` in the epoch's order"""
        return (step * self.world + self.rank) * self.ray_batch

    def batch(self, epoch, step, u=None, seed=None, with_pixel=False):
        """batch `step` of epoch `epoch` of this rank: (targets, (o, d, t)) (+ pixel ids when `with_pixel`)"""
        out = generate_ray_batch(self.images, self.poses, self.focal, self.near, self.far, self.n_sample,
                                 self.perm_seed, epoch, self.window(step), self.ray_batch, u=u, seed=seed,
                                 with_pixel=with_pixel)
        return (out[0], tuple(out[1:4])) + ((out[4],) if with_pixel else ())

    def _batches(self, epoch):
        seeds = _lib.seed_stream(0x5EED0001, advance=epoch)    # jitter: rank-keyed, not replayed by a resumed run
        for step in range(len(self)):
            yield self.batch(epoch, step, seed=next(seeds))

    def __iter__(self):
        epoch, self.epoch = self.epoch, self.epoch + 1
        return _Iterator(self._batches(epoch))

    def __len__(self):
        n = self.n_pixels // (self.ray_batch * self.world)
        return n if self.limit is None else min(n, self.limit)

    def take(self, count):
        """the first `count` batches of each pass; the view cache is shared, the epoch counter is the copy's own"""
        return RayBatchDataset(self.images, self.poses, self.focal, self.near, self.far, self.n_sample,
                               self.ray_batch, self.rank, self.world, self.perm_seed, self.epoch, limit=count)


class DatasetLoader:
    """Same constructor and methods as keras_nerf/data/loader.py:12-113."""

    def __init__(self, data_dir: str, white_background: bool = False, device=None, **kwargs):
        self.data_dir = data_dir
        self.white_background = white_background
        self.device = device

    def _load_json(self, filename: str) -> dict:
        with open(filename, 'r') as f:
            return json.load(f)

    def _load_image_path_and_camera_param(self, json_config: dict) -> tuple:
        image_paths, camera_params = [], []
        for frame in json_config['frames']:                 # loader.py:47-51
            image_paths.append(os.path.join(self.data_dir, f"{frame['file_path']}.png"))
            camera_params.append(frame['transform_matrix'])
        return image_paths, camera_params

    def load_dataset(self, batch_size: int, image_width: int, image_height: int, near: float, far: float,
                     n_sample: int, ray_batch: int = 0, rank: int = 0, world: int = 1) -> list:
        """[train, val, test].  ray_batch = N > 0: the train split is a RayBatchDataset of N rays per step for rank
        `rank` of `world` (every training view decoded and prepared once into one device tensor); val and test stay
        whole-view Datasets of `batch_size` views."""
        image_loader = ImageLoader(image_width, image_height, self.white_background, device=self.device)
        datasets = []
        for subset in ['train', 'val', 'test']:
            json_config = self._load_json(os.path.join(self.data_dir, f"transforms_{subset}.json"))
            focal_length = get_focal_from_fov(json_config['camera_angle_x'], image_width)
            image_paths, camera_params = self._load_image_path_and_camera_param(json_config)
            if subset == 'train' and ray_batch:
                images = None
                for i, path in enumerate(image_paths):
                    img = image_loader(path)
                    if images is None:
                        images = torch.empty((len(image_paths),) + tuple(img.shape), dtype=img.dtype,
                                             device=img.device)
                    images[i] = img
                # ImageLoader's [image_width, image_height] (sic) flattened is what the whole-view path pairs with ray
                # y*W + x; the same view of the bytes keeps that pairing for non-square images
                images = images.view(len(image_paths), image_height, image_width, images.shape[-1])
                datasets.append(RayBatchDataset(images, camera_params, focal_length, near, far, n_sample, ray_batch,
                                                rank=rank, world=world))
                logging.info(f"Loaded {subset} dataset. {len(image_paths)} images, {ray_batch} rays per step.")
                continue
            rays_generator = RaysGenerator(focal_length=focal_length, image_width=image_width,
                                           image_height=image_height, near=near, far=far, n_sample=n_sample,
                                           device=self.device)
            datasets.append(Dataset(image_paths, camera_params, image_loader, rays_generator, batch_size))
            logging.info(f"Loaded {subset} dataset. {len(image_paths)} images.")
        return datasets
