"""Synthetic nerf_synthetic-shaped scene (the dataset is not available offline; SURVEY §8d).

Procedural orbit poses exactly like inference.py:61-67 (pose_spherical(theta, phi=-30, t=4.0)), fov of the lego
scene, near 2 / far 6, and ANALYTIC target images: a ray-traced unit sphere with normal shading,
alpha-composited onto white/black exactly like keras_nerf/data/image.py:25-33.  Replaces DatasetLoader
(loader.py:55-113) for benchmarks and tests; host-side glue (torch ops), not part of the hot path."""
from __future__ import annotations

import torch

from .rays import RaysGenerator
from .utils import get_focal_from_fov, pose_spherical

LEGO_FOV = 0.6911112070083618
# Normal shading scaled to a mean of 0.3: with the brighter 0.5 * (n + 1) the white-background objective is met
# fastest by sigma -> 0 everywhere, the ReLU of the sigma head dies within a few Adam steps and the gradient is zero
# from then on (the "gradient is all zero" state the reference warns about, nerf.py:429-451); measured in
# benchmarks/convergence.py: albedo 1.0 + white background stalls at 10.1 dB, 0.6 reaches 21 dB in 12 epochs.
ALBEDO = 0.6


def analytic_rgba(o: torch.Tensor, d: torch.Tensor, white_background: bool = True, albedo: float = None) -> torch.Tensor:
    """o, d [...,3] -> RGBA [...,4] of a unit sphere at the origin, composited like image.py:25-33."""
    b = (o * d).sum(-1)
    c = (o * o).sum(-1) - 1.0
    disc = b * b - c
    hit = disc > 0
    t = -b - torch.sqrt(disc.clamp_min(0))
    n = torch.nn.functional.normalize(o + d * t[..., None], dim=-1)
    rgb = ((ALBEDO if albedo is None else albedo) * 0.5 * (n + 1.0)).clamp(0, 1)
    alpha = hit.to(o.dtype)[..., None]
    bg = torch.ones_like(rgb) if white_background else torch.zeros_like(rgb)
    img = alpha * rgb + (1.0 - alpha) * bg
    return torch.cat([img, alpha], dim=-1).clamp(0, 1)


class SyntheticScene:
    def __init__(self, image_wh: int, n_coarse: int, n_views: int = 100, phi: float = -30.0, radius: float = 4.0,
                 near: float = 2.0, far: float = 6.0, white_background: bool = True, device=None):
        self.wh, self.n_views, self.phi, self.radius = image_wh, n_views, phi, radius
        self.white = white_background
        self.focal = get_focal_from_fov(LEGO_FOV, image_wh)
        self.gen = RaysGenerator(self.focal, image_wh, image_wh, near, far, n_coarse, device=device)

    def pose(self, k: int):
        return pose_spherical(360.0 * (k % self.n_views) / self.n_views, self.phi, self.radius)

    def view(self, k: int, seed=None):
        """(image[H,W,4], (o[H,W,3], d[H,W,3], t[H,W,Nc])) of view k with fresh stratified jitter."""
        o, d, t = self.gen(self.pose(k), seed=seed)
        return analytic_rgba(o, d, self.white), (o, d, t)

    def ray_crop(self, k: int, h: int, w: int, y0: int, x0: int, seed=None):
        """an h x w image crop of view k at (y0, x0), shaped [1, h, w, .] for NeRF.compile(image_height=h,
        image_width=w): a genuine sub-image (SSIM stays meaningful) that mixes object and background"""
        img, (o, d, t) = self.view(k, seed=seed)
        y0, x0 = max(0, min(y0, self.wh - h)), max(0, min(x0, self.wh - w))
        f = lambda x: x[y0:y0 + h, x0:x0 + w][None].contiguous()  # noqa: E731
        return f(img), (f(o), f(d), f(t))

    def ray_batch(self, k: int, n_rays: int, offset: int = 0, seed=None):
        """a contiguous window of n_rays rays of view k, shaped [1, n_rays/256, 256, .] for NeRF.compile"""
        img, (o, d, t) = self.view(k, seed=seed)
        total = self.wh * self.wh
        assert n_rays <= total and n_rays % 256 == 0
        off = offset % (total - n_rays + 1)
        sl = slice(off, off + n_rays)
        sh = (1, n_rays // 256, 256)
        f = lambda x: x.reshape(total, -1)[sl].reshape(sh + (x.shape[-1],)).contiguous()  # noqa: E731
        return f(img), (f(o), f(d), f(t))


def write_nerf_synthetic_like(data_dir: str, image_wh: int = 64, n_train: int = 8, n_val: int = 2, n_test: int = 2,
                              phi: float = -30.0, radius: float = 4.0) -> str:
    """A nerf_synthetic-shaped directory (transforms_{train,val,test}.json + RGBA PNG frames, the layout
    loader.py:41-76 reads) of the analytic sphere scene, for tests and examples.  Host-only (torch CPU + Pillow)."""
    import json
    import os

    import numpy as np
    from PIL import Image

    focal = get_focal_from_fov(LEGO_FOV, image_wh)
    ys, xs = torch.meshgrid(torch.arange(image_wh, dtype=torch.float32), torch.arange(image_wh, dtype=torch.float32),
                            indexing="ij")
    cam = torch.stack([(xs - image_wh * 0.5) / focal, -(ys - image_wh * 0.5) / focal, -torch.ones_like(xs)], dim=-1)
    k = 0
    for subset, n in (("train", n_train), ("val", n_val), ("test", n_test)):
        os.makedirs(os.path.join(data_dir, subset), exist_ok=True)
        frames = []
        for i in range(n):
            c2w = torch.from_numpy(np.asarray(pose_spherical(360.0 * k / (n_train + n_val + n_test), phi, radius),
                                              dtype=np.float32))
            k += 1
            d = torch.nn.functional.normalize(cam @ c2w[:3, :3].T, dim=-1)
            o = c2w[:3, 3].expand_as(d)
            rgba = analytic_rgba(o, d, white_background=False)      # straight colour * alpha on black == premultiplied
            png = (rgba.numpy() * 255.0 + 0.5).astype(np.uint8)
            Image.fromarray(png, mode="RGBA").save(os.path.join(data_dir, subset, f"r_{i}.png"))
            frames.append({"file_path": f"./{subset}/r_{i}", "rotation": 0.0, "transform_matrix": c2w.tolist()})
        with open(os.path.join(data_dir, f"transforms_{subset}.json"), "w") as f:
            json.dump({"camera_angle_x": LEGO_FOV, "frames": frames}, f)
    return data_dir


# ---- a forward-facing scene in LLFF layout (data.llff) ----------------------------------------------------------------
# Three spheres 1.9 to 7.7 units in front of the cameras and a textured back plane at depth 50: a depth ratio of about
# 26, the situation NDC is for.  (centre, radius, albedo)
LLFF_SPHERES = (((0.35, 0.15, -2.5), 0.6, (0.9, 0.35, 0.2)),
                ((-0.9, -0.4, -4.2), 0.9, (0.25, 0.7, 0.35)),
                ((1.2, 0.9, -6.5), 1.2, (0.3, 0.4, 0.9)))
LLFF_PLANE_Z = -50.0


def llff_like_poses(n_views: int, seed: int = 0) -> torch.Tensor:
    """[n_views, 3, 4] camera-to-world matrices ([right, up, back] axes, cameras looking along -z) on a small planar
    spiral of radius <= 0.3 at z = 0, each turned by up to 3 degrees about x and y"""
    import math
    g = torch.Generator().manual_seed(seed)
    out = torch.zeros((n_views, 3, 4), dtype=torch.float64)
    for k in range(n_views):
        a = 2.0 * math.pi * 1.5 * k / max(n_views, 1)
        r = 0.3 * (0.4 + 0.6 * (k + 1) / n_views)
        yaw, pitch = (torch.rand(2, generator=g, dtype=torch.float64) * 2 - 1) * math.radians(3.0)
        cy, sy, cp, sp = math.cos(yaw), math.sin(yaw), math.cos(pitch), math.sin(pitch)
        ry = torch.tensor([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]], dtype=torch.float64)
        rx = torch.tensor([[1, 0, 0], [0, cp, -sp], [0, sp, cp]], dtype=torch.float64)
        out[k, :, :3] = ry @ rx
        out[k, :, 3] = torch.tensor([r * math.cos(a), r * math.sin(a), 0.0], dtype=torch.float64)
    return out


def render_llff_like(c2w: torch.Tensor, H: int, W: int, focal: float) -> tuple:
    """host ray trace of the forward-facing scene for one [3, 4] pose with the camera model of knerf_generate_rays
    -> (rgb [H, W, 3] in [0, 1], camera-space depth [H, W])"""
    ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64), indexing="ij")
    cam = torch.stack([(xs - W * 0.5) / focal, -(ys - H * 0.5) / focal, -torch.ones_like(xs)], -1)
    c2w = c2w.to(torch.float64)
    d = torch.nn.functional.normalize(cam @ c2w[:, :3].T, dim=-1)
    o = c2w[:, 3].expand_as(d)
    light = torch.nn.functional.normalize(torch.tensor([0.5, 0.8, 0.6], dtype=torch.float64), dim=0)
    t_hit = (LLFF_PLANE_Z - o[..., 2]) / d[..., 2]                          # every ray of the frame looks down -z
    p = o + d * t_hit[..., None]
    # back plane: smooth colour waves (period about 6 units) and a checker of period 8
    check = ((torch.floor(p[..., 0] / 4) + torch.floor(p[..., 1] / 4)) % 2)
    rgb = torch.stack([0.5 + 0.3 * torch.sin(p[..., 0] * 1.05), 0.5 + 0.3 * torch.sin(p[..., 1] * 0.9 + 1.0),
                       0.45 + 0.25 * torch.cos((p[..., 0] + p[..., 1]) * 0.7)], -1) * (0.75 + 0.25 * check[..., None])
    for centre, radius, albedo in LLFF_SPHERES:
        c = torch.tensor(centre, dtype=torch.float64)
        oc = o - c
        b = (oc * d).sum(-1)
        disc = b * b - ((oc * oc).sum(-1) - radius * radius)
        t = -b - torch.sqrt(disc.clamp_min(0))
        hit = (disc > 0) & (t > 0) & (t < t_hit)
        n = torch.nn.functional.normalize(oc + d * t[..., None], dim=-1)
        stripes = 0.8 + 0.2 * torch.sin((n[..., 1] * 9.0))
        shade = (0.35 + 0.65 * (n @ light).clamp_min(0)) * stripes
        col = torch.tensor(albedo, dtype=torch.float64) * shade[..., None]
        rgb = torch.where(hit[..., None], col, rgb)
        t_hit = torch.where(hit, t, t_hit)
    depth = t_hit * (d @ -c2w[:, 2])                                        # along the camera's viewing axis
    return rgb.clamp(0, 1), depth


def write_llff_like(data_dir: str, H: int = 48, W: int = 64, n_views: int = 20, factors=(), seed: int = 0) -> str:
    """An LLFF-layout directory of the forward-facing analytic scene: `poses_bounds.npy` ([n_views, 17] in LLFF's own
    [down, right, back] axis order, hwf = (H, W, focal), bounds = the view's nearest and farthest visible depth) and
    `images/` PNGs of H x W, plus `images_{f}/` at (H // f, W // f) for every f in `factors`, rendered with focal / f.
    Poses from `llff_like_poses(n_views, seed)`.  Host-only (torch CPU + Pillow)."""
    import os

    import numpy as np
    from PIL import Image

    focal = 0.9 * W
    poses = llff_like_poses(n_views, seed)
    rows = []
    for f in (1,) + tuple(factors):
        folder = os.path.join(data_dir, "images" if f == 1 else f"images_{f}")
        os.makedirs(folder, exist_ok=True)
        for k in range(n_views):
            rgb, depth = render_llff_like(poses[k], H // f, W // f, focal / f)
            png = (rgb.numpy() * 255.0 + 0.5).astype(np.uint8)
            Image.fromarray(png, mode="RGB").save(os.path.join(folder, f"view_{k:03d}.png"))
            if f == 1:
                c2w = poses[k].numpy()
                m = np.stack([-c2w[:, 1], c2w[:, 0], c2w[:, 2], c2w[:, 3], np.array([H, W, focal])], 1)
                rows.append(np.concatenate([m.reshape(-1), [float(depth.min()), float(depth.max())]]))
    np.save(os.path.join(data_dir, "poses_bounds.npy"), np.stack(rows).astype(np.float32))
    return data_dir
