"""Float64 NumPy restatement of vanilla NeRF's load_llff.py (no spherify) and run_nerf_helpers.ndc_rays, written from
the papers' code independently of keras_nerf_b200.data.llff, for tests/test_llff_cpu.py and tests/test_gpu_llff.py."""
import numpy as np


def _unit(v):
    return v / np.linalg.norm(v)


def _look(back, up, centre):
    right = _unit(np.cross(up, back))
    return np.stack([right, _unit(np.cross(_unit(back), right)), _unit(back), centre], 1)


def load_poses(poses_bounds, bd_factor=0.75):
    """poses_bounds [N, 17] -> dict of the intermediate float64 results of load_llff_data (recenter=True)"""
    a = np.asarray(poses_bounds, np.float64)
    m = a[:, :15].reshape(-1, 3, 5)
    bds = a[:, 15:].copy()
    swapped = np.concatenate([m[:, :, 1:2], -m[:, :, 0:1], m[:, :, 2:]], 2)
    sc = 1.0 / (bds.min() * bd_factor)
    scaled = swapped.copy()
    scaled[:, :, 3] *= sc
    bds = bds * sc

    def avg(p):
        return _look(p[:, :, 2].sum(0), p[:, :, 1].sum(0), p[:, :, 3].mean(0))

    c = np.eye(4)
    c[:3] = avg(scaled)
    rec = scaled.copy()
    for k in range(len(rec)):
        full = np.eye(4)
        full[:3] = scaled[k, :, :4]
        rec[k, :, :4] = np.linalg.solve(c, full)[:3]
    # render_path_spiral
    center = avg(rec)
    up = _unit(rec[:, :, 1].sum(0))
    close, inf = bds.min() * 0.9, bds.max() * 5.0
    focus = 1.0 / (0.25 / close + 0.75 / inf)
    rads = np.append(np.percentile(np.abs(rec[:, :, 3]), 90, 0), 1.0)
    spiral = []
    for th in np.linspace(0.0, 4.0 * np.pi, 121)[:-1]:
        cpos = center @ (np.array([np.cos(th), -np.sin(th), -np.sin(0.5 * th), 1.0]) * rads)
        z = _unit(cpos - center @ np.array([0.0, 0.0, -focus, 1.0]))
        spiral.append(_look(z, up, cpos))
    return dict(swapped=swapped, scaled=scaled, bds=bds, sc=sc, recentred=rec, spiral=np.array(spiral),
                near=0.9 * bds.min(), far=bds.max())


def split(recentred, llffhold):
    """run_nerf.py's split; llffhold <= 0 keeps load_llff.py's i_test, the view closest to the average pose"""
    n = len(recentred)
    if llffhold > 0:
        test = list(range(0, n, llffhold))
    else:
        centre = recentred[:, :, 3].mean(0)
        test = [int(np.argmin(((recentred[:, :, 3] - centre) ** 2).sum(-1)))]
    return [i for i in range(n) if i not in test], test, test


def world_rays(c2w, H, W, focal):
    """run_nerf_helpers.get_rays (cx = W/2, cy = H/2, no pixel-centre offset): o [H,W,3], unnormalised d [H,W,3]"""
    c2w = np.asarray(c2w, np.float64)
    j, i = np.meshgrid(np.arange(H, dtype=np.float64), np.arange(W, dtype=np.float64), indexing="ij")
    dirs = np.stack([(i - W * 0.5) / focal, -(j - H * 0.5) / focal, -np.ones_like(i)], -1)
    d = dirs @ c2w[:3, :3].T
    return np.broadcast_to(c2w[:3, 3], d.shape).copy(), d


def ndc_rays(H, W, focal, near, rays_o, rays_d):
    """run_nerf_helpers.ndc_rays, float64"""
    t = -(near + rays_o[..., 2]) / rays_d[..., 2]
    rays_o = rays_o + t[..., None] * rays_d
    o0 = -1.0 / (W / (2.0 * focal)) * rays_o[..., 0] / rays_o[..., 2]
    o1 = -1.0 / (H / (2.0 * focal)) * rays_o[..., 1] / rays_o[..., 2]
    o2 = 1.0 + 2.0 * near / rays_o[..., 2]
    d0 = -1.0 / (W / (2.0 * focal)) * (rays_d[..., 0] / rays_d[..., 2] - rays_o[..., 0] / rays_o[..., 2])
    d1 = -1.0 / (H / (2.0 * focal)) * (rays_d[..., 1] / rays_d[..., 2] - rays_o[..., 1] / rays_o[..., 2])
    d2 = -2.0 * near / rays_o[..., 2]
    return np.stack([o0, o1, o2], -1), np.stack([d0, d1, d2], -1)
