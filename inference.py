"""360-degree orbit render -> GIF.  Same command line as the reference's inference.py (its flags at :14-40);
`--precision bf16` (default) selects the tcgen05 path, `--precision fp32` the parity mode.  Under torchrun the
frames are sharded across the GPUs and gathered on rank 0.

--dataset_type llff --data_dir DIR renders the 120-view spiral of an LLFF scene (data.llff.LLFFDatasetLoader) at its
H, W and focal instead, with NDC rays unless --no_ndc (use the settings the model was trained with)."""
import argparse
import logging
import os

import numpy as np
import torch

from keras_nerf_b200 import NeRF, RaysGenerator, get_focal_from_fov, pose_spherical
from keras_nerf_b200.utils.video import mimwrite


def main(argv=None):
    parser = argparse.ArgumentParser()
    parser.add_argument('--name', type=str, default='', help='Name of the nerf model')
    parser.add_argument('--model_dirs', type=str, required=True)
    parser.add_argument('--ray_chunks', type=int, default=4096)
    parser.add_argument('--img_wh', type=int, default=128)
    parser.add_argument('--near', type=float, default=2.0)
    parser.add_argument('--far', type=float, default=6.0)
    parser.add_argument('--fov', type=float, default=0.6911112070083618)
    parser.add_argument('--eagerly', action='store_true')
    parser.add_argument('--white_bg', action='store_true')
    parser.add_argument('--phi', type=float, default=-30.0)
    parser.add_argument('--z_translate', type=float, default=4.0)
    parser.add_argument('--output_dir', type=str, default='output')
    parser.add_argument('--output_freq', type=int, default=10)
    parser.add_argument('--verbose', action='store_true')
    parser.add_argument('--precision', type=str, default='bf16', choices=['bf16', 'fp32', 'fp32_tc'])
    parser.add_argument('--dataset_type', type=str, default='blender', choices=['blender', 'llff'],
                        help="'blender': the orbit of the flags above; 'llff': the spiral path of --data_dir")
    parser.add_argument('--data_dir', type=str, default=None, help='llff: the scene directory')
    parser.add_argument('--factor', type=int, default=8, help='llff: image downsampling factor')
    parser.add_argument('--no_ndc', action='store_true', help='llff: the model was trained with --no_ndc')
    args = parser.parse_args(argv)
    logging.basicConfig(level=logging.DEBUG if args.verbose else logging.INFO,
                        format='%(asctime)s | %(name)s | %(levelname)s | %(message)s')
    logging.info(args)
    if args.name == '':
        args.name = args.model_dirs.rstrip('/').split('/')[-1]
    if not NeRF.has_checkpoint(args.model_dirs):
        raise FileNotFoundError(f"Model not found for {args.model_dirs}")

    strategy = None
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        from keras_nerf_b200.distributed import RayShardedStrategy
        strategy = RayShardedStrategy()
    nerf = NeRF(model_path=args.model_dirs, precision=args.precision)
    H = W = args.img_wh
    if args.dataset_type == 'llff':
        if args.data_dir is None:
            raise ValueError("--dataset_type llff needs --data_dir")
        from keras_nerf_b200.data.llff import LLFFDatasetLoader, largest_divisor
        scene = LLFFDatasetLoader(args.data_dir, factor=args.factor, ndc=not args.no_ndc)
        H, W = scene.H, scene.W
        args.ray_chunks = largest_divisor(H * W, args.ray_chunks)        # NeRF.compile: a divisor of H * W
        poses = list(scene.render_path())
        rays_generator = scene.rays_generator(nerf.n_coarse)
        logging.info(f"LLFF spiral: {H} x {W}, focal {scene.focal:.3f}, ndc={scene.ndc}; "
                     "--img_wh, --near, --far, --fov, --phi and --z_translate are ignored")
    else:
        poses = [pose_spherical(float(theta), args.phi, args.z_translate)
                 for theta in range(0, 360, args.output_freq)]
        rays_generator = RaysGenerator(focal_length=get_focal_from_fov(args.fov, args.img_wh),
                                       image_width=args.img_wh, image_height=args.img_wh, near=args.near,
                                       far=args.far, n_sample=nerf.n_coarse)
    logging.info(f'Camera Matrix Shape: {np.stack(poses).shape}')
    nerf.compile(optimizer='adam', loss='mean_squared_error', batch_size=1, image_width=W,
                 image_height=H, ray_chunks=args.ray_chunks, white_background=args.white_bg,
                 is_training=False)
    nerf.coarse.summary()
    nerf.fine.summary()

    lo, hi = (0, len(poses)) if strategy is None else strategy.shard_bounds(len(poses))
    images = []
    for k in range(lo, hi):                                  # whole frames per rank (SURVEY 8e)
        rays = tuple(r[None] for r in rays_generator(poses[k]))
        _, fine = nerf.predict_and_render_images(rays)
        images.append(fine['image'][0])
    frames = torch.stack(images) if images else torch.empty((0, H, W, 3), device=nerf.device)
    if strategy is not None:
        frames = strategy.gather_rows(frames, len(poses))
        rank = strategy.rank
        torch.distributed.destroy_process_group()
        if rank != 0:
            return None
    os.makedirs(args.output_dir, exist_ok=True)
    logging.info("creating the video from the frames...")
    out = os.path.join(args.output_dir, f"{args.name}.gif")
    mimwrite(out, list(frames.cpu().numpy()), fps=20)
    return out


if __name__ == "__main__":
    main()
