"""Triangle mesh of a trained model -> binary PLY: the level set sigma = --threshold of one network on a
--resolution^3 lattice over [-bound, bound]^3 (marching tetrahedra), vertex colours seen along the normals.
Flags in the style of inference.py; writes <output_dir>/<name>.ply."""
import argparse
import logging
import os

from keras_nerf_b200 import NeRF
from keras_nerf_b200.utils.mesh import write_ply


def main(argv=None):
    parser = argparse.ArgumentParser()
    parser.add_argument('--name', type=str, default='', help='Name of the nerf model')
    parser.add_argument('--model_dirs', type=str, required=True)
    parser.add_argument('--resolution', type=int, default=256, help='lattice points per axis')
    parser.add_argument('--threshold', type=float, default=50.0, help='density of the surface (inside: sigma > it)')
    parser.add_argument('--bound', type=float, default=1.5, help='half side of the cube [-bound, bound]^3')
    parser.add_argument('--network', type=str, default='fine', choices=['fine', 'coarse'])
    parser.add_argument('--precision', type=str, default='bf16', choices=['bf16', 'fp32', 'fp32_tc'])
    parser.add_argument('--no_colors', action='store_true', help='skip the per-vertex colour query')
    parser.add_argument('--output_dir', type=str, default='output')
    parser.add_argument('--verbose', action='store_true')
    args = parser.parse_args(argv)
    logging.basicConfig(level=logging.DEBUG if args.verbose else logging.INFO,
                        format='%(asctime)s | %(name)s | %(levelname)s | %(message)s')
    logging.info(args)
    if args.name == '':
        args.name = args.model_dirs.rstrip('/').split('/')[-1]
    if not NeRF.has_checkpoint(args.model_dirs):
        raise FileNotFoundError(f"Model not found for {args.model_dirs}")

    nerf = NeRF(model_path=args.model_dirs, precision=args.precision)
    nerf.compile(optimizer='adam', loss='mean_squared_error', batch_size=1, image_width=1, image_height=1,
                 ray_chunks=1, is_training=False)
    mesh = nerf.extract_mesh(resolution=args.resolution, threshold=args.threshold, bound=args.bound,
                             network=args.network, colors=not args.no_colors)
    sec = mesh["seconds"]
    logging.info("density grid %d^3: %.3f s, isosurface: %.3f s (V=%d, T=%d), colours: %.3f s", args.resolution,
                 sec["grid"], sec["isosurface"], mesh["vertices"].shape[0], mesh["faces"].shape[0], sec["colors"])
    if mesh["faces"].shape[0] == 0:
        logging.warning("the surface is empty: no lattice point inside the box has sigma > %g", args.threshold)
    out = os.path.join(args.output_dir, f"{args.name}.ply")
    write_ply(out, mesh["vertices"], mesh["faces"], normals=mesh["normals"], colors=mesh["colors"])
    logging.info("wrote %s", out)
    return out


if __name__ == "__main__":
    main()
