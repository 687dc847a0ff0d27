"""Training script.  Same command line as the reference's train.py / train_single.py (flags at train.py:19-54).

Multi-GPU: launch with `torchrun --nproc-per-node N train.py ...` -- one process per GPU replaces
tf.distribute.MirroredStrategy (train.py:75): the loader batches `batch_size x N` views exactly like the
reference's global batch (train.py:84-87) and each rank trains on its own `batch_size` views; the accumulated MLP
gradients are SUM-all-reduced over NCCL before the two Adam steps.

--ray_batch N trains on N random rays per replica and step, drawn across all training views (an epoch visits every
pixel once; data.loader.RayBatchDataset) instead of --batch_size whole views; validation and the monitor still
render --batch_size whole views.  Under torchrun the ranks take disjoint windows of the same epoch order.

--dataset_type llff trains on a forward-facing LLFF scene (poses_bounds.npy + images/, data.llff.LLFFDatasetLoader):
H, W and focal come from the dataset (--factor downsamples), every --llffhold-th view is held out, and the rays are in
normalized device coordinates unless --no_ndc.  --img_wh, --near and --far are ignored then."""
import argparse
import logging
import os

import numpy as np
import torch

from keras_nerf_b200 import NeRF
from keras_nerf_b200.data.loader import DatasetLoader, _Iterator
from keras_nerf_b200.model.nerf.callback import NeRFTrainMonitor


class ReplicaBatches:
    """Keras splits every global batch evenly over the replicas of a MirroredStrategy; rank r takes slice r."""

    def __init__(self, dataset, strategy, per_replica):
        self.dataset, self.strategy, self.per_replica = dataset, strategy, per_replica

    def _slice(self, x):
        r, b = self.strategy.rank, self.per_replica
        return x[r * b:(r + 1) * b]

    def _batches(self):
        for images, rays in self.dataset:
            yield self._slice(images), tuple(self._slice(x) for x in rays)

    def __iter__(self):
        return _Iterator(self._batches())                    # next() and get_next(), like the loader's datasets

    def __len__(self):
        return len(self.dataset)

    def take(self, n):
        return ReplicaBatches(self.dataset.take(n), self.strategy, self.per_replica)


def main(argv=None, multi_gpu=True):
    np.random.seed(42)
    torch.manual_seed(42)                                    # tf.random.set_seed(42) (train.py:10)
    parser = argparse.ArgumentParser()
    parser.add_argument('--name', type=str, default='lego', help='Name of the nerf model')
    parser.add_argument('--data_dir', type=str, default='data/nerf_synthetic/lego')
    parser.add_argument('--num_coarse_samples', type=int, default=64)
    parser.add_argument('--num_fine_samples', type=int, default=128)
    parser.add_argument('--pos_emb_xyz', type=int, default=10)
    parser.add_argument('--pos_emb_dir', type=int, default=4)
    parser.add_argument('--num_layers', type=int, default=8)
    parser.add_argument('--num_units', type=int, default=256)
    parser.add_argument('--skip_layer', type=int, default=4)
    parser.add_argument('--img_wh', type=int, default=512 if multi_gpu else 128)
    parser.add_argument('--near', type=float, default=2.0)
    parser.add_argument('--far', type=float, default=6.0)
    parser.add_argument('--white_bg', action='store_true')
    parser.add_argument('--num_epochs', type=int, default=250)
    parser.add_argument('--batch_size', type=int, default=1)
    parser.add_argument('--num_gpus', type=int, default=1)   # parsed and unused, as in train.py:44
    parser.add_argument('--ray_chunks', type=int, default=1024 if multi_gpu else 2048)
    parser.add_argument('--eagerly', action='store_true')
    parser.add_argument('--model_dirs', type=str, default='model')
    parser.add_argument('--log_dir', type=str, default='logs')
    parser.add_argument('--log_freq', type=int, default=5 if multi_gpu else 1)
    parser.add_argument('--verbose', action='store_true')
    parser.add_argument('--precision', type=str, default='bf16', choices=['bf16', 'fp32', 'fp32_tc'])
    parser.add_argument('--fuse_chunks', type=str, default='auto',
                        help="execute several ray chunks of a training step per library call: 'auto' (up to 32,768 rays), "
                             "'off', or a count.  The chunks of a step are independent, so the step is the same")
    parser.add_argument('--records', type=str, default='fp8', choices=['fp8', 'bf16'],
                        help='bf16 mode: format of the activation / gradient records kept for the weight gradients')
    parser.add_argument('--ray_batch', type=int, default=0,
                        help='train on this many random rays per replica and step, drawn across all training views '
                             '(0: --batch_size whole views per step, the reference\'s pipeline)')
    parser.add_argument('--dataset_type', type=str, default='blender', choices=['blender', 'llff'],
                        help="'blender': a nerf_synthetic directory (transforms_*.json); 'llff': a forward-facing "
                             "scene (poses_bounds.npy + images/)")
    parser.add_argument('--factor', type=int, default=8, help='llff: image downsampling factor')
    parser.add_argument('--llffhold', type=int, default=8, help='llff: hold out every N-th view for val / test')
    parser.add_argument('--no_ndc', action='store_true', help='llff: sample in world space between the bounds')
    args = parser.parse_args(argv)
    logging.basicConfig(level=logging.DEBUG if args.verbose else logging.INFO,
                        format='%(asctime)s | %(name)s | %(levelname)s | %(message)s')
    logging.info(args)

    strategy, replicas, rank = None, 1, 0
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        from keras_nerf_b200.distributed import RayShardedStrategy
        strategy = RayShardedStrategy()
        replicas, rank = strategy.num_replicas_in_sync, strategy.rank
    print('Number of devices: {}'.format(replicas))

    image_height = image_width = args.img_wh
    train_ray_chunks = None                                  # the training step's chunk: --ray_chunks
    if args.dataset_type == 'llff':
        from keras_nerf_b200.data.llff import LLFFDatasetLoader, ray_chunks_for
        loader = LLFFDatasetLoader(args.data_dir, factor=args.factor, llffhold=args.llffhold, ndc=not args.no_ndc)
        image_height, image_width = loader.H, loader.W
        logging.info(f"LLFF scene: {loader.H} x {loader.W}, focal {loader.focal:.3f}, "
                     + ("NDC rays" if loader.ndc else f"near {loader.near:.4f}, far {loader.far:.4f}")
                     + "; --img_wh, --near and --far are ignored")
        datasets = loader.load_dataset(batch_size=args.batch_size * replicas, n_sample=args.num_coarse_samples,
                                       ray_batch=args.ray_batch, rank=rank, world=replicas)
        # the render chunk must divide the views' rays and the training chunk the ray batch: chosen apart, each as
        # close to --ray_chunks as its size allows
        render_chunks, train_ray_chunks = ray_chunks_for(args.batch_size * loader.H * loader.W, args.ray_batch,
                                                         args.ray_chunks)
        logging.info(f"ray chunks: {render_chunks} to render the {loader.H} x {loader.W} views, {train_ray_chunks} "
                     f"per training chunk (--ray_chunks {args.ray_chunks})")
        args.ray_chunks = render_chunks
    else:
        loader = DatasetLoader(args.data_dir, args.white_bg)
        datasets = loader.load_dataset(batch_size=args.batch_size * replicas, image_width=args.img_wh,
                                       image_height=args.img_wh, near=args.near, far=args.far,
                                       n_sample=args.num_coarse_samples, ray_batch=args.ray_batch, rank=rank,
                                       world=replicas)
    if strategy is not None:
        # a ray-batch train split is already this rank's share
        split = 1 if args.ray_batch else 0
        for ds in datasets[split:]:
            ds._rng.seed(42)                                 # every rank walks the same shuffled order
        datasets = datasets[:split] + [ReplicaBatches(ds, strategy, args.batch_size) for ds in datasets[split:]]
    train_dataset, val_dataset, test_dataset = datasets

    last_model_path = os.path.join(args.log_dir, args.name, "model")
    model_path = last_model_path if NeRF.has_checkpoint(last_model_path) else None
    if model_path:
        logging.info("Loading the latest logged model")
    nerf = NeRF(n_coarse=args.num_coarse_samples, n_fine=args.num_fine_samples, pos_emb_xyz=args.pos_emb_xyz,
                pos_emb_dir=args.pos_emb_dir, n_layers=args.num_layers, dense_units=args.num_units,
                skip_layer=args.skip_layer, model_path=model_path, precision=args.precision, strategy=strategy,
                records=args.records)
    log_dir = os.path.join(args.log_dir, args.name)
    if strategy is not None and strategy.rank != 0:
        log_dir = os.path.join(log_dir, f"rank{strategy.rank}")   # one writer per directory
    monitor = NeRFTrainMonitor(dataset=test_dataset, log_dir=log_dir, batch_size=args.batch_size,
                               update_freq=args.log_freq, verbose=args.verbose)
    last_epoch = monitor.last_epoch
    logging.info("Last epoch: {}".format(last_epoch))
    if args.ray_batch:
        train_dataset.epoch = last_epoch                     # continue the permutation sequence, do not replay epoch 0
    nerf.compile(optimizer='adam', loss='mean_squared_error', batch_size=args.batch_size, image_width=image_width,
                 image_height=image_height, ray_chunks=args.ray_chunks, run_eagerly=args.eagerly,
                 white_background=args.white_bg, ray_batch=args.ray_batch, train_ray_chunks=train_ray_chunks,
                 fuse_chunks=None if args.fuse_chunks == 'off' else
                 ('auto' if args.fuse_chunks == 'auto' else int(args.fuse_chunks)))
    if strategy is not None:
        strategy.broadcast_parameters(nerf)
        nerf._repack()
    nerf.fit(train_dataset, epochs=args.num_epochs, validation_data=val_dataset, callbacks=[monitor],
             initial_epoch=last_epoch)
    if strategy is None or strategy.rank == 0:
        os.makedirs(args.model_dirs, exist_ok=True)
        nerf.save_model(os.path.join(args.model_dirs, args.name))
    if strategy is not None:
        strategy.barrier()
        torch.distributed.destroy_process_group()
    return nerf


if __name__ == '__main__':
    main()
