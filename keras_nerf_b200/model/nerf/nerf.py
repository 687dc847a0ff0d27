"""NeRF (reference: keras_nerf/model/nerf/nerf.py) -- same constructor / compile / train_step /
test_step / predict_and_render_images / save_model / load_model signatures, running on libknerf.

Differences that are visible to a caller (all additive):
  * tensors are torch CUDA tensors (numpy / CPU tensors are accepted as inputs);
  * `precision` ("fp32" = SIMT parity mode, "fp32_tc" = the same fp32-grade arithmetic on the tensor cores through
    3-way bf16 operand splitting, "bf16" = tcgen05 throughput mode) and `oob_mode`
    ("zero" = TF-GPU gather semantics, the parity default) constructor keywords;
  * `u_fine=` keywords expose the uniform draws the reference takes from tf.random.uniform;
  * data parallelism = one process per GPU; pass `strategy=RayShardedStrategy()` -- or just initialise
    torch.distributed with more than one rank before constructing the model, in which case a strategy is created
    automatically -- and the accumulated gradients are SUM-all-reduced over NCCL (inside libknerf,
    `knerf_train_chunk_dp`: the coarse network's gradient travels while the fine network is still in its
    backward) before Adam, which is what tf.distribute.MirroredStrategy does inside apply_gradients
    (train.py:75,110; nerf.py:455-458).
"""
from __future__ import annotations

import ctypes as C
import itertools
import json
import logging
import os

import numpy as np
import torch

from ... import _lib
from .mlp import NeRFMLP
from .utils import NeRFUtils


class Adam:
    """Keras `optimizer='adam'` defaults: lr 1e-3, beta_1 0.9, beta_2 0.999, epsilon 1e-7, no amsgrad."""

    def __init__(self, learning_rate=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7):
        self.learning_rate, self.beta_1, self.beta_2, self.epsilon = learning_rate, beta_1, beta_2, epsilon
        self.iterations = 0
        self.m = self.v = None

    def clone(self):
        return Adam(self.learning_rate, self.beta_1, self.beta_2, self.epsilon)

    def apply_flat(self, params: torch.Tensor, grads: torch.Tensor, zero_grads=True):
        if self.m is None:
            self.m, self.v = torch.zeros_like(params), torch.zeros_like(params)
        self.iterations += 1
        _lib.call("knerf_adam_step", _lib.ptr(params), _lib.ptr(grads), _lib.ptr(self.m), _lib.ptr(self.v),
                  params.numel(), float(self.learning_rate), float(self.beta_1), float(self.beta_2),
                  float(self.epsilon), self.iterations, int(zero_grads), _lib.stream())


def get_optimizer(identifier):
    if isinstance(identifier, Adam):
        return identifier.clone()
    if isinstance(identifier, str) and identifier.lower() == "adam":
        return Adam()
    if hasattr(identifier, "learning_rate"):   # duck-typed Keras-style Adam config
        g = lambda k, d: float(getattr(identifier, k, d))  # noqa: E731
        return Adam(g("learning_rate", 1e-3), g("beta_1", 0.9), g("beta_2", 0.999), g("epsilon", 1e-7))
    raise NotImplementedError(f"optimizer {identifier!r}: only Adam is implemented (the reference scripts use 'adam')")


class Mean:
    """tf.keras.metrics.Mean stand-in (nerf.py:167-173)."""

    def __init__(self, name=None):
        self.name, self.total, self.count = name, 0.0, 0

    def update_state(self, values):
        v = torch.as_tensor(values, dtype=torch.float32).reshape(-1)
        self.total += float(v.sum())
        self.count += int(v.numel())

    def result(self):
        return self.total / max(self.count, 1)

    def reset_state(self):
        self.total, self.count = 0.0, 0

    reset_states = reset_state


def image_metrics(a: torch.Tensor, b: torch.Tensor, max_val: float = 1.0):
    """(tf.image.psnr(a, b, max_val), tf.image.ssim(a, b, max_val)) per image (nerf.py:309-312) as one [2, B] CUDA
    tensor, from `knerf_image_metrics` (per-image MSE and 11x11-gaussian-window SSIM in one pass).
    Images smaller than the SSIM window give NaN SSIM (TF raises there)."""
    a, b = a.contiguous(), b.contiguous()
    B, H, W, Cn = a.shape
    out = torch.full((2, B), float("nan"), dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device):
        if H >= 11 and W >= 11:
            n = _lib.load().knerf_image_metrics_workspace_floats(B, H, W, Cn)
            ws = torch.empty(n, dtype=torch.float32, device=a.device)
            _lib.call("knerf_image_metrics", _lib.ptr(a), _lib.ptr(b), B, H, W, Cn, float(max_val), _lib.ptr(out[0]),
                      _lib.ptr(out[1]), _lib.ptr(ws), n, _lib.stream())
        else:
            for i in range(B):
                _lib.call("knerf_mse", _lib.ptr(a[i]), _lib.ptr(b[i]), a[i].numel(), out[0, i:i + 1].data_ptr(),
                          _lib.stream())
    out[0] = 20.0 * float(np.log10(max_val)) - 10.0 * torch.log10(out[0])
    return out


_seed_counter = _lib.seed_stream(0xC0A45E00)      # fine-sample draws of calls that pass neither `u_fine` nor `seed`


class NeRF:
    def __init__(self, n_coarse: int = 64, n_fine: int = 128, pos_emb_xyz: int = 10, pos_emb_dir: int = 4,
                 n_layers: int = 8, dense_units: int = 256, skip_layer=4, model_path: str = None,
                 precision: str = "fp32", oob_mode: str = "zero", scan_mode: str = None, device=None,
                 strategy=None, reproducible: bool = False, records: str = "fp8", **kwargs):
        # keras_nerf/model/nerf/nerf.py:11-43
        self.model_path = model_path
        if self.model_path is None:
            self.n_coarse, self.n_fine = n_coarse, n_fine
            self.pos_emb_xyz, self.pos_emb_dir = pos_emb_xyz, pos_emb_dir
            self.n_layers, self.dense_units, self.skip_layer = n_layers, dense_units, skip_layer
        else:
            self.load_model(model_path)
        if precision not in _lib.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_lib.PRECISIONS)}")
        self.precision = precision
        self.oob_mode = oob_mode
        # fp32 parity mode sums the pdf/cdf in TF-CPU order (bit-identical cdf); bf16 mode uses the warp scan
        self.scan_mode = scan_mode or ("warp" if precision in ("bf16", "bfloat16") else "sequential")
        self.device = torch.device(device) if device is not None else None
        if strategy is None and torch.distributed.is_available() and torch.distributed.is_initialized() \
                and torch.distributed.get_world_size() > 1:
            from ...distributed import RayShardedStrategy
            strategy = RayShardedStrategy(device=self.device)        # replicas must not train unsynchronised
        self.strategy = strategy
        # bf16 inference: the forward kernel's two MMA-issuing threads interleave freely by default (last-bit
        # run-to-run differences, which the out-of-range gather quirk of the fine sampler can amplify in single
        # pixels); reproducible=True makes them hand over in order like the training kernels (-14 % throughput).
        # A per-call option of the library (KNERF_TC_ORDERED), i.e. per model: other models are unaffected.
        self.reproducible = bool(reproducible)
        # bf16 training: storage format of the records the forward / dgrad kernels save for the weight-gradient GEMMs.
        # "fp8" (KNERF_REC_FP8: e4m3 activations, e5m2 gradients under one power-of-two scale per call) halves the
        # step's HBM traffic; forward outputs and the dgrad chain are the same bits either way, the weight gradients
        # differ by 0.3-0.7 % (relative L2 at 98k samples) and training converges alike (profiles/r02_fp8_records.md).
        # "bf16" keeps round 1's records.
        if records not in ("bf16", "fp8"):
            raise ValueError("records must be 'bf16' or 'fp8'")
        self.records = records
        self.coarse = NeRFMLP(n_layers=self.n_layers, dense_units=self.dense_units, skip_layer=self.skip_layer,
                              name='coarse_nerf', device=device)
        self.fine = NeRFMLP(n_layers=self.n_layers, dense_units=self.dense_units, skip_layer=self.skip_layer,
                            name='fine_nerf', device=device)
        self.epsilon = 1e-10
        self.run_eagerly = False
        self._compiled = False

    # ---- checkpoint (nerf.py:45-76) -----------------------------------------------------------
    def save_model(self, path, weights_only=False):
        model_config = {'n_coarse': self.n_coarse, 'n_fine': self.n_fine, 'pos_emb_xyz': self.pos_emb_xyz,
                        'pos_emb_dir': self.pos_emb_dir, 'n_layers': self.n_layers,
                        'dense_units': self.dense_units, 'skip_layer': self.skip_layer}
        os.makedirs(path, exist_ok=True)
        if not weights_only:
            with open(os.path.join(path, 'model_config.json'), 'w') as f:
                json.dump(model_config, f)
        self.coarse.save_weights(os.path.join(path, 'coarse.h5'))
        self.fine.save_weights(os.path.join(path, 'fine.h5'))

    @staticmethod
    def has_checkpoint(path) -> bool:
        """the existence check of the scripts (train_single.py:91-92, inference.py:51-54): `coarse.h5` + `fine.h5`
        in Keras' legacy HDF5 weight layout (utils/hdf5.py); `.npz` archives of an early version are still found"""
        return all(any(os.path.exists(os.path.join(path, n + ext)) for ext in ('.npz', '.h5'))
                   for n in ('coarse', 'fine'))

    def load_model(self, path):
        with open(os.path.join(path, 'model_config.json'), 'r') as f:
            mc = json.load(f)
        self.n_coarse, self.n_fine = mc['n_coarse'], mc['n_fine']
        self.pos_emb_xyz, self.pos_emb_dir = mc['pos_emb_xyz'], mc['pos_emb_dir']
        self.n_layers, self.dense_units, self.skip_layer = mc['n_layers'], mc['dense_units'], mc['skip_layer']

    # ---- compile (nerf.py:78-173) -------------------------------------------------------------
    def compile(self, optimizer, loss, batch_size, image_height, image_width, ray_chunks, white_background=False,
                is_training=True, **kwargs):
        """nerf.py:78-173.  Keyword extensions: `fuse_chunks` (below) and `ray_batch`.

        ray_batch=N > 0: the training step takes N rays drawn across all views (data.loader.RayBatchDataset), so
        train_step((targets[N,3], (o[N,3], d[N,3], t[N,Nc]))) / accumulate_gradients take a flat ray batch, while
        batch_size / image_height / image_width keep describing what predict_and_render_images, test_step and the
        monitor render.  `ray_chunks` must divide N (checked like it is against the number of rays of an image batch)
        and `fuse_chunks` applies to the N rays.  The logs keep their keys: the PSNR is that of the batch MSE and the
        SSIM is NaN (a ray batch has no 11x11 window)."""
        self.run_eagerly = bool(kwargs.get("run_eagerly", False))
        self.optimizer, self.loss = optimizer, loss
        # The fused kernels implement the loss of the reference scripts: MeanSquaredError (train_single.py:127) or
        # train.py:130-136's `compute_distributed_loss` wrapper around it (accepted by name, or by the explicit
        # `knerf_loss = "mse"` attribute on a callable).  Anything else would be silently replaced: refuse it.
        lname = (loss if isinstance(loss, str) else
                 getattr(loss, "knerf_loss", None) or getattr(loss, "name", None) or getattr(loss, "__name__", None)
                 or type(loss).__name__).lower()
        if not any(k in lname for k in ("mean_squared", "meansquared", "mse", "compute_distributed_loss")):
            raise NotImplementedError(f"loss {loss!r}: only the mean-squared-error loss of the reference scripts is "
                                      "implemented (tag an equivalent callable with `knerf_loss = 'mse'`)")
        self.batch_size, self.image_height, self.image_width = batch_size, image_height, image_width
        self.white_background = white_background
        self.ray_chunks = ray_chunks
        self.num_rays = batch_size * image_height * image_width
        if self.ray_chunks >= self.num_rays:
            self.ray_chunks = self.num_rays                                        # nerf.py:95-98
        assert self.num_rays % self.ray_chunks == 0, \
            f'ray_chunks {self.ray_chunks} must be a divisor of the number of rays {self.num_rays}'   # nerf.py:100
        self.sequential_chunks = self.num_rays // self.ray_chunks
        self.ray_batch = int(kwargs.get("ray_batch", 0) or 0)
        if self.ray_batch:
            # the training step's own chunking; rendering keeps the chunks of the image batch
            self._train_rays = self.ray_batch
            train_rc = min(ray_chunks, self.ray_batch)
            assert self.ray_batch % train_rc == 0, \
                f'ray_chunks {train_rc} must be a divisor of the number of rays {self.ray_batch}'
        else:
            self._train_rays, train_rc = self.num_rays, self.ray_chunks
        # `ray_chunks` exists in the reference to bound TensorFlow's activation memory (train.py:46, 1024 by default); the
        # chunks of a step are independent and their gradients are summed, so executing k of them in one call gives the
        # same step (up to the fp32 summation order; with random fine-sample draws, other draws of the same
        # distribution) with fewer, larger launches -- 0.82 -> 1.22 M rays/s on a 160,000-ray step between 1,000- and
        # 32,000-ray calls.  Off unless asked for: fuse_chunks="auto" (calls of up to 32,768 rays) or an int k.
        fuse = kwargs.get("fuse_chunks", None)
        k, nch = 1, self._train_rays // train_rc
        if fuse in ("auto", True):
            k = max(j for j in range(1, nch + 1) if nch % j == 0 and (j == 1 or j * train_rc <= 32768))
        elif isinstance(fuse, int) and not isinstance(fuse, bool) and fuse > 1:
            k = max(j for j in range(1, min(fuse, nch) + 1) if nch % j == 0)
        self._train_ray_chunks, self._train_chunks = train_rc * k, nch // k
        self.device = self.device or _lib.default_device()
        self.nerf_utils = NeRFUtils(self.batch_size, self.image_height, self.image_width, self.ray_chunks,
                                    self.pos_emb_xyz, self.pos_emb_dir, self.white_background, device=self.device,
                                    oob_mode=self.oob_mode, scan_mode=self.scan_mode)
        self._build_model()
        self.is_training = bool(is_training)
        self._alloc_workspace()
        if is_training:
            self._initialize_training_accumulator()
            self._initialize_optimizer_and_metrics(optimizer)
        self._compiled = True

    def _build_model(self):
        # nerf.py:116-136 (weights created on first compile; optional load from model_path)
        dx, dd = 3 + 6 * self.pos_emb_xyz, 3 + 6 * self.pos_emb_dir
        for net in (self.coarse, self.fine):
            if not net.built:
                net.device = self.device
                net.build(dx, dd, self.pos_emb_xyz, self.pos_emb_dir, self.n_coarse, self.n_fine)
        self.cfg = self.coarse.cfg
        if self.model_path is not None:
            self.coarse.load_weights(os.path.join(self.model_path, 'coarse.h5'))
            self.fine.load_weights(os.path.join(self.model_path, 'fine.h5'))
        self._packed = {}
        self._prec = _lib.PRECISIONS[self.precision]
        if self._prec == _lib.BF16:
            lib = _lib.load()
            nbytes = lib.knerf_packed_weight_bytes(C.byref(self.cfg))
            if nbytes <= 0:
                # the fused bf16 chain kernels take models of --num_units <= 256, up to eight layers with at most one skip
                # concat (not into the heads), --pos_emb_xyz <= 10 and --pos_emb_dir <= 4 (csrc/api.cu tc_chain_map); any
                # other shape the reference's CLI accepts (wider, more layers / skips / frequencies) runs in the fp32_tc mode -- per-layer tcgen05 GEMMs for every layer whose width is a multiple of 64,
                # SIMT FFMA for the others -- and says so
                logging.warning("precision='bf16' is not available for this model shape (%s); using precision="
                                "'fp32_tc' (fp32-grade per-layer tensor-core GEMMs)",
                                lib.knerf_last_error().decode() or "unsupported configuration")
                self.precision, self._prec = "fp32_tc", _lib.FP32_TC
        self._prec_flags = self._prec | (_lib.TC_ORDERED if self.reproducible else 0)
        if self._prec == _lib.BF16 and self.records == "fp8":
            self._prec_flags |= _lib.REC_FP8
        self._prec_train = self._prec | (self._prec_flags & _lib.REC_FP8)      # (tests drive the kernels one by one)
        if self._prec == _lib.BF16:
            for name in ("coarse", "fine"):
                self._packed[name] = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            self._repack()

    def _repack(self):
        if self._prec != _lib.BF16:
            return
        with torch.cuda.device(self.device):
            for name, net in (("coarse", self.coarse), ("fine", self.fine)):
                _lib.call("knerf_pack_weights", C.byref(self.cfg), _lib.ptr(net.params),
                          self._packed[name].data_ptr(), _lib.stream())

    def _packed_ptr(self, name):
        return self._packed[name].data_ptr() if name in self._packed else None

    def _alloc_workspace(self):
        lib = _lib.load()
        rows = (self._train_ray_chunks if self.is_training else self.ray_chunks) * (self.n_coarse + self.n_fine)
        need = lib.knerf_workspace_bytes(C.byref(self.cfg), rows, self._prec_train, int(self.is_training))
        if self.ray_batch and self.is_training and need >= 0:
            # the training chunk of a ray batch can be smaller than the render chunk
            render = lib.knerf_workspace_bytes(C.byref(self.cfg), self.ray_chunks * (self.n_coarse + self.n_fine),
                                               self._prec_train, 0)
            need = max(need, render) if render >= 0 else render
        if need < 0:
            raise _lib.KnerfError("knerf_workspace_bytes: " + lib.knerf_last_error().decode())
        self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)

    def _initialize_training_accumulator(self):
        # nerf.py:138-161: one accumulator per trainable variable == one flat buffer per net here
        n = self.coarse.params.numel()
        self._grad_flat = torch.zeros(2 * n, dtype=torch.float32, device=self.device)   # one all-reduce buffer
        self.coarse_gradients_accumulator = self._grad_flat[:n]
        self.fine_gradients_accumulator = self._grad_flat[n:]
        self._losses = torch.zeros(2, dtype=torch.float32, device=self.device)

    def _initialize_optimizer_and_metrics(self, optimizer):
        # nerf.py:163-173
        self.coarse_optimizer = get_optimizer(optimizer)
        self.fine_optimizer = get_optimizer(optimizer)
        self.coarse_loss_tracker = Mean(name="coarse_loss")
        self.coarse_psnr_metric = Mean(name="coarse_psnr")
        self.corase_ssim_metric = Mean(name="coarse_ssim")
        self.fine_loss_tracker = Mean(name="fine_loss")
        self.fine_psnr_metric = Mean(name="fine_psnr")
        self.fine_ssim_metric = Mean(name="fine_ssim")

    # ---- helpers ------------------------------------------------------------------------------
    def _flat_rays(self, rays, n=None):
        o, d, t = (_lib.dev(r, self.device) for r in rays)
        n = self.num_rays if n is None else n
        return o.reshape(n, 3), d.reshape(n, 3), t.reshape(n, self.n_coarse)

    def _u(self, u_fine, n):
        if u_fine is None:
            return None
        return _lib.dev(u_fine, self.device).reshape(n, self.n_fine)

    def _sampler_flags(self):
        return ((_lib.OOB_CLAMP if self.oob_mode == "clamp" else _lib.OOB_ZERO)
                | (_lib.SCAN_SEQUENTIAL if self.scan_mode == "sequential" else 0))

    # ---- rendering (nerf.py:175-304) ----------------------------------------------------------
    def _render_rays(self, o, d, t, u_fine, seed, outs_c, outs_f, t_sorted=None):
        R = o.shape[0]
        with torch.cuda.device(self.device):
            _lib.call("knerf_render_chunk", C.byref(self.cfg), _lib.ptr(self.coarse.params), _lib.ptr(self.fine.params),
                      self._packed_ptr("coarse"), self._packed_ptr("fine"), _lib.ptr(o), _lib.ptr(d), _lib.ptr(t), R,
                      _lib.ptr(u_fine), int(seed), int(bool(self.white_background)),
                      self._sampler_flags(), self._prec_flags,
                      _lib.ptr(outs_c[0]), _lib.ptr(outs_c[1]), _lib.ptr(outs_c[2]),
                      _lib.ptr(outs_f[0]), _lib.ptr(outs_f[1]), _lib.ptr(outs_f[2]), _lib.ptr(t_sorted),
                      self._ws.data_ptr(), self._ws.numel(), _lib.stream())

    def predict_and_render_chunk(self, ray_chunks, u_fine=None, seed=None):
        """nerf.py:218-227: (o[R,3], d[R,3], t[R,Nc]) -> (coarse dict, fine dict)."""
        o, d, t = (_lib.dev(r, self.device) for r in ray_chunks)
        R = o.shape[0]
        assert R <= self.ray_chunks, f"chunk of {R} rays exceeds compiled ray_chunks {self.ray_chunks}"
        S = self.n_coarse + self.n_fine
        mk = lambda *s: torch.empty(s, dtype=torch.float32, device=self.device)  # noqa: E731
        oc, of = (mk(R, 3), mk(R), mk(R, self.n_coarse)), (mk(R, 3), mk(R), mk(R, S))
        u = None if u_fine is None else _lib.dev(u_fine, self.device).reshape(R, self.n_fine)
        self._render_rays(o, d, t, u, next(_seed_counter) if seed is None else seed, oc, of)
        return ({'image': oc[0], 'depth': oc[1], 'weights': oc[2]}, {'image': of[0], 'depth': of[1], 'weights': of[2]})

    def predict_and_render_images(self, rays, u_fine=None, seed=None):
        """nerf.py:229-304: rays = (o[B,H,W,3], d[B,H,W,3], t[B,H,W,Nc]) -> (coarse, fine) dicts of
        image[B,H,W,3], depth[B,H,W], weights[B,H,W,S]."""
        o, d, t = self._flat_rays(rays)
        n, S = self.num_rays, self.n_coarse + self.n_fine
        u = self._u(u_fine, n)
        mk = lambda *s: torch.empty(s, dtype=torch.float32, device=self.device)  # noqa: E731
        ci, cd, cw = mk(n, 3), mk(n), mk(n, self.n_coarse)
        fi, fd, fw = mk(n, 3), mk(n), mk(n, S)
        seed = next(_seed_counter) if seed is None else seed
        rc = self.ray_chunks
        for i in range(self.sequential_chunks):                                   # nerf.py:251
            s = slice(i * rc, (i + 1) * rc)
            # Philox counters are per element of the chunk: give every chunk its own stream
            self._render_rays(o[s], d[s], t[s], None if u is None else u[s], seed + i * 0x9E3779B1,
                              (ci[s], cd[s], cw[s]), (fi[s], fd[s], fw[s]))
        B, H, W = self.batch_size, self.image_height, self.image_width
        coarse = {'image': ci.view(B, H, W, 3), 'depth': cd.view(B, H, W), 'weights': cw.view(B, H, W, self.n_coarse)}
        fine = {'image': fi.view(B, H, W, 3), 'depth': fd.view(B, H, W), 'weights': fw.view(B, H, W, S)}
        return coarse, fine

    def predict_and_render_images_sharded(self, rays, u_fine=None, seed=None, with_weights=False):
        """Multi-GPU form of predict_and_render_images (SURVEY §8e: "rendering just gathers pixels"): every rank
        holds the same rays, renders a contiguous run of whole ray chunks and the pixels (rgb 12 B + depth 4 B per
        ray; the [.., S] compositing weights only on request) are all-gathered, so every rank returns the full
        images.  Same chunk seeds as the single-GPU call: the result does not depend on the number of ranks."""
        st = self.strategy
        if st is None or st.num_replicas_in_sync == 1:
            return self.predict_and_render_images(rays, u_fine=u_fine, seed=seed)
        o, d, t = self._flat_rays(rays)
        n, S, rc = self.num_rays, self.n_coarse + self.n_fine, self.ray_chunks
        u = self._u(u_fine, n)
        lo, hi = st.shard_bounds(self.sequential_chunks)
        m = (hi - lo) * rc
        mk = lambda *s_: torch.empty(s_, dtype=torch.float32, device=self.device)  # noqa: E731
        ci, cd, cw = mk(m, 3), mk(m), mk(m, self.n_coarse)
        fi, fd, fw = mk(m, 3), mk(m), mk(m, S)
        seed = next(_seed_counter) if seed is None else seed
        for i in range(lo, hi):
            s = slice(i * rc, (i + 1) * rc)
            l = slice((i - lo) * rc, (i - lo + 1) * rc)
            self._render_rays(o[s], d[s], t[s], None if u is None else u[s], seed + i * 0x9E3779B1,
                              (ci[l], cd[l], cw[l]), (fi[l], fd[l], fw[l]))
        sizes = [(b - a) * rc for a, b in (st.shard_bounds_of(r, self.sequential_chunks)
                                           for r in range(st.num_replicas_in_sync))]
        # one collective: [rgb_c, depth_c, rgb_f, depth_f] = 8 floats per ray
        packed = torch.cat([ci, cd[:, None], fi, fd[:, None]], dim=1)
        full = st.gather_rows(packed, n, 0, sizes=sizes)
        B, H, W = self.batch_size, self.image_height, self.image_width
        coarse = {'image': full[:, 0:3].reshape(B, H, W, 3), 'depth': full[:, 3].reshape(B, H, W)}
        fine = {'image': full[:, 4:7].reshape(B, H, W, 3), 'depth': full[:, 7].reshape(B, H, W)}
        if with_weights:
            coarse['weights'] = st.gather_rows(cw, n, 0, sizes=sizes).reshape(B, H, W, self.n_coarse)
            fine['weights'] = st.gather_rows(fw, n, 0, sizes=sizes).reshape(B, H, W, S)
        return coarse, fine

    # ---- mesh export (no counterpart in the reference) ------------------------------------------
    def _network(self, network):
        if not self._compiled:
            raise RuntimeError("compile() the model first (the bf16 mode needs its packed weights)")
        if network not in ("coarse", "fine"):
            raise ValueError(f"network must be 'coarse' or 'fine', got {network!r}")
        return (self.coarse if network == "coarse" else self.fine).params, self._packed_ptr(network)

    def _query_rows(self, rows_wanted, S):
        """rays per knerf_mlp_forward call: up to 2^22 samples, halved while the scratch exceeds 1 GiB (the fp32 modes
        keep whole activation rows), at least one ray; -> (rays, workspace)"""
        lib = _lib.load()
        samples = 1 << 22
        while samples > S and lib.knerf_workspace_bytes(C.byref(self.cfg), samples, self._prec_flags, 0) > (1 << 30):
            samples //= 2
        R = max(1, min(rows_wanted, samples // S))
        need = lib.knerf_workspace_bytes(C.byref(self.cfg), R * S, self._prec_flags, 0)
        if need < 0:
            raise _lib.KnerfError("knerf_workspace_bytes: " + lib.knerf_last_error().decode())
        return R, torch.empty(need, dtype=torch.uint8, device=self.device)

    def _forward(self, params, packed, o, d, t, S, out, ws):
        _lib.call("knerf_mlp_forward", C.byref(self.cfg), _lib.ptr(params), packed, _lib.ptr(o), _lib.ptr(d),
                  _lib.ptr(t), o.shape[0], S, self._prec_flags, 0, _lib.ptr(out), ws.data_ptr(), ws.numel(),
                  _lib.stream())

    @staticmethod
    def _grid_frame(resolution, bound):
        """(n[3], origin[3], spacing[3]) of the lattice: `bound` a scalar b (the cube [-b, b]^3) or (min[3], max[3]);
        `resolution` an int or three; point i of axis a at origin[a] + spacing[a] * i (fp32)"""
        n = np.broadcast_to(np.asarray(resolution, dtype=np.int64), (3,)).copy()
        if (n < 2).any():
            raise ValueError(f"resolution must be >= 2 per axis, got {resolution!r}")
        if np.ndim(bound) == 0:
            lo, hi = np.full(3, -float(bound), np.float32), np.full(3, float(bound), np.float32)
        else:
            lo, hi = (np.broadcast_to(np.asarray(b, dtype=np.float32), (3,)).copy() for b in bound)
        if not (np.isfinite(lo).all() and np.isfinite(hi).all() and (hi > lo).all()):
            raise ValueError(f"bound must be finite with min < max per axis, got {bound!r}")
        spacing = ((hi - lo) / (n - 1).astype(np.float32)).astype(np.float32)
        return n, lo, spacing

    def density_grid(self, resolution=256, bound=1.5, network="fine", samples_per_call=None):
        """sigma of `network` on a regular lattice -> CUDA tensor [nx, ny, nz] (x slowest, z fastest).  The lattice is
        evaluated as rays along +z through the fused forward in the model's precision: one ray per (x, y) column,
        origin (x_i, y_j, z_0), direction (0, 0, 1), depths k * spacing_z.  The direction does not change sigma.
        `samples_per_call` (default: up to 2^22 within 1 GiB of scratch) only bounds memory; it does not change a bit."""
        params, packed = self._network(network)
        n, lo, spacing = self._grid_frame(resolution, bound)
        nx, ny, nz = (int(v) for v in n)
        dev = self.device
        f32 = lambda a: torch.as_tensor(a, dtype=torch.float32, device=dev)  # noqa: E731
        axis = lambda a: f32(lo[a]) + torch.arange(int(n[a]), dtype=torch.float32, device=dev) * f32(spacing[a])  # noqa
        xs, ys = axis(0), axis(1)
        tz = torch.arange(nz, dtype=torch.float32, device=dev) * f32(spacing[2])
        cols = nx * ny
        R, ws = self._query_rows(cols, nz)
        if samples_per_call is not None:
            R = max(1, min(R, int(samples_per_call) // nz))
        grid = torch.empty((nx, ny, nz), dtype=torch.float32, device=dev)
        flat = grid.view(cols, nz)
        d_all = torch.zeros((R, 3), dtype=torch.float32, device=dev)
        d_all[:, 2] = 1.0
        t_all = tz.expand(R, nz).contiguous()
        out = torch.empty((R, nz, 4), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            for s in range(0, cols, R):
                e = min(cols, s + R)
                c = torch.arange(s, e, device=dev)
                o = torch.stack([xs[c // ny], ys[c % ny], torch.full((e - s,), float(lo[2]), device=dev)], -1)
                self._forward(params, packed, o, d_all[:e - s], t_all[:e - s], nz, out, ws)
                flat[s:e] = out[:e - s, :, 3]
        return grid

    def vertex_colors(self, vertices, normals, network="fine"):
        """rgb of `network` at every vertex, looking at the surface along its normal: o = v, d = -n (a zero normal
        looks along -z), one sample at t = 0 -> CUDA tensor [V, 3]"""
        params, packed = self._network(network)
        v = _lib.dev(vertices, self.device).reshape(-1, 3)
        d = -_lib.dev(normals, self.device).reshape(-1, 3)
        d[(d == 0).all(-1)] = torch.tensor([0.0, 0.0, -1.0], device=self.device)
        V = v.shape[0]
        rgb = torch.empty((V, 3), dtype=torch.float32, device=self.device)
        if V == 0:
            return rgb
        R, ws = self._query_rows(V, 1)
        t = torch.zeros((R, 1), dtype=torch.float32, device=self.device)
        out = torch.empty((R, 1, 4), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            for s in range(0, V, R):
                e = min(V, s + R)
                self._forward(params, packed, v[s:e], d[s:e].contiguous(), t[:e - s], 1, out, ws)
                rgb[s:e] = out[:e - s, 0, :3]
        return rgb

    def extract_mesh(self, resolution=256, threshold=50.0, bound=1.5, network="fine", colors=True, close=True):
        """Triangle mesh of the level set sigma = `threshold` of `network` on a `resolution` lattice over `bound` (see
        density_grid), by marching tetrahedra (utils/mesh.py).  close=True pads the grid with one layer of zeros, so a
        surface that leaves the box is capped on its faces and the mesh stays closed.  Returns a dict of CUDA tensors:
        vertices [V,3], normals [V,3] (outward: towards decreasing sigma), colors [V,3] (or None), faces [T,3] int32,
        and `seconds`: wall time of each stage (grid, isosurface, colors), each ended by a device synchronise."""
        import time
        from ...utils.mesh import marching_tetrahedra
        t0 = time.perf_counter()
        grid = self.density_grid(resolution, bound, network)
        _, origin, spacing = self._grid_frame(resolution, bound)
        if close:
            grid = torch.nn.functional.pad(grid[None], (1, 1, 1, 1, 1, 1))[0]
            origin = (origin - spacing).astype(np.float32)
        torch.cuda.synchronize(self.device)
        t1 = time.perf_counter()
        v, n, f = marching_tetrahedra(grid, threshold, origin, spacing)
        torch.cuda.synchronize(self.device)
        t2 = time.perf_counter()
        rgb = self.vertex_colors(v, n, network) if colors else None
        torch.cuda.synchronize(self.device)
        t3 = time.perf_counter()
        return {"vertices": v, "normals": n, "colors": rgb, "faces": f,
                "seconds": {"grid": t1 - t0, "isosurface": t2 - t1, "colors": t3 - t2}}

    # ---- metrics (nerf.py:306-330) ------------------------------------------------------------
    def update_and_return_metrics(self, images, coarse_images, fine_images, coarse_loss, fine_loss):
        """coarse_loss / fine_loss: floats, or ONE device tensor [2] (then `fine_loss` is None) that is read back
        together with the PSNR / SSIM values in a single device -> host copy"""
        mc = image_metrics(images, coarse_images)
        mf = image_metrics(images, fine_images)
        if torch.is_tensor(coarse_loss) and fine_loss is None:
            flat = torch.cat([torch.stack([mc, mf]).reshape(-1), coarse_loss.reshape(-1)]).cpu()   # the step's only sync
            vals, (coarse_loss, fine_loss) = flat[:-2].reshape(2, 2, -1), flat[-2:].tolist()
        else:
            vals = torch.stack([mc, mf]).cpu()                                    # one device -> host read
        self.coarse_loss_tracker.update_state(float(coarse_loss))
        self.coarse_psnr_metric.update_state(vals[0, 0])
        self.corase_ssim_metric.update_state(vals[0, 1])
        self.fine_loss_tracker.update_state(float(fine_loss))
        self.fine_psnr_metric.update_state(vals[1, 0])
        self.fine_ssim_metric.update_state(vals[1, 1])
        return {m.name: m.result() for m in self.metrics}

    # ---- training (nerf.py:332-473) -----------------------------------------------------------
    def accumulate_gradients(self, images, rays, u_fine=None, seed=None, want_images=True, reduce=True):
        """The chunk loop of train_step (nerf.py:351-421): fills the two gradient accumulators and the loss
        accumulators; returns (coarse_images, fine_images) [B,H,W,3] (or None).  With a multi-rank strategy and
        reduce=True the accumulators hold the cross-replica SUM when the enqueued work completes.  Compiled with
        `ray_batch`: images are targets [N,3] of a flat ray batch and the returned images are [N,3]."""
        images = _lib.dev(images, self.device)[..., :3]                           # nerf.py:335
        n = self._train_rays
        target = images.reshape(n, 3).contiguous()
        o, d, t = self._flat_rays(rays, n)
        u = self._u(u_fine, n)
        ci = torch.empty((n, 3), dtype=torch.float32, device=self.device) if want_images else None
        fi = torch.empty((n, 3), dtype=torch.float32, device=self.device) if want_images else None
        seed = next(_seed_counter) if seed is None else seed
        rc, nch = self._train_ray_chunks, self._train_chunks      # (= ray_chunks, sequential_chunks unless fuse_chunks)
        oob = self._sampler_flags()
        # data parallel: the all-reduce rides inside the LAST chunk's call (coarse half behind the coarse backward)
        if getattr(self, "_grads_reduced", False):
            # the accumulators already hold a cross-replica SUM: adding local gradients to it and reducing again
            # would count the other replicas' share twice
            raise RuntimeError("the accumulated gradients have been all-reduced: call apply_gradients() before the next "
                               "accumulate_gradients(), or pass reduce=False to accumulate several batches first")
        comm, comm_stream = (None, None) if self.strategy is None or not reduce else self.strategy.knerf_comm()
        self._grads_reduced = comm is not None
        with torch.cuda.device(self.device):
            for i in range(nch):
                s = slice(i * rc, (i + 1) * rc)
                _lib.call("knerf_train_chunk_dp", C.byref(self.cfg), _lib.ptr(self.coarse.params),
                          _lib.ptr(self.fine.params), self._packed_ptr("coarse"), self._packed_ptr("fine"),
                          _lib.ptr(o[s]), _lib.ptr(d[s]), _lib.ptr(t[s]), _lib.ptr(target[s]), rc,
                          None if u is None else _lib.ptr(u[s]), int(seed + i * 0x9E3779B1) & 0x7FFFFFFFFFFFFFFF,
                          int(bool(self.white_background)), oob, self._prec_flags, 1.0 / nch,
                          _lib.ptr(self.coarse_gradients_accumulator), _lib.ptr(self.fine_gradients_accumulator),
                          _lib.ptr(self._losses), None if ci is None else _lib.ptr(ci[s]),
                          None if fi is None else _lib.ptr(fi[s]), self._ws.data_ptr(), self._ws.numel(),
                          _lib.stream(), comm, comm_stream, int(comm is not None and i == nch - 1))
        B, H, W = self.batch_size, self.image_height, self.image_width
        if not want_images:
            return None, None
        if self.ray_batch:
            return ci, fi
        return ci.view(B, H, W, 3), fi.view(B, H, W, 3)

    def apply_gradients(self):
        """nerf.py:455-471: cross-replica SUM (MirroredStrategy semantics), two Adam steps, zero accumulators."""
        if self.strategy is not None and not getattr(self, "_grads_reduced", False):
            self.strategy.all_reduce_sum(self.coarse_gradients_accumulator, self.fine_gradients_accumulator)
        self._grads_reduced = False
        with torch.cuda.device(self.device):
            self.coarse_optimizer.apply_flat(self.coarse.params, self.coarse_gradients_accumulator, zero_grads=True)
            self.fine_optimizer.apply_flat(self.fine.params, self.fine_gradients_accumulator, zero_grads=True)
        self._repack()

    def train_step(self, inputs, u_fine=None, seed=None):
        images, rays = inputs
        ci, fi = self.accumulate_gradients(images, rays, u_fine=u_fine, seed=seed)
        losses = self._losses.clone()
        self._losses.zero_()                                                      # nerf.py:465-466
        if self.run_eagerly or os.environ.get("KNERF_ASSERT_FINITE"):
            # tf.debugging.assert_all_finite on every gradient (nerf.py:381-382,410-411): one host sync
            for name, g in (("Coarse", self.coarse_gradients_accumulator), ("Fine", self.fine_gradients_accumulator)):
                if not bool(torch.isfinite(g).all()):
                    raise FloatingPointError(f"{name} Gradient is not finite")
        if self.run_eagerly:
            # nerf.py:429-451 (eager-only diagnostics): a network whose gradient is identically zero has stopped
            # learning -- typically a dead sigma head
            nz_c = int(torch.count_nonzero(self.coarse_gradients_accumulator))
            nz_f = int(torch.count_nonzero(self.fine_gradients_accumulator))
            if nz_c == 0 and nz_f == 0:
                logging.error('Both Coarse and Fine Gradient are zero')
            elif nz_c == 0:
                logging.warning('Coarse Gradient is zero')
            elif nz_f == 0:
                logging.warning('Fine Gradient is zero')
        self.apply_gradients()
        imgs = _lib.dev(images, self.device)[..., :3]
        if self.ray_batch:      # one [1, 1, N] "image": the PSNR of the batch MSE, no SSIM window
            imgs, ci, fi = (x.reshape(1, 1, self.ray_batch, 3) for x in (imgs, ci, fi))
        return self.update_and_return_metrics(imgs, ci, fi, losses, None)   # losses + metrics: one host read

    def test_step(self, inputs, u_fine=None, seed=None):
        # nerf.py:475-497
        images, rays = inputs
        images = _lib.dev(images, self.device)[..., :3].contiguous()
        coarse, fine = self.predict_and_render_images(rays, u_fine=u_fine, seed=seed)
        out = torch.empty(2, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            for k, res in enumerate((coarse, fine)):
                _lib.call("knerf_mse", _lib.ptr(images), _lib.ptr(res['image'].contiguous()), images.numel(),
                          out[k:k + 1].data_ptr(), _lib.stream())
        lc, lf = out.tolist()
        return self.update_and_return_metrics(images, coarse['image'], fine['image'], lc, lf)

    @property
    def metrics(self):
        # nerf.py:499-508
        return [self.coarse_loss_tracker, self.coarse_psnr_metric, self.corase_ssim_metric,
                self.fine_loss_tracker, self.fine_psnr_metric, self.fine_ssim_metric]

    # ---- a thin Keras-style fit loop (train.py:151-157, train_single.py:137-143) ---------------
    def fit(self, dataset, epochs=1, validation_data=None, callbacks=None, initial_epoch=0, verbose=1):
        global _seed_counter
        if initial_epoch:       # a resumed run continues the draw sequence instead of replaying epoch 0's
            _seed_counter = _lib.seed_stream(0xC0A45E00, advance=int(initial_epoch))
        callbacks = list(callbacks or [])
        for cb in callbacks:
            if hasattr(cb, "set_model"):
                cb.set_model(self)
            else:
                cb.model = self
        history = {}
        for epoch in range(initial_epoch, epochs):
            for m in self.metrics:
                m.reset_state()
            logs = {}
            for step, batch in enumerate(dataset):
                logs = self.train_step(batch)
                for cb in callbacks:
                    if hasattr(cb, "on_train_batch_end"):
                        cb.on_train_batch_end(step, logs)
            if validation_data is not None:
                for m in self.metrics:
                    m.reset_state()
                vlogs = {}
                for batch in validation_data:
                    vlogs = self.test_step(batch)
                logs = {**logs, **{"val_" + k: v for k, v in vlogs.items()}}
            if self.strategy is not None:
                logs = self.strategy.mean_dict(logs)          # the epoch's logs are the mean over the replicas
            for k, v in logs.items():
                history.setdefault(k, []).append(v)
            if verbose:
                logging.info("epoch %d: %s", epoch + 1, {k: round(float(v), 5) for k, v in logs.items()})
            for cb in callbacks:
                if hasattr(cb, "on_epoch_end"):
                    cb.on_epoch_end(epoch, logs)
        self.history = history
        return history
