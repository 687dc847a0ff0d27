"""Roofline numbers for bench.py: each MLP kernel of the training step timed alone with CUDA events on the
launching stream (burst peaks apply), and the secondary BASELINE metric (800x800 render ms/frame)."""
import ctypes as C
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# SURVEY §8(d): algorithmic work per sample (unpadded shapes)
FLOP_FWD_PER_SAMPLE = 1_186_816            # 593,408 MAC
# bf16 INFERENCE executes fewer: `features`, `rgb_features` and the rgb head are folded into one N = 16 step from h7 and
# PE(dir) (no activation before the sigmoid, mlp.py:42-48) whose column 3 is sigma: 593,408 - 256*256 (features)
# - 283*128 (rgb_features) - 128*3 (rgb) - 256 (sigma) + 288*16 MAC.  Throughput figures keep the unfolded count
# (SURVEY §8d) and carry the executed one next to it.
FLOP_FWD_INFER_EXECUTED = 2 * (593_408 - 256 * 256 - 283 * 128 - 128 * 3 - 256 + 288 * 16)
FLOP_TRAIN_PER_SAMPLE = 3_489_024          # fwd + dgrad + wgrad
FLOP_WGRAD_PER_SAMPLE = 1_186_816          # every weight once more
FLOP_DGRAD_PER_SAMPLE = FLOP_TRAIN_PER_SAMPLE - FLOP_FWD_PER_SAMPLE - FLOP_WGRAD_PER_SAMPLE
# bf16 mode, algorithmic HBM bytes per sample (DESIGN.md §3/§4; records of 576 KB + 516 KB per 128 samples)
BYTES_FWD_SAVE = 568 * 1024 / 128                       # forward writes the activation record (+ ReLU' bits) once
BYTES_DGRAD = 8 * 32 + 516 * 1024 / 128                 # reads the 8 x 1-bit ReLU' tiles, writes dZ0..dZ7 + the d_pre operand
BYTES_WGRAD = 1132 * 1024 / 128                         # operand units of the 10 weight-gradient tasks
# the same with fp8 records (KNERF_REC_FP8, the default; tc_layout.cuh kRec8* / kDz8*)
BYTES8_FWD_SAVE = 300 * 1024 / 128                      # PE(xyz) 8 + PE(dir) 4 + h0..h7 256 + ReLU' bits 32 KB per tile
BYTES8_DGRAD = 8 * 32 + 16 + 258 * 1024 / 128           # reads the ReLU' tiles and d_pre, writes dZ0..dZ7 + the d_pre operand
BYTES8_WGRAD = 566 * 1024 / 128                         # 2 x 40 + 7 x 64 + 38 KB per tile
# measured DRAM traffic per sample (dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture,
# divided by the samples of that launch): profiles/ncu_traffic.json, written from the capture named inside it
def _ncu_traffic(records="bf16"):
    import json
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return {}, None
    d = json.load(open(p))
    if records == "fp8":
        d = d.get("fp8_records", {})
    return d.get("dram_bytes_per_sample", {}), d.get("source")


def _time_ms(fn, iters=5, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def dominant_kernel_roofline(model, precision, peaks):
    """The MLP kernels of the fine network (> 95 % of the step) on the bench's training shapes
    (R = ray_chunks rays x 192 samples), each timed alone; `roofline` names the one with the largest time."""
    from keras_nerf_b200 import _lib
    dev = model.device
    R, S = model.ray_chunks, model.n_coarse + model.n_fine
    rows = R * S
    g = torch.Generator(device="cpu").manual_seed(0)
    o = torch.zeros(R, 3, device=dev)
    o[:, 2] = 4.0
    d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1).to(dev)
    t = torch.sort(torch.rand(R, S, generator=g) * 4 + 2, dim=-1).values.to(dev).contiguous()
    rgbs = torch.empty(R, S, 4, device=dev)
    dpre = (torch.randn(R, S, 4, generator=g) * 1e-4).to(dev)
    grads = torch.zeros_like(model.fine.params)
    prec = model._prec_train
    rec8 = bool(prec & _lib.REC_FP8)
    packed = model._packed_ptr("fine")
    ws, wsn = model._ws.data_ptr(), model._ws.numel()
    lib = _lib.load()

    def fwd():
        _lib.call("knerf_mlp_forward", C.byref(model.cfg), _lib.ptr(model.fine.params), packed, _lib.ptr(o), _lib.ptr(d),
                  _lib.ptr(t), R, S, prec, 1, _lib.ptr(rgbs), ws, wsn, _lib.stream())

    def bwd(flags=0):   # flags: _lib.BWD_DGRAD_ONLY / _lib.BWD_WGRAD_ONLY time the two backward kernels apart
        _lib.call("knerf_mlp_backward", C.byref(model.cfg), _lib.ptr(model.fine.params), packed, _lib.ptr(dpre), R, S,
                  prec | flags, _lib.ptr(grads), ws, wsn, _lib.stream())

    # SURVEY §8(d): the MLP rows are TENSOR-bound work (dense contractions).  Each kernel is timed ALONE here, so the
    # denominator is the BURST cuBLAS bf16 figure of MEASURED_PEAKS.json; the fraction against the sustained figure
    # (what a kernel sees inside the long power-capped step) is carried next to it.  The HBM fractions are
    # secondary: they are computed on "design bytes" -- the activation / gradient records this design moves between
    # its kernels, which an ideal fused implementation would not move at all.
    bf16_peak, bf16_sus, hbm_peak = peaks["bf16_tflops"], peaks["bf16_tflops_sustained"], peaks["hbm_gbs"]
    src = f"{peaks['source']} (MEASURED_PEAKS.json: cuBLAS bf16 burst -- kernels timed alone --, copy bandwidth)"
    traffic_ps, traffic_src = _ncu_traffic("fp8" if rec8 else "bf16")
    kernels = {}

    def add(name, ms, flop_ps, bytes_ps, launches):
        tf = flop_ps * rows / (ms * 1e-3) / 1e12
        k = {"ms": ms, "launches": launches, "tflops": tf, "tensor_frac": tf / bf16_peak,
             "tensor_frac_of_sustained": tf / bf16_sus, "ns_per_sample": ms * 1e6 / rows}
        if bytes_ps:
            gb = bytes_ps * rows / (ms * 1e-3) / 1e9
            k.update({"design_bytes_GBps": gb, "design_bytes_hbm_frac": gb / hbm_peak, "design_bytes_per_sample": bytes_ps})
        if name in traffic_ps:
            k["ncu_dram_bytes_per_sample"] = traffic_ps[name]
        k["algorithmic_flop_per_sample"] = flop_ps
        kernels[name] = k

    l0 = lib.knerf_launch_count()
    fwd()
    n_f = int(lib.knerf_launch_count() - l0)
    ms_f = _time_ms(fwd)
    if precision == "bf16":
        add("tc_mlp_fwd_kernel<train>", ms_f, FLOP_FWD_PER_SAMPLE, BYTES8_FWD_SAVE if rec8 else BYTES_FWD_SAVE, n_f)
        add("tc_mlp_dgrad_kernel", _time_ms(lambda: bwd(_lib.BWD_DGRAD_ONLY)), FLOP_DGRAD_PER_SAMPLE,
            BYTES8_DGRAD if rec8 else BYTES_DGRAD, 2 if rec8 else 1)
        add("tc_wgrad_kernel", _time_ms(lambda: bwd(_lib.BWD_WGRAD_ONLY)), FLOP_WGRAD_PER_SAMPLE,
            BYTES8_WGRAD if rec8 else BYTES_WGRAD, 2)
    else:
        tag = ("fp32_tc forward (encode + tcx_pack + tcx_gemm_kernel + skinny heads)" if precision == "fp32_tc"
               else "fp32 forward (encode + sgemm_kernel + skinny heads)")
        add(tag, ms_f, FLOP_FWD_PER_SAMPLE, None, n_f)
        l0 = lib.knerf_launch_count()
        bwd()
        n_b = int(lib.knerf_launch_count() - l0)
        tag = ("fp32_tc backward (tcx_gemm_kernel + tcx_wgrad_kernel + colsum_kernel)" if precision == "fp32_tc"
               else "fp32 backward (sgemm_kernel<T> + wgrad_kernel + colsum_kernel)")
        add(tag, _time_ms(bwd), FLOP_TRAIN_PER_SAMPLE - FLOP_FWD_PER_SAMPLE, None, n_b)

    name = max(kernels, key=lambda k: kernels[k]["ms"])   # the dominant kernel = the one the step spends most time in
    k = kernels[name]
    per_sample = k.get("ncu_dram_bytes_per_sample")
    roof = {"kernel": name, "bound": "tensor", "achieved": k["tflops"], "peak": bf16_peak, "unit": "TFLOP/s",
            "frac": k["tensor_frac"], "peak_kind": "burst (kernel timed alone, CUDA events on the launching stream)",
            "frac_of_sustained_peak": k["tensor_frac_of_sustained"],
            "traffic": per_sample * rows if per_sample else None,
            "traffic_source": (f"{traffic_src}: DRAM bytes per sample x the {rows} samples of this launch"
                               if per_sample else None),
            "design_bytes_hbm_frac": k.get("design_bytes_hbm_frac"),
            "samples_per_launch": rows, "peak_source": src, "kernels": kernels}
    if precision == "bf16":
        roof["records"] = "fp8 (e4m3 activations / e5m2 gradients for the weight-gradient GEMMs)" if rec8 else "bf16"
        roof["design_bytes_per_sample_step"] = sum(kernels[k].get("design_bytes_per_sample", 0) for k in kernels)
    if precision == "fp32_tc":
        roof["note"] = ("fp32-grade mode on the tensor cores: every product is six bf16 MMAs, so 1/6 of the bf16 peak "
                        "(270 TFLOP/s burst) is its ceiling; TFLOP/s count the fp32 work once")
    elif precision != "bf16":
        roof["note"] = "fp32 SIMT FFMA parity mode measured against the bf16 tensor peak"
    return roof


def render_ms_per_frame(precision, dev, strategy=None, wh=800, frames=2):
    """BASELINE config[2]: 800x800 render, 64 coarse + 128 fine, white background (inference.py path); with a
    multi-rank strategy the frame's ray chunks are sharded over the ranks and the pixels all-gathered
    (NeRF.predict_and_render_images_sharded).  COLLECTIVE: every rank calls it; max over ranks of the device time."""
    from keras_nerf_b200 import NeRF
    from keras_nerf_b200.data.synthetic import SyntheticScene
    from keras_nerf_b200.model.nerf import mlp as mlp_mod
    world = 1 if strategy is None else strategy.num_replicas_in_sync
    mlp_mod.set_seed(42)
    model = NeRF(precision=precision, device=dev, strategy=strategy)
    rc = 16000 if precision == "bf16" else 4000      # 40 / 160 chunks per frame: divisible by 1, 2, 4, 8 ranks
    model.compile(optimizer="adam", loss="mse", batch_size=1, image_height=wh, image_width=wh, ray_chunks=rc,
                  white_background=True, is_training=False)
    if strategy is not None:
        strategy.broadcast_parameters(model)
    scene = SyntheticScene(wh, model.n_coarse, n_views=40, device=dev)
    views = [scene.view(k, seed=k)[1] for k in range(2)]

    def one(k=[0]):
        o, d, t = views[k[0] % 2]
        k[0] += 1
        model.predict_and_render_images_sharded((o[None], d[None], t[None]), seed=100 + k[0])

    if strategy is not None:
        strategy.barrier()
    ms = _time_ms(one, iters=frames, warmup=1)
    if strategy is not None:
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
        ms = float(tt.item())
    samples = wh * wh * (model.n_coarse + model.n_coarse + model.n_fine)
    tf = FLOP_FWD_PER_SAMPLE * samples / (ms * 1e-3) / 1e12
    out = {"metric": "render_ms_per_frame_800x800", "value": ms, "unit": "ms", "n_gpus": world, "tflops": tf,
           "ray_chunks": rc, "precision_mode": model.precision, "higher_is_better": False,
           "sharding": "whole ray chunks of the frame over the ranks, pixels (rgb + depth, coarse + fine: 32 B/ray) "
                       "all-gathered inside the timed region" if world > 1 else "single GPU"}
    if model.precision == "bf16":
        out["tflops_executed"] = FLOP_FWD_INFER_EXECUTED * samples / (ms * 1e-3) / 1e12
        out["note"] = ("tflops counts the unfolded 593,408 MAC/sample; the inference kernel folds features into "
                       "rgb_features and the heads and executes 495,616 MAC/sample (tflops_executed)")
    return out
