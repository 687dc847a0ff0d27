#!/usr/bin/env python
"""bench.py -- keras_nerf hot path on B200: train rays/s (coarse+fine), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--precision auto|fp32|bf16] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one NeRF.train_step (BASELINE.json config[3]: 32,768 rays per GPU from 400x400 synthetic views,
64 coarse + 128 fine samples, coarse+fine forward, backward, Adam) -- weak scaling: every rank trains on its
own 32,768 rays and the 4.77 MB MLP gradient is SUM-all-reduced over NCCL.  `value` = rays of all ranks /
max-over-ranks device time with inputs resident in HBM; `e2e` = the same through the public API from pinned
HOST buffers (H2D of images+rays and D2H of the metrics inside the timed region).

--impl reference times the reference's CPU implementation of the same step: TensorFlow is not installable
offline, so this is the CPU oracle (torch-CPU restatement, `oracle/`) on all host cores.  It runs ONE step of the
same 32,768-ray workload (BASELINE config[0]'s size: one coarse+fine train step, then one 128x128 render), once --
about a minute of CPU work -- whatever --steps / --warmup say; the line reports steps = 1, warmup = 0.

--dump-outputs DIR writes what the timed device steps hand their caller, as float32 DIR/<name>.npy (4.8 MB): the
coarse and fine weights after the last step's Adam update and the two loss accumulators (coarse, fine; summed over the
timed steps).  Inputs, initial weights and sample draws are seeded, so two builds run with the same arguments can be
compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "train_rays_per_sec"
UNIT = "rays/s"
RAYS_PER_GPU = 32768
IMG_WH = 400
N_COARSE, N_FINE = 64, 128
FLOP_FWD_PER_SAMPLE = 1_186_816          # SURVEY §8d: 593,408 MAC, unpadded shapes
FLOP_TRAIN_PER_SAMPLE = 3_489_024        # fwd + wgrad + dgrad
CPU_SAMPLE_RAYS = 8192                   # bounded sample of the cpu_baseline leg (about 10-30 s of CPU work)
CPU_RAY_CHUNKS = 2048                    # BASELINE config[0]'s ray_chunks (train_single.py:17)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        self.thread.join(2)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------------
# CPU arms: the oracle (port of the TF reference) on the host cores, bounded sample
# --------------------------------------------------------------------------------------------------------
def cpu_train_rays_per_sec(n_rays=CPU_SAMPLE_RAYS, steps=1, warmup=0, render=False):
    """The oracle's train_step (torch-CPU fp32, all host cores) on `n_rays` rays of the bench workload: a
    (n_rays/256) x 256 crop of a 400x400 synthetic view, 64 + 128 samples, white background, ray_chunks 2048."""
    import torch
    import oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = O.NerfConfig()
    rng = np.random.default_rng(42)
    pc, pf = O.init_params(cfg, rng), O.init_params(cfg, rng)
    ch, cw = n_rays // 256, 256
    assert ch * cw == n_rays and ch <= IMG_WH
    focal = O.get_focal_from_fov(0.6911112070083618, IMG_WH)
    pose = O.pose_spherical(45.0, -30.0, 4.0)
    u_c = O.uniform24(np.random.default_rng(1234), (IMG_WH, IMG_WH, cfg.n_coarse))
    o, d, t = O.generate_rays(pose, IMG_WH, IMG_WH, focal, 2.0, 6.0, cfg.n_coarse, u_c)
    y0, x0 = (IMG_WH - ch) // 2, (IMG_WH - cw) // 2
    crop = lambda x: x[y0:y0 + ch, x0:x0 + cw][None].contiguous()  # noqa: E731
    rays = (crop(o), crop(d), crop(t))
    images = np.random.default_rng(3).uniform(0, 1, (1, ch, cw, 4)).astype(np.float32)
    u_f = O.uniform24(np.random.default_rng(5678), (n_rays, cfg.n_fine))
    ac, af = O.AdamState(), O.AdamState()
    rc = min(CPU_RAY_CHUNKS, n_rays)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = O.train_step(pc, pf, ac, af, cfg, images, rays, u_f, rc, True)
        pc, pf = out["params_coarse"], out["params_fine"]
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    dt = float(np.mean(times))
    res = {"value": n_rays / dt, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": f"{steps} x {n_rays}-ray coarse+fine train step ({ch}x{cw} crop of a 400x400 view, ray_chunks {rc}), "
                     f"oracle/ torch-CPU fp32 restatement of the TF reference (TF unavailable offline), "
                     f"{dt:.2f} s/step"}
    if render:   # BASELINE config[0]'s second half: one full 128x128 render
        side = 128
        f2 = O.get_focal_from_fov(0.6911112070083618, side)
        u2 = O.uniform24(np.random.default_rng(4321), (side, side, cfg.n_coarse))
        o2, d2, t2 = O.generate_rays(pose, side, side, f2, 2.0, 6.0, cfg.n_coarse, u2)
        uf2 = O.uniform24(np.random.default_rng(8765), (side * side, cfg.n_fine))
        t0 = time.perf_counter()
        O.predict_and_render_images(pc, pf, cfg, (o2[None], d2[None], t2[None]), uf2, CPU_RAY_CHUNKS, True)
        res["render_128x128_s"] = time.perf_counter() - t0
    return res, dt


def run_reference(args, emit):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the same workload as the b200 arm (32,768 rays per step = BASELINE config[0]'s 2 x 128 x 128), ONE step, once
    cb, dt = cpu_train_rays_per_sec(RAYS_PER_GPU, steps=1, warmup=0, render=True)
    cfg = workload_config("fp32", CPU_RAY_CHUNKS)
    cfg["reference_arm"] = ("CPU: one step of the same 32,768-ray workload (+ one 128x128 render, BASELINE config[0]), "
                            "run once; a GPU rank count does not apply")
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": 1, "warmup": 0, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "render": {"metric": "render_s_per_frame_128x128", "value": cb.get("render_128x128_s"), "unit": "s"},
            "gpu_launches": 0}
    emit(line)


def workload_config(precision, ray_chunks, records=None):
    return {"workload": "BASELINE config[3]: coarse+fine NeRF train step, 32768 rays/GPU (128x256 crops of 400x400 "
                        "synthetic orbit views), 64 coarse + 128 fine samples, 8x256 MLPs, white bg, Adam, "
                        "ray-sharded DP",
            "rays_per_gpu": RAYS_PER_GPU, "image_wh": IMG_WH, "n_coarse": N_COARSE, "n_fine": N_FINE,
            "precision_mode": precision, "ray_chunks": ray_chunks,
            # bf16 mode only: storage format of the activation / gradient records between the training kernels (forward
            # outputs and the dgrad chain are the same bits with either; `--records bf16` runs round 1's format)
            "records": records if precision == "bf16" else None,
            "l2": "per-step working set (activations of 6.3M samples) is >> 126 MB L2; inputs rotate over 4 batches"}


# --------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="auto", choices=["auto", "fp32", "bf16", "fp32_tc"])
    ap.add_argument("--records", default="fp8", choices=["bf16", "fp8"], help="bf16 mode: format of the saved records")
    ap.add_argument("--ray-chunks", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-render", action="store_true", help="skip the secondary 800x800 render metric")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the weights and loss accumulators after the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the b200 arm")
    # stdout carries exactly ONE JSON line: libraries that print there (NCCL's version banner at communicator
    # creation) are sent to stderr until the line is written
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args, emit)
    args.warmup = max(args.warmup, 3)

    import torch
    import __graft_entry__ as ge
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        ge.build()
    from keras_nerf_b200 import NeRF, _lib
    from keras_nerf_b200.data.synthetic import SyntheticScene
    from keras_nerf_b200.distributed import RayShardedStrategy
    from keras_nerf_b200.model.nerf import mlp as mlp_mod

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    strategy = RayShardedStrategy(backend="nccl", device=dev) if world > 1 else None
    if strategy is not None:
        strategy.barrier()
    lib = _lib.load()
    precision = args.precision
    if precision == "auto":
        precision = "bf16" if lib.knerf_device_supports_bf16() else "fp32"
    ray_chunks = args.ray_chunks or (RAYS_PER_GPU if precision == "bf16" else 4096)

    mlp_mod.set_seed(42)
    model = NeRF(precision=precision, strategy=strategy, device=dev, records=args.records)
    model.compile(optimizer="adam", loss="mse", batch_size=1, image_height=RAYS_PER_GPU // 256, image_width=256,
                  ray_chunks=ray_chunks, white_background=True)
    if strategy is not None:
        strategy.broadcast_parameters(model)
    scene = SyntheticScene(IMG_WH, N_COARSE, n_views=100, device=dev)
    nb = 4
    # 128 x 256 crops (32,768 rays) of four views per rank, placed so that each mixes sphere and background
    crop_h, crop_w = RAYS_PER_GPU // 256, 256
    batches = [scene.ray_crop(rank * 25 + 6 * k, crop_h, crop_w, y0=(40, 230, 110, 180)[k % 4] + 3 * rank,
                              x0=(20, 124, 72, 60)[k % 4] + 5 * rank, seed=1000 + rank * nb + k) for k in range(nb)]
    host = [(img.cpu().pin_memory(), tuple(r.cpu().pin_memory() for r in rays)) for img, rays in batches]
    h2d = sum(x.numel() * 4 for x in (host[0][0],) + host[0][1])

    def sync():
        torch.cuda.synchronize()
        if strategy is not None:
            strategy.barrier()
            torch.cuda.synchronize()

    def step_device(i):
        img, rays = batches[i % nb]
        model.accumulate_gradients(img, rays, seed=7000 + i, want_images=False)
        model.apply_gradients()

    for i in range(args.warmup):
        step_device(i)
    model._losses.zero_()
    sync()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = lib.knerf_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.steps):
        step_device(args.warmup + i)
    ev1.record()
    sync()
    launches = int(lib.knerf_launch_count() - l0)
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, x in (("coarse_params", model.coarse.params), ("fine_params", model.fine.params),
                        ("losses", model._losses)):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), x.detach().float().cpu().numpy())
    loss_dev = [v / args.steps for v in model._losses.tolist()]
    model._losses.zero_()

    # ---- e2e: public API, pinned host inputs, H2D + train_step + metrics D2H inside the timed region ----
    # input pipeline of a user's training loop (what tf.data's prefetch does for the reference, loader.py:106): the
    # host -> device copy of step i + 1 is issued on a copy stream while step i computes.  Every step's copy is inside
    # the timed region; the first one is not hidden.
    copy_stream = torch.cuda.Stream(device=dev)

    def upload(i):
        img, rays = host[i % nb]
        with torch.cuda.stream(copy_stream):
            out = (img.to(dev, non_blocking=True), tuple(r.to(dev, non_blocking=True) for r in rays))
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return out, ev

    def e2e_loop(n):
        logs, nxt = {}, upload(0)
        for i in range(n):
            (img, rays), ev = nxt
            torch.cuda.current_stream().wait_event(ev)
            if i + 1 < n:
                nxt = upload(i + 1)
            logs = model.train_step((img, rays))
            for x in (img,) + tuple(rays):
                x.record_stream(torch.cuda.current_stream())
        return logs

    e2e_loop(2)
    sync()
    t0 = time.perf_counter()
    logs = e2e_loop(args.steps)
    sync()
    e2e_s = time.perf_counter() - t0
    clk = clocks.stop() if rank == 0 else None

    tt = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if strategy is not None:
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
    ms, e2e_ms = tt.tolist()
    # BASELINE's second metric, config[2]: 800x800 render, the frame's rays sharded over the N ranks (collective)
    from benchmarks.roofline import dominant_kernel_roofline, render_ms_per_frame
    render = None
    if not args.no_render:
        try:
            render = render_ms_per_frame(precision, dev, strategy)
        except Exception as e:  # the secondary metric must never take the headline down
            render = {"error": str(e)[:200]}
    def rank0_done(signal):
        """rank 0 times the CPU baseline on the host cores: the other ranks must not spin meanwhile (an NCCL barrier
        keeps one host thread per rank busy in cudaStreamSynchronize and slowed the 16-thread CPU leg 6x) -- they block
        on the rendezvous store until rank 0 is through"""
        store = torch.distributed.distributed_c10d._get_default_store()
        if signal:
            store.set("knerf_bench_rank0_done", "1")
        else:
            store.wait(["knerf_bench_rank0_done"])

    if rank != 0:
        if strategy is not None:
            rank0_done(False)
            strategy.barrier()
            torch.distributed.destroy_process_group()
        return
    peaks = load_peaks()
    total_rays = RAYS_PER_GPU * world * args.steps
    value = total_rays / (ms * 1e-3)
    e2e_value = total_rays / (e2e_ms * 1e-3)
    roof = dominant_kernel_roofline(model, precision, peaks)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32", "data": "synthetic",
            "config": workload_config(precision, ray_chunks, args.records),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 8 + 4 * 4, "ms_per_step": e2e_ms / args.steps,
                    "pipeline": "step i + 1's H2D copy on a copy stream while step i computes; one D2H read per step"},
            "gpu_launches": launches, "clocks": clk, "roofline": roof,
            "step_tflops": FLOP_TRAIN_PER_SAMPLE * (N_COARSE + N_COARSE + N_FINE) * RAYS_PER_GPU * world
            * args.steps / (ms * 1e-3) / 1e12,
            "losses": {"device_run": loss_dev, "e2e_last": {k: float(v) for k, v in logs.items()}}}
    line["render"] = render
    if not args.no_cpu_baseline:
        line["cpu_baseline"], _ = cpu_train_rays_per_sec()      # rank 0's host cores; the other ranks wait
    else:
        line["cpu_baseline"] = None
    emit(line)
    if strategy is not None:
        rank0_done(True)
        strategy.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
