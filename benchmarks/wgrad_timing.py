#!/usr/bin/env python
"""Per-CTA counters of the weight-gradient kernel (tc_wgrad_kernel) at the two shapes of bench.py's training step:
32,768 rays x 64 (coarse pass) and x 192 samples (fine pass).  Needs the -DKNERF_TC_TIMING build:

    python -c 'import __graft_entry__ as g; print(g.build_timing_variant())'
    KNERF_LIB_PATH=keras_nerf_b200/lib/libknerf_timing.so python benchmarks/wgrad_timing.py [records=fp8|bf16] [rays=32768]

Each shape runs forward, dgrad-only, then wgrad-only calls; the counters of the last wgrad-only call are read (the
others are cleared).  Times are CTA means (kcycles) unless marked; `end min/max` = earliest over latest CTA end time,
both measured from the earliest CTA start (%globaltimer)."""
import ctypes as C
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_PROF = 12


def run_shape(R, S, records):
    from keras_nerf_b200 import NeRF, _lib
    from keras_nerf_b200.model.nerf import mlp as mlp_mod
    dev = torch.device("cuda", 0)
    mlp_mod.set_seed(42)
    model = NeRF(precision="bf16", device=dev, records=records)   # 64 coarse + 128 fine samples: the workspace fits S = 192
    model.compile(optimizer="adam", loss="mse", batch_size=1, image_height=R // 64, image_width=64, ray_chunks=R,
                  white_background=True)
    g = torch.Generator(device="cpu").manual_seed(0)
    o = torch.zeros(R, 3, device=dev)
    o[:, 2] = 4.0
    d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1).to(dev)
    t = torch.sort(torch.rand(R, S, generator=g) * 4 + 2, dim=-1).values.to(dev).contiguous()
    rgbs = torch.empty(R, S, 4, device=dev)
    dpre = (torch.randn(R, S, 4, generator=g) * 1e-4).to(dev)
    grads = torch.zeros_like(model.fine.params)
    prec = model._prec_train
    packed = model._packed_ptr("fine")
    ws, wsn = model._ws.data_ptr(), model._ws.numel()
    lib = _lib.load()
    _lib.call("knerf_mlp_forward", C.byref(model.cfg), _lib.ptr(model.fine.params), packed, _lib.ptr(o), _lib.ptr(d),
              _lib.ptr(t), R, S, prec, 1, _lib.ptr(rgbs), ws, wsn, _lib.stream())

    def bwd(flags):
        _lib.call("knerf_mlp_backward", C.byref(model.cfg), _lib.ptr(model.fine.params), packed, _lib.ptr(dpre), R, S,
                  prec | flags, _lib.ptr(grads), ws, wsn, _lib.stream())

    bwd(_lib.BWD_DGRAD_ONLY)
    buf = (C.c_ulonglong * (160 * N_PROF))()
    for _ in range(3):
        torch.cuda.synchronize()
        lib.knerf_debug_wgrad_timing(buf, 160 * N_PROF)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        bwd(_lib.BWD_WGRAD_ONLY)
        e1.record()
        torch.cuda.synchronize()
    n = lib.knerf_debug_wgrad_timing(buf, 160 * N_PROF)
    if n == 0:
        raise SystemExit("library built without -DKNERF_TC_TIMING (see the module docstring)")
    a = np.frombuffer(buf, dtype=np.uint64).reshape(160, N_PROF).astype(np.float64)
    a = a[a[:, 9] > 0]                                   # CTAs of the launch
    m = a.mean(0)
    t0 = a[:, 9].min()
    end = a[:, 10] - t0
    cyc = m[11]
    return {
        "shape": f"{R} x {S}", "records": records, "ctas": len(a), "ms (events, incl. finish kernels)": e0.elapsed_time(e1),
        "kernel ms (globaltimer)": (a[:, 10].max() - t0) / 1e6,
        "CTA kcycles": cyc / 1e3,
        "producer wait empty": m[0] / 1e3, "issuer0 wait full": m[1] / 1e3, "issuer1 wait full": m[2] / 1e3,
        "issuer0 wait acc_free": m[3] / 1e3, "issuer1 wait acc_free": m[4] / 1e3,
        "flush wait acc_done": m[6] / 1e3, "flush total": m[5] / 1e3,
        "flush per item": m[5] / max(m[7], 1) / 1e3, "items per CTA": m[7], "tiles per CTA": m[8],
        "items min/max": f"{a[:, 7].min():.0f}/{a[:, 7].max():.0f}",
        "end min/max": end.min() / end.max(),
    }


def main():
    records = sys.argv[1] if len(sys.argv) > 1 else "fp8"
    R = int(sys.argv[2]) if len(sys.argv) > 2 else 32768
    rows = [run_shape(R, S, records) for S in (64, 192)]
    print(f"| counter (CTA mean, kcycles unless noted) | " + " | ".join(r["shape"] for r in rows) + " |")
    print("|---|" + "---|" * len(rows))
    for k in rows[0]:
        if k == "shape":
            continue
        vals = [r[k] if isinstance(r[k], str) else (f"{r[k]:.3f}" if abs(r[k]) < 10 else f"{r[k]:.0f}") for r in rows]
        print(f"| {k} | " + " | ".join(vals) + " |")


if __name__ == "__main__":
    main()
