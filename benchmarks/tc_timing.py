#!/usr/bin/env python
"""In-kernel cycle breakdown of the tcgen05 chain kernels (forward and dgrad) at R rays x 192 samples.  Needs the
-DKNERF_TC_TIMING build:

    python -c 'import __graft_entry__ as g; print(g.build_timing_variant())'
    KNERF_LIB_PATH=keras_nerf_b200/lib/libknerf_timing.so python benchmarks/tc_timing.py [rays=8192] [records=bf16|fp8] [fwd|dgrad]

fwd: the forward kernel at inference (train=0) and training (train=1).  dgrad: forward, then three dgrad-only backward
calls; the counters of the last one are read.  Counters are CTA means (tc_roles.cuh slots); `epilogue cycles per step`
are per work unit (two tiles per CTA) and tile slot, `prologue` the same for the tile's first A operand."""
import ctypes as C
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main():
    R = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
    S = 192
    from keras_nerf_b200 import NeRF, _lib
    from keras_nerf_b200.model.nerf import mlp as mlp_mod
    dev = torch.device("cuda", 0)
    mlp_mod.set_seed(42)
    records = sys.argv[2] if len(sys.argv) > 2 else "bf16"
    mode = sys.argv[3] if len(sys.argv) > 3 else "fwd"
    if mode not in ("fwd", "dgrad"):
        raise SystemExit("mode: fwd or dgrad")
    model = NeRF(precision="bf16", device=dev, records=records)
    model.compile(optimizer="adam", loss="mse", batch_size=1, image_height=R // 64, image_width=64, ray_chunks=R,
                  white_background=True)
    g = torch.Generator(device="cpu").manual_seed(0)
    o = torch.zeros(R, 3, device=dev)
    o[:, 2] = 4.0
    d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1).to(dev)
    t = torch.sort(torch.rand(R, S, generator=g) * 4 + 2, dim=-1).values.to(dev).contiguous()
    rgbs = torch.empty(R, S, 4, device=dev)
    packed = model._packed_ptr("fine")
    ws, wsn = model._ws.data_ptr(), model._ws.numel()
    lib = _lib.load()
    buf = (C.c_ulonglong * (160 * 40))()
    tiles = R * S / 128 / 148
    units = tiles / 2

    def report(label, n, steps):
        if n == 0:
            print("library built without -DKNERF_TC_TIMING")
            return False
        m = np.frombuffer(buf, dtype=np.uint64).reshape(160, 40)[:148].astype(np.float64).mean(0)
        print(f"{label}: tiles/CTA {tiles:.1f}; per CTA kcycles: producer-wait-empty {m[0]/1e3:.0f}, "
              f"mma-wait-A {m[1]/1e3:.0f}, mma-wait-stage {m[2]/1e3:.0f}, mma-total {m[3]/1e3:.0f}, "
              f"compute-wait-acc {m[4]/1e3:.0f}, compute-total {m[5]/1e3:.0f}")
        for tl in range(2):
            line = " ".join(f"{m[6 + tl * 16 + s] / units:.0f}" for s in range(steps))
            line += f"; prologue {m[15 + tl * 16] / units:.0f}"
            print(f"  epilogue cycles per step, tile slot {tl}: {line}")
        return True

    def forward(train):
        _lib.call("knerf_mlp_forward", C.byref(model.cfg), _lib.ptr(model.fine.params), packed, _lib.ptr(o),
                  _lib.ptr(d), _lib.ptr(t), R, S, model._prec_train, train, _lib.ptr(rgbs), ws, wsn, _lib.stream())
        torch.cuda.synchronize()

    if mode == "fwd":
        for train in (0, 1):
            for it in range(3):
                forward(train)
                n = lib.knerf_debug_tc_timing(buf, 160 * 40)
            if not report(f"forward train={train}", n, 9):
                return
    else:
        forward(1)
        dpre = (torch.randn(R, S, 4, generator=g) * 1e-4).to(dev)
        grads = torch.zeros_like(model.fine.params)
        for it in range(3):
            _lib.call("knerf_mlp_backward", C.byref(model.cfg), _lib.ptr(model.fine.params), packed, _lib.ptr(dpre), R,
                      S, model._prec_train | _lib.BWD_DGRAD_ONLY, _lib.ptr(grads), ws, wsn, _lib.stream())
            torch.cuda.synchronize()
            n = lib.knerf_debug_dgrad_timing(buf, 160 * 40)
        report("dgrad", n, 8)

if __name__ == "__main__":
    main()
