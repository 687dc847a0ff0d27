"""GPU (-m gpu): the backward split into its two halves (KNERF_BWD_DGRAD_ONLY, then KNERF_BWD_WGRAD_ONLY, the way the
kernel benchmarks time them) gives the gradients of the whole backward -- also when the weight-gradient half is run
twice: every call must hand out its work items from the start again."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("records", ["bf16", "fp8"])
@pytest.mark.parametrize("R,S", [(37, 192), (1031, 192)])   # fewer work items than CTAs / more
def test_split_backward_matches_whole(R, S, records):
    import keras_nerf_b200 as K
    from keras_nerf_b200 import _lib
    from keras_nerf_b200.model.nerf import mlp as mlp_mod
    mlp_mod.set_seed(42)
    m = K.NeRF(precision="bf16", records=records)
    m.compile(optimizer="adam", loss="mse", batch_size=1, image_height=1, image_width=R, ray_chunks=R,
              white_background=True)
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(R)
    o = torch.zeros(R, 3)
    o[:, 2] = 4.0
    d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g) * 0.2 + torch.tensor([0, 0, -1.0]), dim=-1)
    t = torch.sort(torch.rand(R, S, generator=g) * 4 + 2, dim=-1).values.contiguous()
    dpre = (torch.randn(R, S, 4, generator=g) * 1e-3).to(dev)
    o, d, t = o.to(dev), d.to(dev), t.to(dev)
    rgbs = torch.empty(R, S, 4, device=dev)
    packed = m._packed_ptr("fine")
    _lib.call("knerf_mlp_forward", C.byref(m.cfg), _lib.ptr(m.fine.params), packed, _lib.ptr(o), _lib.ptr(d), _lib.ptr(t),
              R, S, m._prec_train, 1, _lib.ptr(rgbs), m._ws.data_ptr(), m._ws.numel(), _lib.stream())

    def bwd(flags):
        grads = torch.zeros_like(m.fine.params)
        _lib.call("knerf_mlp_backward", C.byref(m.cfg), _lib.ptr(m.fine.params), packed, _lib.ptr(dpre), R, S,
                  m._prec_train | flags, _lib.ptr(grads), m._ws.data_ptr(), m._ws.numel(), _lib.stream())
        return grads

    whole = bwd(0)
    dgrad = bwd(_lib.BWD_DGRAD_ONLY)
    wgrad = [bwd(_lib.BWD_WGRAD_ONLY) for _ in range(2)]
    scale = float(whole.abs().max())
    assert scale > 0
    for w in wgrad:
        assert float((dgrad + w - whole).abs().max()) <= 1e-5 * scale   # fp32 summation order only
