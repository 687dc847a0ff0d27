"""GPU (-m gpu): the MMA shape of the forward's last GEMM step with the heads folded into it (tc_layout.cuh FwdProg):
one tcgen05.mma.cta_group::2 with M = 256 and N = 16, i.e. 8 B rows per CTA, through the self-test kernel's own K-major
descriptors (LBO = SBO = 128 B).  The chain kernel's descriptors and weight layout for that step are checked end to end
by the forward-vs-fp32 tests of test_gpu_tc.py."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def kmajor_blob(x):
    """[rows, K] -> chunk-major [K/8][rows][8] (tc_ptx.cuh)"""
    rows, K = x.shape
    return x.reshape(rows, K // 8, 8).permute(1, 0, 2).contiguous()


@pytest.mark.parametrize("K", [16, 64, 256])
def test_umma_selftest_2cta_n16(K):
    from keras_nerf_b200 import _lib
    dev = torch.device("cuda")
    N = 16
    g = torch.Generator().manual_seed(K)
    A = torch.randn(256, K, generator=g).to(torch.bfloat16)
    B = torch.randn(N, K, generator=g).to(torch.bfloat16)
    a_d = torch.stack([kmajor_blob(A[:128]), kmajor_blob(A[128:])]).contiguous().to(dev)
    b_d = torch.stack([kmajor_blob(B[:N // 2]), kmajor_blob(B[N // 2:])]).contiguous().to(dev)
    out = torch.full((256, N), float("nan"), device=dev)
    _lib.call("knerf_selftest_umma2", a_d.data_ptr(), b_d.data_ptr(), N, K, _lib.ptr(out), _lib.stream())
    torch.cuda.synchronize()
    ref = A.float() @ B.float().T
    err = float((out.cpu() - ref).abs().max())
    assert err <= 1e-3 * max(1.0, float(ref.abs().max())), err
