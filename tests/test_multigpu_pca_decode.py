"""2-GPU check of the PCA decode from one thread (skipped when fewer than 2 devices): the TMA kernels need more than
48 KB of shared memory, an opt-in that belongs to each device, so the second device must get it as well."""
import numpy as np
import pytest
import torch

from conftest import rel_l2

pytestmark = pytest.mark.gpu
GRAD_TOL = 2e-5     # as test_gpu_parity: the adjoint adds each block's fp32 partial sums with atomics, in any order


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_pca_decode_tma_path_on_two_devices_from_one_thread():
    from liftreg_b200 import _native, ops
    rs = np.random.RandomState(0)
    B, K, N = 2, 56, 3 * 24 * 28 * 32          # K = 56: both directions take the TMA kernels (~86 KB of shared memory)
    coefs, basis, mean, gout = (rs.standard_normal(s).astype(np.float32) for s in ((B, K), (N, K), (N,), (B, N)))
    want = gout.astype(np.float64) @ basis.astype(np.float64)
    outs = []
    for dev in (torch.device("cuda", 0), torch.device("cuda", 1)):
        d_basis, d_gout = torch.from_numpy(basis).to(dev), torch.from_numpy(gout).to(dev)
        outs.append(ops.pca_decode(torch.from_numpy(coefs).to(dev), d_basis, torch.from_numpy(mean).to(dev)).cpu())
        # the adjoint is called here rather than through autograd, whose backward runs on a thread per device
        gcoefs = torch.zeros((B, K), device=dev)
        with torch.cuda.device(dev):
            _native.check(_native.lib().lr_pca_decode_backward(ops._ptr(d_gout), ops._ptr(d_basis), B, K, N, ops._ptr(gcoefs),
                                                               ops._stream()), "lr_pca_decode_backward")
        assert rel_l2(gcoefs.cpu().numpy(), want) <= GRAD_TOL, dev
    assert torch.equal(outs[0], outs[1])        # the forward has no atomics: the same bits on both devices
