"""Per-row statistic of the single-GPU NT-Xent forward.

The FIXED-mode forward (normalised rows, tau >= ~0.045) computes each tile of the symmetric S = Z Z^T once and takes
the row sums of its mirror tile from the column sums.  A tile that is skipped or counted twice moves the loss by only
~3e-7 (relative) at M = 65536, far inside the loss tolerance, so these tests check the statistic itself: for every row
a, stat_a = wscale / L_a with L_a = sum_{b != a} exp2(t_ab), t_ab = zs_a . zs_b, where zs are the fp16 rows the tensor
cores read (unit rows pre-scaled by sqrt(log2(e) / tau)), taken from the saved blob.  The witness is a chunked fp32
product of the same rows, so it differs from the kernel only by summation order and the exp2 approximation
(max relative error 7.5e-5 per element on the polynomial path).  One missing 128-column tile shifts L_a by
~128 / M relative: 2e-3 at M = 65536.
"""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# per-row maximum of |L_kernel / L_witness - 1| measured on a B200 (profiles/r3_tuning_log.md §2): up to 8.6e-5 with
# the full-matrix forward, up to 1.5e-5 with the symmetric one; one missing tile at R = 512 shifts L_a by 2e-3
STAT_TOL = 1e-4


@pytest.fixture(scope="module")
def C():
    assert torch.cuda.is_available()
    from ssv_b200 import _cabi
    assert _cabi.lib().ssvb_device_check() == 0, "not a B200"
    return _cabi


def _align(x, a=256):
    return (x + a - 1) // a * a


def run_fwd(C, zi, zj, tau):
    """One ssvb_ntxent_fwd with its own buffers; returns (loss, stat [M], staged rows [M x dpad] as fp32)."""
    L = C.lib()
    n, d = zi.shape
    m = 2 * n
    mpad, dpad = int(L.ssvb_ntxent_mpad(n)), int(L.ssvb_ntxent_dpad(d))
    saved = torch.empty(int(L.ssvb_ntxent_saved_bytes(n, d)), dtype=torch.uint8, device="cuda")
    wsb = int(L.ssvb_ntxent_workspace_bytes(n, d))
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    loss = torch.empty(1, dtype=torch.float32, device="cuda")
    C.check(L.ssvb_ntxent_fwd(C.ptr(zi), C.ptr(zj), n, d, d, d, 1, ctypes.c_float(tau), C.ptr(loss), C.ptr(saved),
                              C.ptr(ws), wsb, C.stream_ptr()), "ssvb_ntxent_fwd")
    torch.cuda.synchronize()
    # saved blob: zhat [mpad x dpad] fp16, inv_norm [mpad] fp32, stat [mpad] fp32, each at a 256-byte boundary
    zh_bytes = mpad * dpad * 2
    off_inv = _align(zh_bytes)
    off_stat = off_inv + _align(mpad * 4)
    zs = saved[:zh_bytes].view(torch.float16).view(mpad, dpad)[:m].float()
    stat = saved[off_stat:off_stat + m * 4].view(torch.float32).clone()
    return loss.clone(), stat, zs


def witness_L(zs, chunk=4096):
    """L_a = sum_{b != a} exp2(zs_a . zs_b) in fp32 (zs pre-scaled: the dot product is the log2-domain logit)."""
    m = zs.shape[0]
    out = torch.empty(m, dtype=torch.float64, device=zs.device)
    for r0 in range(0, m, chunk):
        r1 = min(m, r0 + chunk)
        e = torch.exp2(zs[r0:r1] @ zs.T)
        idx = torch.arange(r0, r1, device=zs.device)
        e[idx - r0, idx] = 0.0
        out[r0:r1] = e.sum(1, dtype=torch.float64)
    return out


def wscale_of(m):
    k = 0
    while (2 << k) <= m:
        k += 1
    return float(1 << min(max(k - 4, 0), 14))


def inputs(n, d, seed):
    g = torch.Generator().manual_seed(seed)
    zi = torch.randn(n, d, generator=g).cuda()
    zj = (zi.cpu() + 0.5 * torch.randn(n, d, generator=g)).cuda()  # correlated views, as in training
    return zi, zj


def max_row_err(C, n, d, tau, seed=0):
    zi, zj = inputs(n, d, seed)
    _, stat, zs = run_fwd(C, zi, zj, tau)
    m = 2 * n
    l_kernel = wscale_of(m) / stat.double()
    l_ref = witness_L(zs)
    return ((l_kernel / l_ref) - 1.0).abs().max().item()


# n -> M = 2n rows, R = ceil(M / 128) row blocks: R = 1, 2 (ragged), 3 (ragged), 4, 5 (ragged), 8
@pytest.mark.parametrize("n", [32, 100, 129, 256, 300, 512])
@pytest.mark.parametrize("d", [32, 64, 128])
@pytest.mark.parametrize("tau", [0.05, 0.5])
def test_row_statistic_small(C, n, d, tau):
    err = max_row_err(C, n, d, tau, seed=n + d)
    assert err <= STAT_TOL, f"n={n} d={d} tau={tau}: max per-row relative error {err:.3e}"


@pytest.mark.parametrize("n,d,tau", [(4100, 128, 0.5), (32768, 128, 0.5), (32768, 64, 0.1)])
def test_row_statistic_large(C, n, d, tau):
    err = max_row_err(C, n, d, tau, seed=7)
    assert err <= STAT_TOL, f"n={n} d={d} tau={tau}: max per-row relative error {err:.3e}"


def test_forward_bitwise_deterministic(C):
    zi, zj = inputs(8192, 128, 3)
    l1, s1, _ = run_fwd(C, zi, zj, 0.5)
    l2, s2, _ = run_fwd(C, zi, zj, 0.5)
    assert torch.equal(l1, l2)
    assert torch.equal(s1, s2)
