"""DinoLoss for wide prototype heads, 8192 < K <= 65536 (DINO's published head is 65536 wide).

These K take the cluster kernels of csrc/next_rows.cu: one thread-block cluster of C = ceil(K / 8192) CTAs per row,
each CTA holding one 8192-column slice in registers, the row statistics combined through distributed shared memory.
K <= 8192 keeps the one-CTA-per-row kernels (test_gpu_next_rows.py); K > 65536 is refused.

Module tests compare with the fp64 oracle `O.dino` at the tolerances of test_dino_oracle (loss rel <= 1e-5, gradient
rel-L2 <= 1e-4: the kernels are fp32 throughout).  The per-row tests drive the C ABI with NaN-filled buffers and check
every loss partial, every Tsum row and every gradient row against fp64; each of their tolerances is shown to be at least
10x below what dropping one full 8192-column slice from the row's normaliser would do to the metric (the failure a
missing or doubled DSMEM entry produces).
"""
import ctypes

import numpy as np
import pytest
import torch

from conftest import rel_scalar
from oracle import ssl_oracle as O
from test_gpu_parity import S, dev, randn  # noqa: F401  (S is a fixture)
from test_gpu_sim_bwd_rows import C  # noqa: F401  (fixture: the C ABI binding on a B200)

pytestmark = pytest.mark.gpu

SLICE = 8192           # columns per CTA of the cluster kernels
MAX_K = 8 * SLICE      # portable cluster size 8

LOSS_TOL = 1e-5        # module loss, relative (test_dino_oracle)
GRAD_TOL = 1e-4        # module gradient, relative L2 (test_dino_oracle)
# per-row tolerances against fp64, about 3x the measured maxima (profiles/r7_dino_wide.md lists them per case); one
# dropped slice moves every row by >= 0.1 in each metric
PART_TOL = 4e-7        # loss partial per (sample, view) row, relative: measured <= 1.0e-7
TSUM_TOL = 1.2e-6      # Tsum row, relative L2: measured <= 3.8e-7
DROW_TOL = 1.2e-6      # gradient row, relative L2: measured <= 3.5e-7


def oracle_chunked(teacher, student, ts, tt, center, grad=None, scale=1.0, chunk=4):
    """O.dino over blocks of `chunk` samples (the loss is a mean over samples).  Returns the loss and, if `grad` (the
    kernel's gradient, numpy) is given, rel-L2 of grad against scale * dstudent, accumulated block by block."""
    bs = teacher.shape[0]
    loss, num, den = 0.0, 0.0, 0.0
    for b0 in range(0, bs, chunk):
        b1 = min(bs, b0 + chunk)
        lc, dc = O.dino(teacher[b0:b1], student[b0:b1], ts, tt, center)
        loss += lc * (b1 - b0) / bs
        if grad is not None:
            ref = dc * ((b1 - b0) / bs * scale)
            num += float(np.sum((grad[b0:b1].astype(np.float64) - ref) ** 2))
            den += float(np.sum(ref ** 2))
    return loss, (num ** 0.5 / den ** 0.5 if grad is not None else None)


def module_case(S, teacher, student, center, ts, tt, s_dev=None):
    t, c = dev(teacher, False), dev(center, False)
    s = dev(student) if s_dev is None else s_dev
    loss = S.DinoLoss()(t, s, ts, tt, c)
    (3.0 * loss).backward()
    ref_loss, gerr = oracle_chunked(teacher, student, ts, tt, center, s.grad.cpu().numpy(), 3.0)
    assert np.isfinite(s.grad.cpu().numpy()).all()
    lerr = rel_scalar(loss.item(), ref_loss)
    print(f"K={teacher.shape[2]}: loss rel {lerr:.2e}, grad rel-L2 {gerr:.2e}")
    assert lerr <= LOSS_TOL, f"loss {loss.item()} vs {ref_loss}: rel {lerr:.3e}"
    assert gerr <= GRAD_TOL, f"gradient rel-L2 {gerr:.3e}"
    return t, s, c, ref_loss


# ------------------------------------------------------------------------------------------------ module parity
@pytest.mark.parametrize("bs,nv,k,ts,tt", [
    (64, 12, 65536, 0.1, 0.04),   # DINO: 2 global + 10 local crops, C = 8
    (4, 2, 8193, 0.1, 0.04),      # scalar path (K % 4 != 0), C = 2, one-column last slice
    (1, 3, 40000, 0.1, 0.04),     # bs = 1, C = 5, ragged last slice
    (130, 4, 16384, 0.1, 0.07),   # C = 2, 1040 student CTAs: several waves
    (8, 2, 65536, 0.05, 0.02),    # peaky softmaxes
])
def test_dino_wide_oracle(S, bs, nv, k, ts, tt):
    teacher, student, center = randn(0, bs, 2, k), randn(1, bs, nv, k), 0.2 * randn(2, k)
    t, s, c, ref_loss = module_case(S, teacher, student, center, ts, tt)
    # the reference's call pattern (models/dino.py:161-162): both teacher views, the second through a flipped view
    loss2 = 0.5 * S.DinoLoss()(t, s, ts, tt, c) + 0.5 * S.DinoLoss()(t.flip(1), s, ts, tt, c)
    assert rel_scalar(loss2.item(), ref_loss) <= LOSS_TOL


def test_dino_wide_misaligned_student(S):
    """A student at a storage offset of one float with K % 4 == 0: the rows are not 16-byte aligned, so the scalar
    cluster kernels run at a K the float4 kernels would otherwise take."""
    bs, nv, k = 6, 3, 20480
    teacher, student, center = randn(3, bs, 2, k), randn(4, bs, nv, k), 0.2 * randn(5, k)
    buf = torch.empty(bs * nv * k + 1, device="cuda")
    buf[1:].copy_(torch.from_numpy(student).view(-1))
    s = buf[1:].view(bs, nv, k).detach().requires_grad_(True)
    assert s.is_contiguous() and s.data_ptr() % 16 == 4
    module_case(S, teacher, student, center, 0.1, 0.04, s_dev=s)


@pytest.mark.parametrize("k", [SLICE, SLICE + 1, MAX_K])
def test_dino_wide_boundaries(S, k):
    """K = 8192 is the last width of the one-CTA-per-row kernels, 8193 the first of the cluster kernels, 65536 the last."""
    teacher, student, center = randn(6, 3, 2, k), randn(7, 3, 4, k), 0.2 * randn(8, k)
    module_case(S, teacher, student, center, 0.1, 0.04)


def test_dino_wide_rejects_k_above_65536(S):
    k = MAX_K + 1
    t, s, c = torch.randn(1, 2, k, device="cuda"), torch.randn(1, 2, k, device="cuda", requires_grad=True), \
        torch.zeros(k, device="cuda")
    with pytest.raises(RuntimeError, match="65536"):
        S.DinoLoss()(t, s, 0.1, 0.04, c)


@pytest.mark.parametrize("bs,nv,k", [(64, 12, MAX_K), (4, 2, SLICE + 1)])
def test_dino_wide_deterministic(S, bs, nv, k):
    teacher, student, center = dev(randn(9, bs, 2, k), False), randn(10, bs, nv, k), dev(0.2 * randn(11, k), False)
    out = []
    for _ in range(2):
        s = dev(student)
        loss = S.DinoLoss()(teacher, s, 0.1, 0.04, center)
        loss.backward()
        out.append((loss.detach().clone(), s.grad.clone()))
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1]), "two runs differ"


def test_dino_wide_cuda_graph(S):
    """Forward + backward at DINO's shape captured in a CUDA graph (by hand: the temperatures are floats, which
    `make_graphed_callables` does not take) and replayed on new inputs copied into the static tensors: bit-identical
    with eager."""
    bs, nv, k, ts, tt = 64, 12, MAX_K, 0.1, 0.04
    fn = S.DinoLoss()
    st_t, st_c = dev(randn(20, bs, 2, k), False), dev(0.2 * randn(21, k), False)
    st_s = dev(randn(22, bs, nv, k))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            st_s.grad = None
            fn(st_t, st_s, ts, tt, st_c).backward()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    st_s.grad = None
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        st_loss = fn(st_t, st_s, ts, tt, st_c)
        st_loss.backward()
    for seed in (30, 40):
        teacher, student, center = randn(seed, bs, 2, k), randn(seed + 1, bs, nv, k), 0.2 * randn(seed + 2, k)
        with torch.no_grad():
            st_t.copy_(torch.from_numpy(teacher))
            st_s.copy_(torch.from_numpy(student))
            st_c.copy_(torch.from_numpy(center))
        g.replay()
        t, s, c = dev(teacher, False), dev(student), dev(center, False)
        loss = fn(t, s, ts, tt, c)
        loss.backward()
        torch.cuda.synchronize()
        assert torch.equal(st_loss.detach(), loss.detach()), "graph replay loss differs from eager"
        assert torch.equal(st_s.grad, s.grad), "graph replay gradient differs from eager"
    ref_loss, gerr = oracle_chunked(teacher, student, ts, tt, center, s.grad.cpu().numpy())
    assert rel_scalar(loss.item(), ref_loss) <= LOSS_TOL and gerr <= GRAD_TOL


def test_dino_center_update_wide(S):
    """update_teacher_center at K = 65536 on the teacher outputs of a DINO batch ([bs, 2, K] -> 2 bs rows)."""
    k, m = MAX_K, 0.9
    rows0, rows1 = randn(12, 64, 2, k), randn(13, 64, 2, k)
    c0 = S.update_teacher_center(None, dev(rows0, False), m)
    ref0 = O.dino_center_update(None, rows0.reshape(-1, k), m)
    np.testing.assert_allclose(c0.cpu().numpy(), ref0, rtol=2e-6, atol=1e-7)
    c1 = S.update_teacher_center(dev(ref0, False), dev(rows1, False), m)
    np.testing.assert_allclose(c1.cpu().numpy(), O.dino_center_update(ref0, rows1.reshape(-1, k), m), rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(c0.cpu().numpy(), rows0.reshape(-1, k).astype(np.float64).mean(0), rtol=1e-4, atol=1e-6)


# ------------------------------------------------------------------------------------------------ per-row witnesses
def ru(x, a):
    return (x + a - 1) // a * a


def workspace_layout(bs, nv, k):
    """ssvb_dino_workspace_bytes restated: [bs * nv] fp32 loss partials, padded to 256 bytes, then Tsum [bs x k] fp32,
    plus 256 bytes.  Returns (float offset of Tsum, total bytes)."""
    part_bytes = ru(bs * nv * 4, 256)
    return part_bytes // 4, part_bytes + bs * k * 4 + 256


def run_cabi(C, t, s, c, ts, tt, go):
    """ssvb_dino_fwd then ssvb_dino_bwd with the test's own NaN-filled workspace and gradient buffers."""
    L = C.lib()
    bs, nv, k = s.shape
    wsb = int(L.ssvb_dino_workspace_bytes(bs, nv, k))
    tsum_off, total = workspace_layout(bs, nv, k)
    assert total == wsb, f"workspace layout restated as {total} bytes, library says {wsb}"
    ws = torch.full((wsb // 4,), float("nan"), device="cuda")
    loss = torch.full((1,), float("nan"), device="cuda")
    st = C.stream_ptr()
    C.check(L.ssvb_dino_fwd(C.ptr(t), C.ptr(s), C.ptr(c), bs, nv, k, ctypes.c_float(ts), ctypes.c_float(tt), C.ptr(loss),
                            C.ptr(ws), wsb, st), "ssvb_dino_fwd")
    torch.cuda.synchronize()
    part = ws[:bs * nv].clone().view(bs, nv)
    tsum = ws[tsum_off:tsum_off + bs * k].clone().view(bs, k)
    ws.fill_(float("nan"))
    ds = torch.full_like(s, float("nan"))
    gout = torch.full((1,), go, device="cuda")
    C.check(L.ssvb_dino_bwd(C.ptr(t), C.ptr(s), C.ptr(c), bs, nv, k, ctypes.c_float(ts), ctypes.c_float(tt), C.ptr(gout),
                            C.ptr(ds), C.ptr(ws), wsb, st), "ssvb_dino_bwd")
    torch.cuda.synchronize()
    return loss.item(), part, tsum, ds


def witness(t, s, c, ts, tt, go, drop=None):
    """fp64 Tsum [bs, k], loss partials [bs, nv] and gradient [bs, nv, k]; `drop` = a column slice whose exponentials
    are left out of every normaliser (teacher views and student rows), the numerators unchanged."""
    bs, nv, k = s.shape

    def softmax(x):
        e = torch.exp(x - x.amax(-1, keepdim=True))
        z = e.sum(-1, keepdim=True)
        if drop is not None:
            z = z - e[..., drop].sum(-1, keepdim=True)
        return e / z, z

    T, _ = softmax((t.double() - c.double()) / tt)
    tsum = T.sum(1)
    x = s.double() / ts
    p, _ = softmax(x)
    logp = torch.log(p)
    part = -(tsum[:, None, :] * logp).sum(-1)
    grad = (2.0 * p - tsum[:, None, :]) * (go / (ts * bs * nv))
    return tsum, part, grad


def row_rel_l2(got, ref):
    return (got.double() - ref).norm(dim=-1) / ref.norm(dim=-1)


# (bs, nv, K): C = ceil(K / 8192); scalar path where K % 4 != 0
ROW_CASES = [(4, 2, SLICE + 1), (3, 5, 40000), (5, 3, 20002), (16, 12, MAX_K)]


@pytest.mark.parametrize("bs,nv,k", ROW_CASES)
def test_dino_wide_rows(C, bs, nv, k):
    """Every loss partial, Tsum row and gradient row of the cluster kernels against fp64.  Logits of about unit scale
    (teacher = centre + 2 temp_t N(0, 1), student = 2 temp_s N(0, 1)) spread each row's mass over all its slices, so
    dropping any one full slice from a normaliser moves every row."""
    ts, tt, go = 0.1, 0.04, 0.7
    g = torch.Generator().manual_seed(bs * 1000 + k)
    c = (0.2 * torch.randn(k, generator=g)).cuda()
    t = (c.cpu() + 2 * tt * torch.randn(bs, 2, k, generator=g)).cuda()
    s = (2 * ts * torch.randn(bs, nv, k, generator=g)).cuda()
    loss, part, tsum, ds = run_cabi(C, t, s, c, ts, tt, go)
    for name, x in (("loss partials", part), ("Tsum", tsum), ("gradient", ds)):
        assert torch.isfinite(x).all(), f"{name}: non-finite entries (a slice or row never stored)"
    w_tsum, w_part, w_grad = witness(t, s, c, ts, tt, go)
    j = (bs + nv) % (k // SLICE)                     # a full slice, chosen by the shape
    p_tsum, p_part, p_grad = witness(t, s, c, ts, tt, go, drop=slice(j * SLICE, (j + 1) * SLICE))
    metrics = {
        "partial": ((part.double() - w_part).abs() / w_part.abs(), (part.double() - p_part).abs() / p_part.abs(), PART_TOL),
        "tsum": (row_rel_l2(tsum, w_tsum), row_rel_l2(tsum, p_tsum), TSUM_TOL),
        "grad": (row_rel_l2(ds, w_grad), row_rel_l2(ds, p_grad), DROW_TOL),
    }
    for name, (err, power, tol) in metrics.items():
        print(f"bs={bs} nv={nv} K={k} {name}: max {err.max().item():.3e}, dropped slice {j}: min {power.min().item():.3e},"
              f" tol {tol:.1e}")
        assert err.max().item() <= tol, f"{name}: max per-row error {err.max().item():.3e} > {tol:.1e}"
        assert power.min().item() >= 10 * tol, f"{name}: one dropped slice moves a row only {power.min().item():.3e}"
    ref_loss = w_part.sum().item() / (bs * nv)
    assert rel_scalar(loss, ref_loss) <= LOSS_TOL, (loss, ref_loss)
