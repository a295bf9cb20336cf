"""GPU parity tests: the CUDA path (through the C ABI) vs the CPU oracle on identical seeded inputs,
and vs the golden fixtures produced by the reference itself.

Tolerances are BASELINE.json's: loss relative error <= 1e-3, gradient relative L2 error <= 1e-2
(bf16 tensor-core operands, fp32 accumulation); ring-buffer bookkeeping bit-exact.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_l2, rel_scalar, ulp_diff
from oracle import ssl_oracle as O

pytestmark = pytest.mark.gpu
ROOT = __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__)))
PKG = __import__("os").path.join(ROOT, "self-supervised-vision_b200")

LOSS_TOL = 1e-3
GRAD_TOL = 1e-2


@pytest.fixture(scope="module")
def S():
    import ssv_b200
    assert torch.cuda.is_available()
    from ssv_b200 import _cabi
    assert _cabi.lib().ssvb_device_check() == 0, "not a B200"
    return ssv_b200


def dev(x, grad=True):
    t = torch.as_tensor(np.asarray(x, dtype=np.float32)).cuda()
    return t.requires_grad_(grad)


def randn(seed, *shape):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g, dtype=torch.float32).numpy()


def clustered(seed, n, d, rho=0.8):
    a = randn(seed, n, d)
    b = (rho * a + (1 - rho ** 2) ** 0.5 * randn(seed + 1, n, d)).astype(np.float32)
    if n >= 4:
        a[1] = a[0] + 0.01 * randn(seed + 2, d)
        b[3] = a[2] + 0.01 * randn(seed + 3, d)
    return a, b


def check(loss, grads, ref_loss, ref_grads, what, loss_tol=LOSS_TOL, grad_tol=GRAD_TOL):
    lerr = rel_scalar(loss, ref_loss)
    assert np.isfinite(float(loss)), f"{what}: loss not finite"
    assert lerr <= loss_tol, f"{what}: loss {float(loss)} vs {ref_loss} rel {lerr:.3e}"
    for i, (g, r) in enumerate(zip(grads, ref_grads)):
        g = g.detach().cpu().numpy()
        assert np.isfinite(g).all(), f"{what}: grad {i} not finite"
        gerr = rel_l2(g, r)
        assert gerr <= grad_tol, f"{what}: grad {i} rel-L2 {gerr:.3e}"


# ------------------------------------------------------------------------------------------------ NT-Xent
@pytest.mark.parametrize("tag", ["a", "b", "c", "d", "cfg1"])
def test_ntxent_golden(S, tag):
    g = load_golden("ntxent")
    norm, tau = bool(g[f"{tag}_cfg"][0]), float(g[f"{tag}_cfg"][1])
    zi, zj = dev(g[f"{tag}_zi"]), dev(g[f"{tag}_zj"])
    loss = S.SimclrLoss(norm, tau)(zi, zj)
    loss.backward()
    if tag == "d":
        assert abs(loss.item()) < 1e-5 and zi.grad.abs().max().item() < 1e-5
        return
    check(loss.item(), [zi.grad, zj.grad], float(g[f"{tag}_loss"]), [g[f"{tag}_dzi"], g[f"{tag}_dzj"]], f"ntxent[{tag}]")


@pytest.mark.parametrize("n,d,norm,tau,clu", [
    (256, 128, True, 0.5, False),      # BASELINE configs[0]
    (100, 64, True, 0.5, False),       # ragged: M=200 not a tile multiple, one 64-wide k block
    (129, 128, True, 0.07, True),      # peaky softmax, near-duplicate negatives, diagonal straddles tiles
    (384, 96, False, 1.0, False),      # raw inputs -> online-max path, padded feature dim
    (640, 128, True, 0.02, True),      # tau below the fixed-shift bound -> online-max path
    (2048, 128, True, 0.5, False),     # several row blocks x column chunks (atomic accumulation path)
    (1024, 32, True, 0.1, False),
    (300, 256, True, 0.5, False),      # 128 < d <= 256: four k-blocks, 128-column tiles, backward in two halves
    (700, 192, True, 0.1, True),       # ... padded to 256, several row blocks, peaky
    (384, 200, False, 1.0, False),     # ... raw inputs -> online-max path
])
def test_ntxent_oracle(S, n, d, norm, tau, clu):
    zi, zj = clustered(3, n, d) if clu else (randn(0, n, d), randn(1, n, d))
    if not norm:
        zi, zj = zi * 0.3, zj * 0.3
    ref = O.ntxent(zi, zj, norm, tau)
    a, b = dev(zi), dev(zj)
    loss = S.SimclrLoss(norm, tau)(a, b)
    loss.backward()
    check(loss.item(), [a.grad, b.grad], ref[0], ref[1:], f"ntxent n={n} d={d} tau={tau}")


def test_ntxent_grad_scale_and_determinism(S):
    zi, zj = randn(0, 300, 128), randn(1, 300, 128)
    a, b = dev(zi), dev(zj)
    fn = S.SimclrLoss(True, 0.5)
    l1 = fn(a, b)
    (3.0 * l1).backward()
    g3 = a.grad.clone()
    a.grad = None
    l2 = fn(a, b)
    l2.backward()
    assert torch.equal(l1, l2), "loss must be run-to-run deterministic"
    assert rel_l2(g3.cpu().numpy(), 3.0 * a.grad.cpu().numpy()) < 1e-6


def test_ntxent_permutation_invariance(S):
    zi, zj = randn(0, 200, 128), randn(1, 200, 128)
    perm = torch.randperm(200, generator=torch.Generator().manual_seed(5)).numpy()
    fn = S.SimclrLoss(True, 0.2)
    l0 = fn(dev(zi, False), dev(zj, False)).item()
    l1 = fn(dev(zi[perm], False), dev(zj[perm], False)).item()
    assert abs(l0 - l1) / abs(l0) < 1e-5


def test_ntxent_large_self_consistency(S):
    """BASELINE size (N=32768 per view, M=65536): chunked fp32 closed form on the GPU (bench.parity_witness: plain
    torch.matmul, TF32 off) as witness for the loss AND for the gradient rows of a 4096-row slab of each view, plus
    exact properties of the whole gradient: sum_a dz_a . z_a == 0 (normalised rows), finite values."""
    from bench import parity_witness
    n, d, tau = 32768, 128, 0.5
    g = torch.Generator(device="cuda").manual_seed(0)
    zi = torch.randn(n, d, device="cuda", generator=g)
    zj = torch.randn(n, d, device="cuda", generator=g)
    a, b = zi.clone().requires_grad_(True), zj.clone().requires_grad_(True)
    loss = S.SimclrLoss(True, tau)(a, b)
    loss.backward()
    par = parity_witness(a, b, a.grad, loss.item(), 1, 0, None, rows=4096, tau=tau, dzj=b.grad)
    assert par["loss_rel"] <= LOSS_TOL, par
    assert par["grad_rel_l2"] <= GRAD_TOL, par
    assert torch.isfinite(a.grad).all() and torch.isfinite(b.grad).all()
    radial = (a.grad * zi).sum(1).abs().max().item()
    assert radial < 1e-6 * max(1.0, a.grad.abs().max().item() * zi.norm(dim=1).max().item()) + 1e-7


@pytest.mark.parametrize("n,tau", [(16384, 0.1), (8192, 0.07)])
def test_ntxent_large_peaky_gradient_witness(S, n, tau):
    """Peaky softmax at large M (clustered positives, low temperature): numerical gradient witness on a 4096-row slab."""
    from bench import parity_witness
    g = torch.Generator(device="cuda").manual_seed(1)
    zi = torch.randn(n, 128, device="cuda", generator=g)
    zj = 0.8 * zi + 0.6 * torch.randn(n, 128, device="cuda", generator=g)
    a, b = zi.clone().requires_grad_(True), zj.clone().requires_grad_(True)
    loss = S.SimclrLoss(True, tau)(a, b)
    loss.backward()
    par = parity_witness(a, b, a.grad, loss.item(), 1, 0, None, rows=4096, tau=tau, dzj=b.grad)
    assert par["loss_rel"] <= LOSS_TOL and par["grad_rel_l2"] <= GRAD_TOL, par


# ------------------------------------------------------------------------------------------------ MoCo
@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_moco_golden(S, tag):
    g = load_golden("moco")
    norm, tau = bool(g[f"{tag}_cfg"][0]), float(g[f"{tag}_cfg"][1])
    q, k, mem = dev(g[f"{tag}_q"]), dev(g[f"{tag}_k"]), dev(g[f"{tag}_mem"], False)
    loss = S.MocoLoss(norm, tau)(q, k, mem)
    loss.backward()
    check(loss.item(), [q.grad, k.grad], float(g[f"{tag}_loss"]), [g[f"{tag}_dq"], g[f"{tag}_dk"]], f"moco[{tag}]")


@pytest.mark.parametrize("n,k,d,tau", [(256, 65536, 128, 0.07), (100, 1000, 128, 0.07), (300, 4100, 64, 0.2),
                                       (200, 5000, 256, 0.07), (64, 1000, 160, 0.2)])
def test_moco_oracle(S, n, k, d, tau):
    q, kk = randn(0, n, d), randn(1, n, d)
    mem = randn(2, k, d)
    mem /= np.linalg.norm(mem, axis=1, keepdims=True)
    mem[:7] = 0.0
    ref = O.moco(q, kk, mem, True, tau)
    a, b, m = dev(q), dev(kk), dev(mem, False)
    loss = S.MocoLoss(True, tau)(a, b, m)
    loss.backward()
    check(loss.item(), [a.grad, b.grad], ref[0], ref[1:], f"moco n={n} k={k}")


def test_moco_with_device_bank(S):
    """cfg2: 256 queries x 65536-entry queue + enqueue with a wrap; bank-resident bf16 shadow path."""
    n, ksz, d, tau = 256, 65536, 128, 0.07
    bank = S.MemoryBank(ksz, d)
    fill = randn(5, ksz, d)
    ref_bank, ref_ptr = np.zeros((ksz, d), np.float32), 0
    # fill the queue in 4 big batches, then advance the pointer so that the next enqueue wraps
    for i in range(4):
        chunk = fill[i * 16384:(i + 1) * 16384]
        bank.add_batch(torch.from_numpy(chunk).cuda())
        nrm = np.maximum(np.linalg.norm(chunk.astype(np.float64), axis=1, keepdims=True), 1e-12)
        ref_bank[i * 16384:(i + 1) * 16384] = (chunk / nrm).astype(np.float32)
    assert bank.ptr == 0
    bank.add_batch(torch.from_numpy(fill[:ksz - 100]).cuda())
    assert bank.ptr == ksz - 100
    q, kk = randn(0, n, d), randn(1, n, d)
    a, b = dev(q), dev(kk)
    mem = bank.get_vectors().to("cuda")
    loss = S.MocoLoss(True, tau)(a, b, mem)
    loss.backward()
    ref = O.moco(q, kk, mem.cpu().numpy(), True, tau)
    check(loss.item(), [a.grad, b.grad], ref[0], ref[1:], "moco cfg2 (bank)")
    before = mem.cpu().numpy().copy()
    bank.add_batch(b.detach())
    exp_bank, exp_ptr = O.ring_enqueue(before, ksz - 100, kk, True)
    assert bank.ptr == exp_ptr == 156
    got = bank.bank.cpu().numpy()
    changed = np.where((got != before).any(1))[0]
    assert set(changed) <= set(list(range(ksz - 100, ksz)) + list(range(156)))
    # SURVEY §8 a3: rows match fp32 `x / max(sqrt(sum x^2), 1e-12)` to <= 1 ulp.  The oracle here is the fp64 result
    # rounded to fp32; an fp32 evaluation (the reference's own, or ours) carries <= 1 ulp from the fp32 norm plus <= 1 ulp
    # from the quotient, so the bound against the fp64-rounded value is 2 ulp (the <= 1 ulp bound against the reference's
    # own fp32 output is asserted on the golden fixture in test_ring_buffers_golden)
    assert ulp_diff(got, exp_bank) <= 2, f"ring rows differ by {ulp_diff(got, exp_bank)} ulp"


def test_moco_enqueue_between_forward_and_backward(S):
    """ADVICE r1: a bank enqueue between MocoLoss forward and backward must never yield silently wrong gradients.
    * device-resident MemoryBank + normalize=True (fused single-pass kernel): the forward already produced
      sum_j p_aj m_j, the backward never reads the queue -> any loop order is valid and the gradient is that of the queue
      AS IT WAS at forward time (what the reference computes: its loss sees a per-step copy, models/moco.py:117);
    * normalize=False (two-pass form, backward re-reads the queue): the enqueue bumps the storage's version counter and
      autograd refuses the stale backward."""
    bank = S.MemoryBank(1024, 64)
    bank.add_batch(torch.from_numpy(randn(3, 1024, 64)).cuda())
    a, b = dev(randn(0, 32, 64)), dev(randn(1, 32, 64))
    then = bank.get_vectors().cpu().numpy().copy()
    loss = S.MocoLoss(True, 0.2)(a, b, bank.get_vectors())
    bank.add_batch(b.detach())
    loss.backward()
    ref = O.moco(a.detach().cpu().numpy(), b.detach().cpu().numpy(), then, True, 0.2)
    check(loss.item(), [a.grad, b.grad], ref[0], ref[1:], "moco fused, enqueue before backward")
    # the shadow stays in sync across enqueues
    for _ in range(2):
        a.grad = b.grad = None
        mem = bank.get_vectors()
        loss = S.MocoLoss(True, 0.2)(a, b, mem)
        loss.backward()
        ref = O.moco(a.detach().cpu().numpy(), b.detach().cpu().numpy(), mem.cpu().numpy(), True, 0.2)
        check(loss.item(), [a.grad, b.grad], ref[0], ref[1:], "moco after enqueue")
        bank.add_batch(b.detach())
    a.grad = b.grad = None
    loss = S.MocoLoss(False, 1.0)(a, b, bank.get_vectors())
    bank.add_batch(b.detach())
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        loss.backward()


@pytest.mark.parametrize("n,k,d,tau", [(256, 8192, 128, 0.07), (100, 1000, 128, 0.07), (300, 4100, 64, 0.2), (7, 130, 32, 0.5)])
def test_moco_fused_single_pass_vs_two_pass(S, n, k, d, tau):
    """The fused single-pass kernel (bank-resident queue) against the oracle and against the two-pass online-max form
    on the same data, incl. zero rows (a partly filled ring), ragged K (queue tail inside a tile) and N not a multiple
    of 128."""
    bank = S.MemoryBank(k, d)
    fill = randn(2, k - 5, d)
    bank.add_batch(torch.from_numpy(fill).cuda())          # the last 5 rows stay zero
    q, kk = randn(0, n, d), randn(1, n, d)
    mem = bank.get_vectors()
    ref = O.moco(q, kk, mem.cpu().numpy(), True, tau)
    a, b = dev(q), dev(kk)
    loss = S.MocoLoss(True, tau)(a, b, mem)                 # fused (shadow found)
    loss.backward()
    check(loss.item(), [a.grad, b.grad], ref[0], ref[1:], f"moco fused n={n} k={k}")
    a2, b2 = dev(q), dev(kk)
    loss2 = S.MocoLoss(True, tau)(a2, b2, mem.clone())      # plain tensor: two-pass form
    loss2.backward()
    assert rel_scalar(loss.item(), loss2.item()) <= 1e-5
    assert rel_l2(a.grad.cpu().numpy(), a2.grad.cpu().numpy()) <= 5e-3


def test_swav_reference_loop_order_enqueue_before_backward(S):
    """The reference's SwAV step enqueues the new features BEFORE loss.backward() (models/swav.py:140-144):
    FeatureBank.return_vectors hands the loss a snapshot, so that order is valid and the gradients are those of the
    bank as it was at forward time."""
    fb = S.FeatureBank(300, 64)
    bank0 = randn(9, 300, 64)
    bank0 /= np.linalg.norm(bank0, axis=1, keepdims=True)   # the bank holds encoder outputs, which are unit rows (swav.py:41)
    fb.add_vectors(torch.from_numpy(bank0).cuda())
    z1 = randn(0, 64, 64); z1 /= np.linalg.norm(z1, axis=1, keepdims=True)
    z2 = randn(1, 64, 64); z2 /= np.linalg.norm(z2, axis=1, keepdims=True)
    c = randn(2, 100, 64); c /= np.linalg.norm(c, axis=1, keepdims=True)
    a, b, p = dev(z1), dev(z2), dev(c)
    bank_then = fb.return_vectors("cuda")
    ref = O.swav(z1, z2, c, bank_then.cpu().numpy(), 0.1, 0.05, 3)
    loss = S.SwavLoss(0.1, 0.05, 3)(a, b, p, bank_then)
    fb.add_vectors(torch.cat([a, b], 0).detach().cpu())
    loss.backward()
    check(loss.item(), [a.grad, b.grad, p.grad], ref[0], ref[1:], "swav, enqueue before backward")


# ------------------------------------------------------------------------------------------------ ring buffers
def test_ring_buffers_golden(S):
    g = load_golden("banks")
    mb, fb = S.MemoryBank(10, 4), S.FeatureBank(7, 3 + 1)  # d must be a multiple of 4: pad the 3-wide golden
    assert not mb.bank.any().item() and mb.ptr == 0
    for step in range(5):
        mb.add_batch(torch.from_numpy(g[f"mb_batch{step}"]).cuda())
        assert mb.ptr == int(g[f"mb_ptr{step}"])
        got = mb.get_vectors().cpu().numpy()
        # fp32 x / max(sqrt(sum x^2), 1e-12) with true division, as F.normalize.  The sum of squares is accumulated in a
        # different order than torch's CPU kernel (and with FMA contraction), so the norm may differ by 1 ulp and the
        # quotient by one more: <= 2 ulp against the reference's own fp32 rows is the tight bound (measured: 2), the
        # "<= 1 ulp" of SURVEY §8 a3 would require reproducing ATen's summation order.  Bookkeeping (ptr, which rows were
        # overwritten) is exact.
        assert ulp_diff(got, g[f"mb_bank{step}"]) <= 2, "normalised ring rows must be within 2 ulp of the reference's"
        assert ((got == 0) == (g[f"mb_bank{step}"] == 0)).all()
        fbatch = np.concatenate([g[f"fb_batch{step}"], np.zeros((len(g[f"fb_batch{step}"]), 1), np.float32)], 1)
        fb.add_vectors(torch.from_numpy(fbatch))  # CPU input, like models/swav.py:141
        assert fb.ptr == int(g[f"fb_ptr{step}"])
        assert np.array_equal(fb.return_vectors("cuda").cpu().numpy()[:, :3], g[f"fb_bank{step}"])


def test_prototypes_and_l2norm(S):
    g = load_golden("banks")
    pw = g["proto_weight"]                      # RefPrototypes(hidden_dim=6, prototype_size=9): weight [9 x 6]
    p = S.Prototypes(8, pw.shape[0]).cuda()     # feature dim padded 6 -> 8 (rows must be 16-byte multiples)
    w = np.zeros((pw.shape[0], 8), np.float32)
    w[:, :pw.shape[1]] = pw
    with torch.no_grad():
        p.embedding.weight.copy_(torch.from_numpy(w))
    out = p("cuda")
    assert rel_l2(out.detach().cpu().numpy()[:, :pw.shape[1]], g["proto_out"]) < 1e-6
    x = dev(randn(0, 37, 24))
    y = S.banks.l2_normalize(x)
    gy = torch.from_numpy(randn(1, 37, 24)).cuda()
    y.backward(gy)
    xr = torch.from_numpy(randn(0, 37, 24)).requires_grad_(True)
    yr = torch.nn.functional.normalize(xr, dim=-1)
    yr.backward(gy.cpu())
    assert rel_l2(y.detach().cpu().numpy(), yr.detach().numpy()) < 1e-6
    assert rel_l2(x.grad.cpu().numpy(), xr.grad.numpy()) < 1e-5


# ------------------------------------------------------------------------------------------------ row-dot
def test_rowdot_golden(S):
    g = load_golden("rowdot")
    o, t = dev(g["o"]), dev(g["t"])
    loss = S.SimSiamLoss()(o, t)
    loss.backward()
    check(loss.item(), [o.grad, t.grad], float(g["ss_loss"]), [g["ss_do"], g["ss_dt"]], "simsiam", 1e-5, 1e-5)
    o, t = dev(g["o"]), dev(g["t"])
    loss = S.MSELoss()(o, t)
    loss.backward()
    check(loss.item(), [o.grad, t.grad], float(g["mse_loss"]), [g["mse_do"], g["mse_dt"]], "mse", 1e-5, 1e-5)


@pytest.mark.parametrize("n,d", [(512, 128), (4096, 1024), (33, 20)])
def test_rowdot_oracle(S, n, d):
    o = randn(0, n, d) / np.sqrt(d)
    t = randn(1, n, d) / np.sqrt(d)
    a, b = dev(o), dev(t, False)  # BYOL: target has no grad path
    loss = S.MSELoss()(a, b)
    loss.backward()
    ref = O.mse(o, t)
    check(loss.item(), [a.grad], ref[0], ref[1:2], "mse", 1e-5, 1e-5)
    a, b = dev(o), dev(t)
    loss = S.SimSiamLoss()(a, b)
    loss.backward()
    ref = O.simsiam(o, t)
    check(loss.item(), [a.grad, b.grad], ref[0], ref[1:], "simsiam", 1e-4, 1e-5)


# ------------------------------------------------------------------------------------------------ ReLIC
@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_relic_golden(S, tag):
    g = load_golden("relic")
    norm, tau, alpha = bool(g[f"{tag}_cfg"][0]), float(g[f"{tag}_cfg"][1]), float(g[f"{tag}_cfg"][2])
    zi, zj, zo = dev(g[f"{tag}_zi"]), dev(g[f"{tag}_zj"]), dev(g[f"{tag}_zo"])
    loss = S.RelicLoss(norm, tau, alpha)(zi, zj, zo)
    loss.backward()
    check(loss.item(), [zi.grad, zj.grad, zo.grad], float(g[f"{tag}_loss"]),
          [g[f"{tag}_dzi"], g[f"{tag}_dzj"], g[f"{tag}_dzo"]], f"relic[{tag}]")


@pytest.mark.parametrize("n,d,tau", [(512, 128, 1.0), (4096, 128, 1.0), (300, 64, 0.2), (260, 256, 0.5)])
def test_relic_oracle(S, n, d, tau):
    zi, zj, zo = randn(0, n, d), randn(1, n, d), randn(2, n, d)
    ref = O.relic(zi, zj, zo, True, tau, 0.5)
    a, b, c = dev(zi), dev(zj), dev(zo)
    loss = S.RelicLoss(True, tau, 0.5)(a, b, c)
    loss.backward()
    check(loss.item(), [a.grad, b.grad, c.grad], ref[0], ref[1:], f"relic n={n}")


# ------------------------------------------------------------------------------------------------ Sinkhorn
@pytest.mark.parametrize("tag", ["a", "b"])
def test_sinkhorn_golden(S, tag):
    g = load_golden("swav")
    codes = S.SwavLoss(0.1, 0.05, 3).compute_codes_sinkhorn(dev(g[f"sk_{tag}_scores"], False))
    assert rel_l2(codes.cpu().numpy(), g[f"sk_{tag}_codes"]) < 1e-4


@pytest.mark.parametrize("b,k,iters", [(4096, 3000, 3), (3512, 3000, 3), (257, 5000, 2), (64, 30, 0), (100, 8, 5)])
def test_sinkhorn_oracle(S, b, k, iters):
    z = randn(0, b, 128)
    c = randn(1, k, 128)
    z /= np.linalg.norm(z, axis=1, keepdims=True)
    c /= np.linalg.norm(c, axis=1, keepdims=True)
    scores = (z @ c.T).astype(np.float32)
    ref = O.sinkhorn(scores, 0.05, iters)
    codes = S.SwavLoss(0.1, 0.05, iters).compute_codes_sinkhorn(dev(scores, False)).cpu().numpy()
    assert np.isfinite(codes).all()
    assert rel_l2(codes, ref) < 1e-4
    np.testing.assert_allclose(codes.sum(1), 1.0, rtol=1e-4)
    if iters > 0:  # prototype marginals are uniform up to the last column normalisation
        assert abs(codes.sum() - b) / b < 1e-4


# ------------------------------------------------------------------------------------------------ Barlow Twins
@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_barlow_golden(S, tag):
    g = load_golden("barlow")
    norm, lm = bool(g[f"{tag}_cfg"][0]), float(g[f"{tag}_cfg"][1])
    zi, zj = dev(g[f"{tag}_zi"]), dev(g[f"{tag}_zj"])
    loss = S.BarlowLoss(norm, lm)(zi, zj)
    loss.backward()
    check(loss.item(), [zi.grad, zj.grad], float(g[f"{tag}_loss"]), [g[f"{tag}_dzi"], g[f"{tag}_dzj"]], f"barlow[{tag}]")


def barlow_inputs(n, d, corr=0.7):
    g = torch.Generator().manual_seed(7)
    sig = (torch.rand(d, generator=g) * 1.5 + 0.5).numpy()
    mu = torch.randn(d, generator=g).numpy()
    zi = randn(0, n, d) * sig + mu
    zj = corr * zi + (1 - corr) * (randn(1, n, d) * sig + mu)
    return zi.astype(np.float32), zj.astype(np.float32)


@pytest.mark.parametrize("n,d,norm", [(512, 4096, False), (256, 1000, False), (200, 264, True), (200, 264, False),
                                      (2048, 8192, False)])   # norm False: closed-form backward in the GEMM epilogue (ragged M / N tails)
def test_barlow_oracle(S, n, d, norm):
    zi, zj = barlow_inputs(n, d)
    a, b = dev(zi), dev(zj)
    loss = S.BarlowLoss(norm, 0.005)(a, b)
    loss.backward()
    if n * d * d > 3e10:   # cfg3 (2048 x 8192): fp64 oracle on CPU takes too long; chunked fp32 torch witness on GPU
        with torch.no_grad():
            xi = torch.from_numpy(zi).cuda().double()
            xj = torch.from_numpy(zj).cuda().double()
        xi.requires_grad_(True); xj.requires_grad_(True)
        ti = (xi - xi.mean(0)) / xi.std(0)
        tj = (xj - xj.mean(0)) / xj.std(0)
        c = ti.t() @ tj / n
        eye = torch.eye(d, device="cuda", dtype=torch.float64)
        ref_loss = (((c - eye) ** 2) * (0.005 + (1 - 0.005) * eye)).sum()
        ref_loss.backward()
        ref = (ref_loss.item(), xi.grad.cpu().numpy(), xj.grad.cpu().numpy())
    else:
        ref = O.barlow(zi, zj, norm, 0.005)
    check(loss.item(), [a.grad, b.grad], ref[0], ref[1:], f"barlow n={n} d={d}")


# ------------------------------------------------------------------------------------------------ SwAV
@pytest.mark.parametrize("tag", ["nobank", "bank", "c"])
def test_swav_golden(S, tag):
    g = load_golden("swav")
    z1, z2, c = dev(g[f"sw_{tag}_z1"]), dev(g[f"sw_{tag}_z2"]), dev(g[f"sw_{tag}_c"])
    bank = dev(g[f"sw_{tag}_bank"], False) if f"sw_{tag}_bank" in g else None
    loss = S.SwavLoss(0.1, 0.05, 3)(z1, z2, c, bank)
    loss.backward()
    check(loss.item(), [z1.grad, z2.grad, c.grad], float(g[f"sw_{tag}_loss"]),
          [g[f"sw_{tag}_dz1"], g[f"sw_{tag}_dz2"], g[f"sw_{tag}_dc"]], f"swav[{tag}]")


@pytest.mark.parametrize("nb,nbank,k,d", [(512, 3000, 3000, 128), (300, 0, 100, 64), (64, 70, 1000, 32),
                                          (200, 1000, 1000, 96),    # split-K gradient GEMMs with ragged K slices / N tails
                                          (64, 0, 4100, 32)])       # K > 4096: generic cross-entropy kernel, Sinkhorn
                                                                    # one view at a time through the shared-memory passes
def test_swav_oracle(S, nb, nbank, k, d):
    def unit(x):
        return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)
    z1 = unit(randn(0, nb, d))
    z2 = unit(0.6 * z1 + 0.4 * randn(1, nb, d))
    c = unit(randn(2, k, d))
    bank = unit(randn(3, nbank, d)) if nbank else None
    ref = O.swav(z1, z2, c, bank, 0.1, 0.05, 3)
    a, b, p = dev(z1), dev(z2), dev(c)
    loss = S.SwavLoss(0.1, 0.05, 3)(a, b, p, dev(bank, False) if nbank else None)
    loss.backward()
    check(loss.item(), [a.grad, b.grad, p.grad], ref[0], ref[1:], f"swav nb={nb} k={k}")


@pytest.mark.parametrize("iters,temp,eps", [(0, 0.1, 0.05), (1, 0.1, 0.05), (5, 0.2, 0.03)])
def test_swav_iteration_counts(S, iters, temp, eps):
    """sinkhorn_iters = 0 (no iteration: the final-pass + code-matrix path), 1 (the scaling vectors come from the first
    alpha kernel alone) and 5, with other temperatures / eps: the codes rebuilt inside the cross-entropy kernel must
    match the reference's dense iteration (utils/losses.py:213-235) for any count."""
    def unit(x):
        return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)
    z1 = unit(randn(0, 160, 64))
    z2 = unit(0.6 * z1 + 0.4 * randn(1, 160, 64))
    c = unit(randn(2, 500, 64))
    bank = unit(randn(3, 90, 64))
    ref = O.swav(z1, z2, c, bank, temp, eps, iters)
    a, b, p = dev(z1), dev(z2), dev(c)
    loss = S.SwavLoss(temp, eps, iters)(a, b, p, dev(bank, False))
    loss.backward()
    check(loss.item(), [a.grad, b.grad, p.grad], ref[0], ref[1:], f"swav iters={iters}")


def test_swav_dist_ce_unaligned_rows(S):
    """ssvb_swav_dist_ce takes the float4 cross-entropy kernel on 16-byte aligned score / code rows and the generic one
    (swav_ce_kernel) on rows that are not: on the same scores and codes, once from aligned buffers and once from copies
    that start one float into a larger buffer, the loss and the ssvb_swav_bwd gradients driven by each call's dscores
    agree.  K % 4 != 0, so both kernels mask the padding columns."""
    import ctypes
    from ssv_b200 import _cabi as C
    L, st = C.lib(), C.stream_ptr()
    nb, nbank, k, d, temp = 200, 100, 1001, 96, 0.1

    def unit(x):
        return torch.from_numpy((x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)).cuda()
    z1, z2, bank, proto = unit(randn(0, nb, d)), unit(randn(1, nb, d)), unit(randn(2, nbank, d)), unit(randn(3, k, d))
    bp, kp = nb + nbank, int(L.ssvb_swav_kpad(k))
    wsb = int(L.ssvb_swav_workspace_bytes(nb, nbank, k, d))
    saved = torch.empty(int(L.ssvb_swav_saved_bytes(nb, nbank, k, d)), dtype=torch.uint8, device="cuda")
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    scores = torch.zeros(2 * bp, kp, device="cuda")
    C.check(L.ssvb_swav_dist_scores(C.ptr(z1), C.ptr(z2), C.ptr(bank), C.ptr(proto), nb, nbank, k, d, d, d, d, d,
                                    C.ptr(scores), C.ptr(saved), st), "ssvb_swav_dist_scores")
    codes = torch.zeros_like(scores)
    codes[:, :k] = torch.softmax(scores[:, :k] / 0.05, dim=1)

    def unaligned(t):
        u = torch.zeros(t.numel() + 4, device="cuda")[1:1 + t.numel()].view(t.shape)
        u.copy_(t)
        assert u.data_ptr() % 16 == 4
        return u

    def run(sc, cd):
        loss, go = torch.empty(1, device="cuda"), torch.ones(1, device="cuda")
        C.check(L.ssvb_swav_dist_ce(C.ptr(sc), C.ptr(cd), nb, nbank, bp, k, d, ctypes.c_float(temp), C.ptr(loss),
                                    C.ptr(saved), C.ptr(ws), wsb, st), "ssvb_swav_dist_ce")
        g = [torch.empty(nb, d, device="cuda"), torch.empty(nb, d, device="cuda"), torch.empty(k, d, device="cuda")]
        C.check(L.ssvb_swav_bwd(C.ptr(z1), C.ptr(z2), C.ptr(bank), C.ptr(proto), nb, nbank, k, d, d, d, d, d,
                                ctypes.c_float(temp), C.ptr(go), C.ptr(saved), *(C.ptr(x) for x in g), d, d, d, C.ptr(ws),
                                wsb, st), "ssvb_swav_bwd")
        torch.cuda.synchronize()
        return loss.item(), [x.cpu().numpy() for x in g]

    la, ga = run(scores, codes)
    lu, gu = run(unaligned(scores), unaligned(codes))
    lerr = rel_scalar(lu, la)
    gerr = [rel_l2(u, a) for u, a in zip(gu, ga)]
    print(f"unaligned vs aligned: loss rel {lerr:.3e}, gradient rel-L2 {', '.join(f'{e:.3e}' for e in gerr)}")
    assert np.isfinite(la) and all(np.isfinite(g).all() for g in ga + gu)
    # measured on one B200 at 1000 W: loss rel 0, gradient rel-L2 <= 2.2e-5 (dscores that round to a neighbouring bf16)
    assert lerr <= 1e-6, (lu, la)
    assert max(gerr) <= 6.5e-5, gerr


# ------------------------------------------------------------------------------------------------ GEMM epilogue paths
@pytest.mark.parametrize("switches", [
    {"SSVB_GEMM_NO_TMA_STORE": "1"},
], ids=["row-store-epilogue"])
def test_alternative_paths_match_oracle(switches):
    """`SSVB_GEMM_NO_TMA_STORE=1` (read once per process, hence the subprocess) forces the per-thread row-store GEMM
    epilogue that rows without 16-byte alignment take instead of the staged TMA store: Barlow (fused loss epilogue, then
    the backward through the fp32 dT buffers with a separate column reduction) and SwAV (fp32 scores, no split-K), against
    the oracle."""
    import os
    import subprocess
    import sys
    code = r"""
import sys, numpy as np, torch
sys.path[:0] = [%r, %r]
import ssv_b200 as S
from oracle import ssl_oracle as O
g = torch.Generator().manual_seed(3)
zi = (torch.randn(200, 264, generator=g) * 1.3 + 0.2).numpy(); zj = (0.7 * zi + 0.3 * torch.randn(200, 264, generator=g).numpy()).astype(np.float32)
a, b = torch.from_numpy(zi).cuda().requires_grad_(True), torch.from_numpy(zj).cuda().requires_grad_(True)
loss = S.BarlowLoss(False, 0.005)(a, b); loss.backward()
ref = O.barlow(zi, zj, False, 0.005)
rl2 = lambda x, y: np.linalg.norm(x - y) / np.linalg.norm(y)
assert abs(loss.item() - ref[0]) / abs(ref[0]) <= 1e-3, (loss.item(), ref[0])
assert rl2(a.grad.cpu().numpy(), ref[1]) <= 1e-2 and rl2(b.grad.cpu().numpy(), ref[2]) <= 1e-2
unit = lambda x: (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)
z1 = unit(torch.randn(200, 96, generator=g).numpy()); z2 = unit(0.6 * z1 + 0.4 * torch.randn(200, 96, generator=g).numpy())
c = unit(torch.randn(1000, 96, generator=g).numpy())
t1, t2, tc = (torch.from_numpy(x).cuda().requires_grad_(True) for x in (z1, z2, c))
l2 = S.SwavLoss(0.1, 0.05, 3)(t1, t2, tc, None); l2.backward()
r2 = O.swav(z1, z2, c, None, 0.1, 0.05, 3)
assert abs(l2.item() - r2[0]) / abs(r2[0]) <= 1e-3
assert rl2(t1.grad.cpu().numpy(), r2[1]) <= 1e-2 and rl2(tc.grad.cpu().numpy(), r2[3]) <= 1e-2
print("fallback-ok")
""" % (ROOT, PKG)
    env = dict(os.environ, **switches)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "fallback-ok" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]
