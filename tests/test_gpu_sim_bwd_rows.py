"""Per-row checks of the similarity backward (sim_bwd_kernel) and of the per-row statistics it consumes.

The whole-gradient checks elsewhere compare relative L2 at 1e-2.  A weight tile that is skipped, added twice or added to
the wrong row block moves the gradient by ~sqrt(128 / M) of one row block's norm, ~4e-4 of the whole matrix at
M = 8192: far inside that tolerance.  These tests drive the C ABI with their own buffers and check, for EVERY row, the
backward's fp32 accumulator against a witness computed from the same staged 16-bit rows and the kernel's own per-row
statistic, so the backward is isolated from the forward:

    FIXED  (unit rows, tau >= ~0.045; rows pre-scaled so zs_a . zs_b is the log2-domain logit):
        W_ab = exp2(zs_a . zs_b) * (stat_a + stat_b)            stat = wscale / L   (wscale = 2^k, see make_plan)
    ONLINE (otherwise): W_ab = exp2(c s_ab - stat_a) + exp2(c s_ab - stat_b)    stat = log2-domain LSE
    W_aa = 0;  dacc_a = sum_{b < M} W_ab zs_b

Metric: |dacc_kernel,a - dacc_witness,a| / rho_a with rho_a = sqrt(sum_b W_ab^2 |zs_b|^2), the scale of the 16-bit
rounding of the weights (independent of the data), maximised over all rows.  Every accumulator test also removes one
128 x 128 tile (row block and column block chosen by the seed) from the witness and asserts that the kernel's metric
against that perturbed witness exceeds the tolerance at least 10x, so a tolerance cannot become vacuous at a shape.

The workspace is filled with a NaN sentinel before each backward: a row block or column half that is never stored
shows up as a non-finite metric.  The accumulator is the last piece the workspace layout carves (csrc/ntxent.cu
ws_layout); the layout is restated here and checked against the library's workspace size.

Tolerances: measured maxima on one B200 are in profiles/r4_bwd_rows.md; each tolerance is about 3x the largest
maximum of its class and at least 10x below the one-tile perturbation.
"""
import ctypes
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

LOG2E = 1.4426950408889634
FIXED, ONLINE = 0, 1

# tolerances (profiles/r4_bwd_rows.md lists the measured maximum of every shape)
ACC_TOL_F16 = 1.5e-3      # backward accumulator, fp16 weights (normalised rows): measured <= 4.7e-4
ACC_TOL_BF16 = 7e-3       # backward accumulator, bf16 weights (raw rows, ONLINE): measured <= 2.3e-3
FINISH_TOL = 5e-7         # gradient finish restated in fp64 (fp32 reordering only): measured <= 1.5e-7
LSE_TOL = 4e-5            # forward log2-domain LSE per row, absolute: measured <= 1.3e-5
LREL_TOL = 4e-5           # FIXED forward (dpad = 256) row sum L per row, relative: measured <= 1.1e-5
MOCO_LSE_TOL = 6e-6       # fused MoCo lse2 per row, absolute: measured <= 2.0e-6
MOCO_PM_TOL = 7e-3        # fused MoCo sum_j p_aj m_j per row, relative to rho (bf16 weights): measured <= 2.2e-3
MOCO_GRAD_TOL = 5e-7      # MoCo gradient finish restated with the fp32 exponent: measured <= 1.3e-7
ATOMIC_TOL = 1e-6         # run-to-run difference of the red.add accumulator, relative to rho: measured 0


@pytest.fixture(scope="module")
def C():
    assert torch.cuda.is_available()
    from ssv_b200 import _cabi
    assert _cabi.lib().ssvb_device_check() == 0, "not a B200"
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False  # the witnesses are plain fp32 / fp64 products
    yield _cabi
    torch.backends.cuda.matmul.allow_tf32 = prev


# ------------------------------------------------------------------------------------------------ host plan, restated
def ru(x, a):
    return (x + a - 1) // a * a


def cdiv(a, b):
    return (a + b - 1) // b


def num_sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def plan_chunks_tiles(row_blocks, col_tiles, min_tiles, sms):
    """sim_host.cuh plan_chunks_tiles: (tiles_per_chunk, nchunks)."""
    max_ch = col_tiles // min_tiles if col_tiles // min_tiles > 1 else 1
    best, best_score = 1, -1.0
    for nch in range(1, min(max_ch, 256) + 1):
        tpc = cdiv(col_tiles, nch)
        if cdiv(col_tiles, tpc) != nch:
            continue
        waves = cdiv(row_blocks * nch, sms)
        score = row_blocks * col_tiles / (waves * sms * tpc) - 0.002 * nch
        if score > best_score:
            best, best_score = nch, score
    tpc = cdiv(col_tiles, best)
    return tpc, cdiv(col_tiles, tpc)


def bwd_plan(local_rows, cols, sms):
    """The backward's plan_chunks(p, 128, 8)."""
    return plan_chunks_tiles(cdiv(local_rows, 128), cdiv(cols, 128), 8, sms)


def ws_dacc_offset(local_rows, cols, dpad, sms):
    """ntxent.cu ws_layout: (byte offset of dacc, total bytes).  Carver aligns every piece to 256 bytes."""
    lr = ru(local_rows, 256)
    rb = cdiv(local_rows, 128)
    bn = 128 if dpad > 128 else 256
    _, nch = plan_chunks_tiles(rb, cdiv(cols, bn), 1024 // bn, sms)
    part = (4 * nch + 2) * lr
    if local_rows == cols and dpad <= 128:
        band = rb // 2 + 1
        _, nch_s = plan_chunks_tiles(rb, (band + 1) // 2, 4, sms)
        part = max(part, (4 * nch_s + (rb - 1) // 2) * lr)
    part = max(part, ru(cols, 256))
    off = 0
    for nbytes in (lr * 4, part * 4, part * 4, (cdiv(lr, 256) + 8) * 4, 16):
        off = ru(off, 256) + nbytes
    off = ru(off, 256)
    return off, ru(off + lr * dpad * 4, 256)


def wscale_of(m):
    k = 0
    while (2 << k) <= m:
        k += 1
    return float(1 << min(max(k - 4, 0), 14))


def ntx_mode(normalize, tau):
    c = LOG2E / tau
    return FIXED if (normalize and 2 * c <= 64) else ONLINE


# ------------------------------------------------------------------------------------------------ inputs
def inputs(n, d, seed, normalize, tau, ld=None):
    """Two views [n x d] (optionally views of a wider [n x ld] buffer).  Correlated positives only where the softmax
    stays flat (tau >= 0.5); raw (un-normalised) rows are scaled to about unit norm."""
    g = torch.Generator().manual_seed(seed)
    zi = torch.randn(n, d, generator=g)
    zj = torch.randn(n, d, generator=g)
    if tau >= 0.5:
        zj = zi + 0.5 * zj
    if not normalize:
        zi, zj = zi / math.sqrt(d), zj / math.sqrt(d)
    if ld is None:
        return zi.cuda(), zj.cuda()
    bi = torch.full((n, ld), float("nan"))
    bj = torch.full((n, ld), float("nan"))
    bi[:, :d], bj[:, :d] = zi, zj
    return bi.cuda()[:, :d], bj.cuda()[:, :d]


def staged_dtype(normalize):
    return torch.float16 if normalize else torch.bfloat16


# ------------------------------------------------------------------------------------------------ single-GPU runs
def run_ntx(C, zi, zj, tau, normalize, go=1.0, out_ld=None, sentinel=-7.25):
    """ssvb_ntxent_fwd + ssvb_ntxent_bwd with the test's own buffers (workspace NaN-filled before the backward)."""
    L = C.lib()
    n, d = zi.shape
    m = 2 * n
    mpad, dpad = int(L.ssvb_ntxent_mpad(n)), int(L.ssvb_ntxent_dpad(d))
    saved = torch.empty(int(L.ssvb_ntxent_saved_bytes(n, d)), dtype=torch.uint8, device="cuda")
    wsb = int(L.ssvb_ntxent_workspace_bytes(n, d))
    dacc_off, total = ws_dacc_offset(m, m, dpad, num_sms())
    assert total == wsb, f"workspace layout restated as {total} bytes, library says {wsb}"
    assert dacc_off == wsb - ru(m, 256) * dpad * 4
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    loss = torch.empty(1, dtype=torch.float32, device="cuda")
    st = C.stream_ptr()
    C.check(L.ssvb_ntxent_fwd(C.ptr(zi), C.ptr(zj), n, d, zi.stride(0), zj.stride(0), int(normalize), ctypes.c_float(tau),
                              C.ptr(loss), C.ptr(saved), C.ptr(ws), wsb, st), "ssvb_ntxent_fwd")
    ws.fill_(0xFF)  # NaN sentinel: every fp32 word of the workspace
    ld = out_ld or d
    bi = torch.full((n, ld), sentinel, device="cuda")
    bj = torch.full((n, ld), sentinel, device="cuda")
    dzi, dzj = bi[:, :d], bj[:, :d]
    gout = torch.full((1,), go, dtype=torch.float32, device="cuda")
    C.check(L.ssvb_ntxent_bwd(C.ptr(zi), C.ptr(zj), n, d, zi.stride(0), zj.stride(0), int(normalize), ctypes.c_float(tau),
                              C.ptr(gout), C.ptr(saved), C.ptr(dzi), C.ptr(dzj), ld, ld, C.ptr(ws), wsb, st),
            "ssvb_ntxent_bwd")
    torch.cuda.synchronize()
    # saved blob: zhat [mpad x dpad] 16-bit, inv_norm [mpad] fp32, stat [mpad] fp32, each at a 256-byte boundary
    zh_bytes = mpad * dpad * 2
    off_inv = ru(zh_bytes, 256)
    off_stat = off_inv + ru(mpad * 4, 256)
    zs = saved[:zh_bytes].view(staged_dtype(normalize)).view(mpad, dpad)[:m].float()
    return dict(
        n=n, d=d, m=m, dpad=dpad, tau=tau, normalize=normalize, mode=ntx_mode(normalize, tau), zs=zs,
        inv=saved[off_inv:off_inv + m * 4].view(torch.float32).clone(),
        stat=saved[off_stat:off_stat + m * 4].view(torch.float32).clone(),
        dacc=ws[dacc_off:dacc_off + m * dpad * 4].view(torch.float32).view(m, dpad).clone(),
        dzi=dzi, dzj=dzj, bi=bi, bj=bj, go=go, loss=loss.clone(), zi=zi, zj=zj)


# ------------------------------------------------------------------------------------------------ witnesses
def weights(zs, rows, rowstat, colstat, mode, c, dtype):
    """W[rows, :] (diagonal zeroed) from the staged rows and the statistics, in `dtype`."""
    s = zs[rows].to(dtype) @ zs.to(dtype).T
    if mode == FIXED:
        w = torch.exp2(s) * (rowstat[rows].to(dtype)[:, None] + colstat.to(dtype)[None, :])
    else:
        t = c * s
        w = torch.exp2(t - rowstat[rows].to(dtype)[:, None]) + torch.exp2(t - colstat.to(dtype)[None, :])
    w[torch.arange(len(rows), device=zs.device), rows] = 0.0
    return w


def acc_witness(zs, rows, rowstat, colstat, mode, c, chunk=4096):
    """(dacc witness [len(rows) x dpad], rho [len(rows)]) in fp64 for small M, chunked fp32 otherwise."""
    dtype = torch.float64 if zs.shape[0] <= 8192 else torch.float32
    zsd = zs.to(dtype)
    sq = (zsd * zsd).sum(1)
    wit = torch.empty(len(rows), zs.shape[1], dtype=torch.float64, device=zs.device)
    rho = torch.empty(len(rows), dtype=torch.float64, device=zs.device)
    for r0 in range(0, len(rows), chunk):
        w = weights(zs, rows[r0:r0 + chunk], rowstat, colstat, mode, c, dtype)
        wit[r0:r0 + chunk] = (w @ zsd).double()
        rho[r0:r0 + chunk] = ((w * w) @ sq).double().sqrt()
        del w
    return wit, rho


def row_metric(got, wit, rho):
    return (got.double() - wit).norm(dim=1) / rho


def one_tile_metric(got, wit, rho, zs, rows, rowstat, colstat, mode, c, seed):
    """Max metric of the kernel against the witness with ONE 128 x 128 tile removed (row block of the local rows and
    column block chosen by the seed)."""
    nrb, ncb = cdiv(len(rows), 128), cdiv(zs.shape[0], 128)
    rb, cb = seed % nrb, (seed // 7 + 1) % ncb
    sel = torch.arange(rb * 128, min(len(rows), rb * 128 + 128), device=zs.device)
    w = weights(zs, rows[sel], rowstat, colstat, mode, c, torch.float64)
    tile = w[:, cb * 128:cb * 128 + 128] @ zs[cb * 128:cb * 128 + 128].double()
    return row_metric(got[sel], wit[sel] - tile, rho[sel]).max().item()


def check_acc(got, wit, rho, tol, what, power):
    assert torch.isfinite(got).all(), f"{what}: non-finite accumulator entries (a row block or column half never stored)"
    err = row_metric(got, wit, rho)
    worst = err.max().item()
    print(f"{what}: max row metric {worst:.3e} (row {int(err.argmax())}), one-tile {power:.3e}, tol {tol:.1e}")
    assert worst <= tol, f"{what}: max per-row accumulator error {worst:.3e} > {tol:.1e} (row {int(err.argmax())})"
    assert power >= 10 * tol, f"{what}: one missing tile moves the metric only to {power:.3e} (< 10 x {tol:.1e})"
    return worst


def acc_tol(normalize):
    return ACC_TOL_F16 if normalize else ACC_TOL_BF16


# ------------------------------------------------------------------------------------------------ 1. backward accumulator
# (n, d, tau, normalize): M = 2n rows, R = ceil(M / 128) row blocks, KB = dpad / 64
ACC_CASES = [
    (32, 32, 0.5, True),      # R = 1, KB = 1 (DP = 64: two draining warpgroups)
    (100, 64, 0.05, True),    # R = 2 ragged, KB = 1, FIXED at tau = 0.05
    (150, 96, 0.5, True),     # R = 3 ragged, KB = 2, d padded to 128
    (300, 128, 0.05, True),   # R = 5, KB = 2
    (200, 192, 0.5, True),    # KB = 4: two dhalf launches writing column halves
    (129, 256, 0.05, True),   # KB = 4, R = 3 ragged
    (300, 128, 0.02, True),   # ONLINE, fp16 weights (normalised rows, tau below the FIXED range)
    (100, 128, 1.0, False),   # ONLINE, bf16 weights (raw rows)
    (1050, 128, 0.5, True),   # R = 17: nchunks > 1 (red.add), 17 tiles not a multiple of the chunk count
    (1050, 64, 0.5, False),   # nchunks > 1, KB = 1, ONLINE bf16
    (1050, 256, 0.1, True),   # nchunks > 1, KB = 4
    (4100, 128, 0.02, True),  # R = 65, ONLINE
    (32768, 128, 0.5, True),  # headline: M = 65536, d = 128, tau = 0.5
]


def test_acc_cases_reach_both_chunk_regimes(C):
    sms = num_sms()
    plans = [bwd_plan(2 * n, 2 * n, sms) for n, _, _, _ in ACC_CASES]
    assert any(nch == 1 for _, nch in plans), plans
    assert any(nch > 1 for _, nch in plans), plans
    assert any(nch > 1 and cdiv(2 * n, 128) % nch for (n, _, _, _), (_, nch) in zip(ACC_CASES, plans)), plans


@pytest.mark.parametrize("n,d,tau,normalize", ACC_CASES)
def test_bwd_accumulator_rows(C, n, d, tau, normalize):
    seed = n + d
    zi, zj = inputs(n, d, seed, normalize, tau)
    r = run_ntx(C, zi, zj, tau, normalize)
    zs, stat, mode, c = r["zs"], r["stat"], r["mode"], LOG2E / tau
    rows = torch.arange(r["m"], device="cuda")
    wit, rho = acc_witness(zs, rows, stat, stat, mode, c)
    power = one_tile_metric(r["dacc"], wit, rho, zs, rows, stat, stat, mode, c, seed)
    _, nch = bwd_plan(r["m"], r["m"], num_sms())
    check_acc(r["dacc"], wit, rho, acc_tol(normalize), f"n={n} d={d} tau={tau} norm={normalize} nchunks={nch}", power)


# ------------------------------------------------------------------------------------------------ 2. gradient finish
def finish_witness(r):
    """ntx_grad_finish_kernel restated in fp64 from the kernel's own dacc, staged partner rows and inv_norm."""
    n, d, m, tau = r["n"], r["d"], r["m"], r["tau"]
    fixed = r["mode"] == FIXED
    c = LOG2E / tau
    prescale = math.sqrt(c) if fixed else 1.0
    wscale = wscale_of(m) if fixed else 1.0
    acc = r["dacc"][:, :d].double()
    partner = torch.cat([torch.arange(n, m), torch.arange(0, n)]).cuda()
    zp = r["zs"][partner, :d].double()
    g = (acc / (wscale * prescale) - 2.0 * zp / prescale) * (r["go"] / (m * tau))
    z = torch.cat([r["zi"], r["zj"]]).double()
    inv = r["inv"].double()[:, None] if r["normalize"] else torch.ones(m, 1, dtype=torch.float64, device="cuda")
    zh = z * inv
    scale = (g * inv).norm(dim=1)  # the size of the fp32 operations of the row
    if r["normalize"]:
        g = (g - (g * zh).sum(1, keepdim=True) * zh) * inv
    return g, scale


@pytest.mark.parametrize("n,d,tau,normalize,go,ld_in,ld_out", [
    (300, 36, 0.5, True, 0.75, 48, 40),     # FIXED, first float4 half partial
    (260, 200, 0.1, True, -1.3, 212, 204),  # FIXED, second float4 half partial
    (200, 200, 1.0, False, -1.3, 204, 216),  # ONLINE raw rows (bf16 partner rows)
    (100, 36, 0.02, True, 2.0, 40, 44),     # ONLINE normalised
])
def test_grad_finish_rows(C, n, d, tau, normalize, go, ld_in, ld_out):
    sentinel = -7.25
    zi, zj = inputs(n, d, n + 1, normalize, tau, ld=ld_in)
    r = run_ntx(C, zi, zj, tau, normalize, go=go, out_ld=ld_out, sentinel=sentinel)
    ref, scale = finish_witness(r)
    got = torch.cat([r["dzi"], r["dzj"]]).double()
    assert torch.isfinite(got).all()
    err = ((got - ref).norm(dim=1) / scale).max().item()
    print(f"finish n={n} d={d} go={go}: max row error {err:.3e}")
    assert err <= FINISH_TOL, f"gradient finish: max per-row error {err:.3e} > {FINISH_TOL:.1e}"
    for b in (r["bi"], r["bj"]):
        assert (b[:, d:] == sentinel).all(), "the finish kernel wrote past column d"


# ------------------------------------------------------------------------------------------------ 3./4. row stripes
def run_dist(C, world, n, d, normalize, tau, seed):
    """prep -> rows_fwd for every emulated rank into one zhat_all / stat_all, then rows_bwd per rank with a NaN-filled
    workspace; returns the staged rows, stat_all and every rank's accumulator [2n x dpad]."""
    L = C.lib()
    zi, zj = inputs(world * n, d, seed, normalize, tau)
    m, lr = 2 * n * world, 2 * n
    mpad, dpad = int(L.ssvb_ntxent_mpad(n * world)), int(L.ssvb_ntxent_dpad(d))
    wsb = int(L.ssvb_ntxent_dist_workspace_bytes(world, n, d))
    dacc_off, total = ws_dacc_offset(lr, m, dpad, num_sms())
    assert total == wsb, f"workspace layout restated as {total} bytes, library says {wsb}"
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    zhat = torch.zeros(mpad, dpad, dtype=staged_dtype(normalize), device="cuda")
    stat_all = torch.empty(world, 2, lr, device="cuda")
    inv = [torch.empty(lr, device="cuda") for _ in range(world)]
    pos = [torch.empty(lr, device="cuda") for _ in range(world)]
    sums = torch.zeros(world, device="cuda")
    st = C.stream_ptr()
    sl = [slice(r * n, (r + 1) * n) for r in range(world)]
    for r in range(world):
        C.check(L.ssvb_ntxent_dist_prep(C.ptr(zi[sl[r]]), C.ptr(zj[sl[r]]), n, d, d, d, int(normalize), ctypes.c_float(tau),
                                        world, r, C.ptr(zhat), C.ptr(inv[r]), C.ptr(pos[r]), st), "dist_prep")
    for r in range(world):
        C.check(L.ssvb_ntxent_dist_rows_fwd(C.ptr(zhat), world, r, n, d, int(normalize), ctypes.c_float(tau), C.ptr(pos[r]),
                                            C.ptr(stat_all[r]), C.ptr(sums[r:]), C.ptr(ws), wsb, st), "rows_fwd")
    gout = torch.full((1,), 1.5, device="cuda")
    dacc = []
    for r in range(world):
        ws.fill_(0xFF)
        dzi, dzj = torch.empty(n, d, device="cuda"), torch.empty(n, d, device="cuda")
        C.check(L.ssvb_ntxent_dist_rows_bwd(C.ptr(zi[sl[r]]), C.ptr(zj[sl[r]]), n, d, d, d, int(normalize),
                                            ctypes.c_float(tau), world, r, C.ptr(zhat), C.ptr(stat_all), C.ptr(inv[r]),
                                            C.ptr(gout), C.ptr(dzi), C.ptr(dzj), d, d, C.ptr(ws), wsb, st), "rows_bwd")
        dacc.append(ws[dacc_off:dacc_off + lr * dpad * 4].view(torch.float32).view(lr, dpad).clone())
    torch.cuda.synchronize()
    return zhat[:m].float(), stat_all, dacc


DIST_CASES = [
    (2, 100, 128, True, 0.5),    # FIXED, 2L = 200: rank 1's diagonal starts at column 200 (inside a 64-column half)
    (3, 150, 96, False, 1.0),    # ONLINE bf16, ragged
    (4, 96, 64, True, 0.02),     # ONLINE fp16, KB = 1
    (8, 64, 128, True, 0.5),     # FIXED, 2L = 128
    (4, 1050, 128, True, 0.5),   # FIXED, 17 row blocks per rank, nchunks > 1
]


@pytest.mark.parametrize("world,n,d,normalize,tau", DIST_CASES)
def test_dist_rows_bwd_accumulator(C, world, n, d, normalize, tau):
    seed = 10 * world + n
    zs, stat_all, dacc = run_dist(C, world, n, d, normalize, tau, seed)
    mode, c, lr, m = ntx_mode(normalize, tau), LOG2E / tau, 2 * n, 2 * n * world
    l2 = stat_all[:, 0, :].reshape(-1)
    # the column statistic exactly as dist_stat_kernel derives it (shift = 0 in FIXED mode)
    stat = wscale_of(m) * torch.exp2(-l2) if mode == FIXED else l2
    for r in range(world):
        rows = torch.arange(r * lr, (r + 1) * lr, device="cuda")
        wit, rho = acc_witness(zs, rows, stat, stat, mode, c)
        power = one_tile_metric(dacc[r], wit, rho, zs, rows, stat, stat, mode, c, seed + r)
        check_acc(dacc[r], wit, rho, acc_tol(normalize), f"world={world} rank={r} n={n} d={d} tau={tau}", power)


def lse2_witness(zs, rows, mode, c, chunk=4096):
    """log2-domain LSE over b != a of the logit the forward sees (FIXED: zs_a . zs_b, ONLINE: c zs_a . zs_b), fp64."""
    out = torch.empty(len(rows), dtype=torch.float64, device=zs.device)
    zd = zs.double()
    for r0 in range(0, len(rows), chunk):
        rr = rows[r0:r0 + chunk]
        t = zd[rr] @ zd.T
        if mode == ONLINE:
            t = t * c
        t[torch.arange(len(rr), device=zs.device), rr] = -math.inf
        out[r0:r0 + chunk] = torch.logsumexp(t * math.log(2.0), dim=1) / math.log(2.0)
    return out


@pytest.mark.parametrize("world,n,d,normalize,tau", DIST_CASES)
def test_dist_rows_fwd_statistic(C, world, n, d, normalize, tau):
    zs, stat_all, _ = run_dist(C, world, n, d, normalize, tau, 10 * world + n)
    mode, c, lr = ntx_mode(normalize, tau), LOG2E / tau, 2 * n
    for r in range(world):
        rows = torch.arange(r * lr, (r + 1) * lr, device="cuda")
        err = (stat_all[r, 0].double() - lse2_witness(zs, rows, mode, c)).abs()
        print(f"rows_fwd world={world} rank={r}: max |lse2 error| {err.max().item():.3e}")
        assert err.max().item() <= LSE_TOL, f"rank {r}: max per-row lse2 error {err.max().item():.3e} (row {int(err.argmax())})"


# ------------------------------------------------------------------------------------------------ 4. full-matrix forward
@pytest.mark.parametrize("n,d,tau,normalize", [(300, 128, 0.02, True), (1050, 64, 0.02, True), (100, 128, 1.0, False),
                                               (4100, 96, 1.0, False)])
def test_fwd_statistic_online_rows(C, n, d, tau, normalize):
    zi, zj = inputs(n, d, n + d, normalize, tau)
    r = run_ntx(C, zi, zj, tau, normalize)
    assert r["mode"] == ONLINE
    rows = torch.arange(r["m"], device="cuda")
    err = (r["stat"].double() - lse2_witness(r["zs"], rows, ONLINE, LOG2E / tau)).abs()
    print(f"fwd ONLINE n={n} d={d} tau={tau}: max |lse2 error| {err.max().item():.3e}")
    assert err.max().item() <= LSE_TOL, f"max per-row lse2 error {err.max().item():.3e} (row {int(err.argmax())})"


@pytest.mark.parametrize("n,d,tau", [(200, 192, 0.5), (129, 256, 0.05), (1050, 256, 0.1)])
def test_fwd_statistic_fixed_dpad256_rows(C, n, d, tau):
    zi, zj = inputs(n, d, n + d, True, tau)
    r = run_ntx(C, zi, zj, tau, True)
    assert r["mode"] == FIXED and r["dpad"] == 256
    rows = torch.arange(r["m"], device="cuda")
    l_ref = torch.exp2(lse2_witness(r["zs"], rows, FIXED, 1.0))
    err = (wscale_of(r["m"]) / r["stat"].double() / l_ref - 1.0).abs()
    print(f"fwd FIXED dpad=256 n={n} d={d} tau={tau}: max |L/L_ref - 1| {err.max().item():.3e}")
    assert err.max().item() <= LREL_TOL, f"max per-row relative error of L {err.max().item():.3e}"


# ------------------------------------------------------------------------------------------------ 5. fused MoCo
def unit_rows(x):
    return x / x.norm(dim=1, keepdim=True)


def run_moco(C, n, k, d, tau, zero_rows, seed):
    L = C.lib()
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(n, d, generator=g).cuda()
    kk = (q.cpu() + 0.7 * torch.randn(n, d, generator=g)).cuda()
    dpad = int(L.ssvb_ntxent_dpad(d))
    mem = unit_rows(torch.randn(k, d, generator=g)).cuda()
    mem[:zero_rows] = 0.0
    qb = torch.zeros(k, dpad, dtype=torch.bfloat16, device="cuda")  # the test's own bf16 staging of the queue
    qb[:, :d] = mem.to(torch.bfloat16)
    sb, wsb = int(L.ssvb_moco_saved_bytes(n, k, d)), int(L.ssvb_moco_workspace_bytes(n, k, d))
    saved = torch.full((sb,), 0xFF, dtype=torch.uint8, device="cuda")  # NaN sentinel: rows never written stay NaN
    ws = torch.full((wsb,), 0xFF, dtype=torch.uint8, device="cuda")
    loss = torch.empty(1, device="cuda")
    st = C.stream_ptr()
    C.check(L.ssvb_moco_fwd(C.ptr(q), C.ptr(kk), None, C.ptr(qb), 1, n, k, d, d, d, d, 1, ctypes.c_float(tau),
                            C.ptr(loss), C.ptr(saved), C.ptr(ws), wsb, st), "ssvb_moco_fwd")
    gout = torch.full((1,), -0.8, device="cuda")
    dq, dk = torch.empty(n, d, device="cuda"), torch.empty(n, d, device="cuda")
    C.check(L.ssvb_moco_bwd(C.ptr(q), C.ptr(kk), None, C.ptr(qb), 1, n, k, d, d, d, d, 1, ctypes.c_float(tau),
                            C.ptr(gout), C.ptr(saved), C.ptr(dq), C.ptr(dk), d, d, C.ptr(ws), wsb, st), "ssvb_moco_bwd")
    torch.cuda.synchronize()
    # moco.cu moco_saved: qhat bf16 [npad x dpad], inv_q, inv_k, pos, lse2 [npad] fp32, pm fp32 [npad x dpad]
    npad = ru(n, 128)
    offs, off = [], 0
    for nbytes in (npad * dpad * 2, npad * 4, npad * 4, npad * 4, npad * 4, npad * dpad * 4):
        off = ru(off, 256)
        offs.append(off)
        off += nbytes
    assert ru(off, 256) == sb, "moco saved layout changed"
    f32 = lambda i, cnt: saved[offs[i]:offs[i] + cnt * 4].view(torch.float32)
    return dict(q=q, kk=kk, qb=qb, c=LOG2E / tau, tau=tau, go=-0.8, dq=dq, dk=dk,
                qh=saved[:n * dpad * 2].view(torch.bfloat16).view(n, dpad).float(),
                inv_q=f32(1, n).clone(), inv_k=f32(2, n).clone(), pos=f32(3, n).clone(), lse2=f32(4, n).clone(),
                pm=f32(5, n * dpad).view(n, dpad).clone())


def moco_witness(r, drop_tile=None):
    """fp64: E_aj = exp2(c s_aj - c), L_a = sum_j E_aj + exp2(c pos_a - c), lse2 = c + log2 L, pm = sum_j E_aj m_j / L."""
    c = r["c"]
    mb = r["qb"].double()
    e = torch.exp2(c * (r["qh"].double() @ mb.T) - c)
    if drop_tile is not None:
        e[:, drop_tile * 128:drop_tile * 128 + 128] = 0.0
    lsum = e.sum(1) + torch.exp2(c * r["pos"].double() - c)
    p = e / lsum[:, None]
    return c + torch.log2(lsum), p @ mb, ((p * p) @ (mb * mb).sum(1)).sqrt()


@pytest.mark.parametrize("n,k,d,tau,zero_rows", [
    (256, 65536, 128, 0.07, 0),   # cfg2
    (200, 4100, 128, 0.07, 0),    # n not a multiple of 128, queue tail inside a tile
    (256, 4100, 64, 0.2, 37),     # zero queue rows
    (100, 16384, 128, 0.07, 5),
])
def test_moco_fused_rows(C, n, k, d, tau, zero_rows):
    r = run_moco(C, n, k, d, tau, zero_rows, seed=n + k)
    lse_w, pm_w, rho = moco_witness(r)
    assert torch.isfinite(r["lse2"]).all() and torch.isfinite(r["pm"]).all()
    e_lse = (r["lse2"].double() - lse_w).abs()
    e_pm = (r["pm"].double() - pm_w).norm(dim=1) / rho
    # one queue tile (seed-chosen) removed from the witness
    tile = (n + k) % cdiv(k, 128)
    lse_p, pm_p, _ = moco_witness(r, drop_tile=tile)
    p_lse = (r["lse2"].double() - lse_p).abs().max().item()
    p_pm = ((r["pm"].double() - pm_p).norm(dim=1) / rho).max().item()
    print(f"moco n={n} k={k}: max |lse2 error| {e_lse.max().item():.3e} (one tile {p_lse:.3e}), "
          f"max pm row metric {e_pm.max().item():.3e} (one tile {p_pm:.3e})")
    assert e_lse.max().item() <= MOCO_LSE_TOL, f"max per-row lse2 error {e_lse.max().item():.3e} (row {int(e_lse.argmax())})"
    assert e_pm.max().item() <= MOCO_PM_TOL, f"max per-row pm error {e_pm.max().item():.3e} (row {int(e_pm.argmax())})"
    assert p_lse >= 10 * MOCO_LSE_TOL and p_pm >= 10 * MOCO_PM_TOL, f"one missing queue tile: {p_lse:.3e}, {p_pm:.3e}"
    # gradient finish (moco_grad_finish_kernel) restated from the saved blob
    c, scale = r["c"], r["go"] / (n * r["tau"])
    qh = r["q"].double() * r["inv_q"].double()[:, None]
    kh = r["kk"].double() * r["inv_k"].double()[:, None]
    # p_a0 - 1 as the kernel evaluates it: fmaf(pos, c, -lse2) and exp2 in fp32.  Near p_a0 = 1 the subtraction
    # cancels, so one ulp of the fp32 exponent alone moves p_a0 - 1 by ~1e-5 relative (1.3e-5 at n = 200, K = 4100
    # against an fp64 exponent; 1.2e-7 with this one)
    c32 = (torch.tensor(LOG2E, dtype=torch.float32) / torch.tensor(r["tau"], dtype=torch.float32)).double()
    arg = (r["pos"].double() * c32 - r["lse2"].double()).float()
    p0m1 = (torch.exp2(arg) - 1.0).double()[:, None]
    gq = (p0m1 * kh + r["pm"][:, :d].double()) * scale
    gk = p0m1 * qh * scale
    den_q, den_k = (gq * r["inv_q"].double()[:, None]).norm(dim=1), (gk * r["inv_k"].double()[:, None]).norm(dim=1)
    gq = (gq - (gq * qh).sum(1, keepdim=True) * qh) * r["inv_q"].double()[:, None]
    gk = (gk - (gk * kh).sum(1, keepdim=True) * kh) * r["inv_k"].double()[:, None]
    eq = ((r["dq"].double() - gq).norm(dim=1) / den_q).max().item()
    ek = ((r["dk"].double() - gk).norm(dim=1) / den_k).max().item()
    print(f"moco finish: dq {eq:.3e} dk {ek:.3e}")
    assert eq <= MOCO_GRAD_TOL and ek <= MOCO_GRAD_TOL, (eq, ek)


# ------------------------------------------------------------------------------------------------ 6. determinism
@pytest.mark.parametrize("n,d,tau,normalize", [(300, 128, 0.5, True), (4100, 128, 0.5, True), (1050, 256, 0.1, True)])
def test_bwd_run_to_run(C, n, d, tau, normalize):
    zi, zj = inputs(n, d, 5, normalize, tau)
    a = run_ntx(C, zi, zj, tau, normalize)
    b = run_ntx(C, zi, zj, tau, normalize)
    _, nch = bwd_plan(a["m"], a["m"], num_sms())
    bitwise = torch.equal(a["dacc"], b["dacc"])
    if nch == 1:  # plain stores, fixed order inside the tensor-core accumulator
        assert bitwise and torch.equal(a["dzi"], b["dzi"]) and torch.equal(a["dzj"], b["dzj"])
        return
    # nchunks > 1: float red.add of the chunk partials (DESIGN §3 allows atomics on gradient accumulators)
    rows = torch.arange(a["m"], device="cuda")
    _, rho = acc_witness(a["zs"], rows, a["stat"], a["stat"], a["mode"], LOG2E / tau)
    diff = row_metric(a["dacc"], b["dacc"].double(), rho).max().item()
    print(f"run-to-run n={n} d={d} nchunks={nch}: bit-identical {bitwise}, max row difference {diff:.3e}")
    assert diff <= ATOMIC_TOL, f"run-to-run accumulator difference {diff:.3e} > {ATOMIC_TOL:.1e}"
