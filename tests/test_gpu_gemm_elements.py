"""Per-element checks of the tcgen05 GEMM (csrc/gemm_kernels.cuh) behind Barlow Twins and SwAV.

The oracle tests compare these losses as whole tensors (loss rel <= 1e-3, gradient rel-L2 <= 1e-2).  A wrong tile of
a 2048 x 8192 gradient moves that metric very little, and at the Barlow headline shape the inherent bf16 error already
uses half of the gradient tolerance.  These tests drive the C ABI with their own buffers and check EVERY element of
every GEMM output against a witness: the fp64 product of the library's own staged 16-bit operands, read back from the
`saved` / `workspace` buffers (whose carving is restated here and checked against the library's byte counts), scaled
by the same fp32 alpha.

Metric: |got - ref| / rho per element, rho = |alpha| * sum_k |a_k b_k| (the fp64 product of |A| and |B|), the natural
scale of fp32 accumulation of exact bf16 products; maximised over all elements, arg-max reported.  Every metric test
also removes one 64-wide K block (split-K: one K slice) of one seed-chosen output tile from the witness and asserts that
the kernel's metric against that perturbed witness is at least 10x the tolerance.

Before each call `saved`, `workspace` and every output are NaN-filled: an element the library must write and did not is
non-finite, and columns outside [0, N) of an output row (the gradient row padding, the tail after a dC slab) must
still hold the sentinel.  The one region written by the hardware beyond N, the SwAV score padding [k, kpad) inside
the last 16-byte piece of a row, is restated in `check_swav_scores`.

The persistent schedule's hard parts (several units per CTA: TMEM accumulator and staging-buffer parity wraps; K-block
counts that are not a multiple of the smem ring depth; split-K with a short last slice) only run at some shapes; the
GEMM plan is restated here and `test_plan_reaches_every_regime` asserts that the parameter lists reach each of them on
the GPU the suite runs on.

Tolerances are about 3x the maxima measured on one B200 (profiles/r5_gemm_elements.md) and each test asserts its
one-block effect to be at least 10x the tolerance.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "self-supervised-vision_b200")

# tolerances (profiles/r5_gemm_elements.md lists the measured maximum of every shape)
GEMM_TOL = 2e-5      # fp32 GEMM outputs, |got - ref| / rho per element: measured <= 6.3e-6 (K = 7024 unsplit)
DC_TOL = 5e-7        # Barlow dC beyond its bf16 rounding, |.| / (2 w rho): measured <= 1.5e-7 (cfg3)
LOSS_TOL = 4e-5      # Barlow loss against the fp64 loss of the same staged operands, relative: measured <= 1.3e-5
Q_TOL = 1.2e-6       # q_i / q_j (dC .* C row / column partials + finish), relative to their own scale: <= 4.1e-7
PART_TOL = 2e-6      # backward column partials per stripe, relative to the sum of |terms|: 31 x 2^-24 bounds 32 rows
FINISH_TOL = 1.5e-7  # finished Barlow gradient (normalize = 1) restated from the library's own dT and partials: <= 4.9e-8

LAMBDA = 0.005
K_STAT_SPLIT, K_ROW_SPLIT, K_MAX_FUSED_STRIPES, K_MAX_GEMM_CTAS = 32, 8, 256, 160  # csrc/barlow.cu


@pytest.fixture(scope="module")
def C():
    assert torch.cuda.is_available()
    from ssv_b200 import _cabi
    assert _cabi.lib().ssvb_device_check() == 0, "not a B200"
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False  # rho is an fp32 product of |A| and |B|
    yield _cabi
    torch.backends.cuda.matmul.allow_tf32 = prev


# ------------------------------------------------------------------------------------------------ layouts, restated
def ru(x, a):
    return (x + a - 1) // a * a


def cdiv(a, b):
    return (a + b - 1) // b


def carve(pieces):
    """host_util.h Carver: every piece starts at a 256-byte boundary; (offsets by name, total bytes)."""
    offs, off = {}, 0
    for name, nbytes in pieces:
        off = ru(off, 256)
        offs[name] = off
        off += nbytes
    return offs, ru(off, 256)


def fused_stripes(n):
    t = cdiv(n, 128) * 4
    return t if t <= K_MAX_FUSED_STRIPES else 0


def barlow_saved_layout(n, d):
    return carve([("xi", n * d * 2), ("xj", n * d * 2), ("dC", d * d * 2), ("mean_i", d * 4), ("rstd_i", d * 4),
                  ("mean_j", d * 4), ("rstd_j", d * 4), ("inv_i", n * 4), ("inv_j", n * 4), ("q_i", d * 4),
                  ("q_j", d * 4)])


def barlow_ws_layout(n, d):
    stripes = max(K_STAT_SPLIT, K_ROW_SPLIT, fused_stripes(n))
    offs, total = carve([("colpart", 2 * stripes * 2 * d * 4), ("loss_partials", K_MAX_GEMM_CTAS * 4),
                         ("dti", n * d * 4), ("dtj", n * d * 4), ("colred", 4 * d * 4),
                         ("xrow", cdiv(d, 256) * d * 4), ("xcol", cdiv(d, 128) * 4 * d * 4)])
    offs["view_stride"] = stripes * 2 * d  # floats between the two views' column partials
    return offs, total


def barlow_dist_saved_layout(n, d):
    return carve([("xi", n * d * 2), ("xj", n * d * 2), ("mean_i", d * 4), ("rstd_i", d * 4), ("mean_j", d * 4),
                  ("rstd_j", d * 4), ("inv_i", n * 4), ("inv_j", n * 4)])


def swav_dims(nb, nbank, k, d):
    return dict(bp=nb + nbank, dpad=ru(d, 8), kp4=ru(k, 4), kp8=ru(k, 8))


def swav_saved_layout(nb, nbank, k, d):
    m = swav_dims(nb, nbank, k, d)
    return carve([("z", 2 * m["bp"] * m["dpad"] * 2), ("c", k * m["dpad"] * 2), ("ds", 2 * m["bp"] * m["kp8"] * 2)])


def swav_ws_layout(L, nb, nbank, k, d):
    m = swav_dims(nb, nbank, k, d)
    return carve([("scores", 2 * m["bp"] * m["kp4"] * 4), ("codes", 2 * m["bp"] * m["kp4"] * 4),
                  ("loss_part", m["bp"] * 4), ("dz", 2 * m["bp"] * m["dpad"] * 4), ("dc", k * m["dpad"] * 4),
                  ("sk", int(L.ssvb_sinkhorn_workspace_bytes(m["bp"], k)))])


def piece(buf, offs, name, dtype, shape):
    esz = torch.empty(0, dtype=dtype).element_size()
    numel = int(np.prod(shape))
    return buf[offs[name]:offs[name] + numel * esz].view(dtype).view(*shape)


def nan_bytes(nbytes):
    return torch.full((max(int(nbytes), 16),), 0xFF, dtype=torch.uint8, device="cuda")  # NaN in fp32 and bf16


def nan_f32(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device="cuda")


# ------------------------------------------------------------------------------------------------ GEMM plan, restated
def num_sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def gemm_plan(M, N, K, bn, sms, dual=False, split=False, max_ctas=0):
    """gemm_host.cuh: tile counts, gemm_plan_splits and gemm_grid of one launch."""
    tiles = cdiv(M, 128) * cdiv(N, bn)
    nkb = cdiv(K, 64)
    splits = 1
    if split and tiles * 2 <= sms:
        splits = max(min(sms // tiles, nkb // 4), 1)
    kb_per = cdiv(nkb, splits)
    splits = cdiv(nkb, kb_per)
    units = tiles * (2 if dual else 1) * splits
    grid = min(units, sms)
    if max_ctas > 0:
        grid = min(grid, max_ctas)
    return dict(M=M, N=N, K=K, bn=bn, tiles=tiles, nkb=nkb, splits=splits, kb_per=kb_per,
                last=nkb - (splits - 1) * kb_per, units=units, grid=grid)


def barlow_fwd_plan(n, d, sms):
    return gemm_plan(d, d, n, 256, sms, max_ctas=K_MAX_GEMM_CTAS)


def barlow_bwd_plan(n, d, sms):
    return gemm_plan(n, d, d, 256, sms, dual=True)


def xcorr_plan(n_local, d, sms):
    return gemm_plan(d, d, n_local, 256, sms)


def scores_plan(nb, nbank, k, d, sms):
    m = swav_dims(nb, nbank, k, d)
    return gemm_plan(2 * m["bp"], k, m["dpad"], 256, sms)


def swav_bwd_plans(nb, nbank, k, d, sms, tma_store=True):
    """(dz plan, dproto plan); split-K needs the staged TMA-store epilogue (gemm_will_split)."""
    m = swav_dims(nb, nbank, k, d)
    return (gemm_plan(2 * m["bp"], m["dpad"], k, 128, sms, split=tma_store),
            gemm_plan(k, m["dpad"], 2 * m["bp"], 128, sms, split=tma_store))


# ------------------------------------------------------------------------------------------------ metric machinery
def f32(x):
    return float(np.float32(x))


def absmm(a, b):
    """|a| @ |b| in fp32 (TF32 off): the scale rho, not the witness."""
    return (a.abs().float() @ b.abs().float()).double()


def max_metric(err):
    """(max, (row, col)) of a 2-D metric; a non-finite entry is reported as infinite."""
    err = torch.where(torch.isfinite(err), err, torch.full_like(err, float("inf")))
    i = int(err.argmax())
    return err.view(-1)[i].item(), (i // err.shape[1], i % err.shape[1]) if err.dim() == 2 else (i,)


def check_metric(err, tol, what, power):
    assert power is not None
    worst, at = max_metric(err)
    print(f"{what}: max metric {worst:.3e} at {at}, one block {power:.3e}, tol {tol:.1e}")
    assert worst <= tol, f"{what}: max per-element error {worst:.3e} > {tol:.1e} at (row, col) = {at}"
    assert power >= 10 * tol, f"{what}: one missing K block moves the metric only to {power:.3e} (< 10 x {tol:.1e})"
    return worst


def pick_tile(plan, seed):
    """A seed-chosen output tile (tm, tn) and K block range [kb0, kb1) of one unit (split-K: one K slice)."""
    tm = seed % cdiv(plan["M"], 128)
    tn = (seed // 3 + 1) % cdiv(plan["N"], plan["bn"])
    if plan["splits"] > 1:
        s = (seed // 5) % plan["splits"]
        return tm, tn, s * plan["kb_per"], min(plan["nkb"], (s + 1) * plan["kb_per"])
    kb = (seed // 7) % plan["nkb"]
    return tm, tn, kb, kb + 1


def tile_slices(plan, tm, tn, kb0, kb1):
    return (slice(tm * 128, min(plan["M"], tm * 128 + 128)), slice(tn * plan["bn"], min(plan["N"], tn * plan["bn"] + plan["bn"])),
            slice(kb0 * 64, min(plan["K"], kb1 * 64)))


def gemm_check(got, a64, b64, alpha, plan, seed, what, tol=GEMM_TOL):
    """got [M x N] fp32 against alpha * a64 @ b64 (a64 [M x K], b64 [K x N], the staged operands in fp64)."""
    assert got.shape == (plan["M"], plan["N"]), (got.shape, plan)
    ref = (a64 @ b64) * alpha
    rho = absmm(a64, b64) * abs(alpha)
    err = (got.double() - ref).abs() / rho
    rs, cs, ks = tile_slices(plan, *pick_tile(plan, seed))
    blk = (a64[rs, ks] @ b64[ks, cs]) * alpha
    power = ((got[rs, cs].double() - (ref[rs, cs] - blk)).abs() / rho[rs, cs]).max().item()
    return check_metric(err, tol, what, power)


def c_api(C):
    return C.lib(), C.stream_ptr()


# ------------------------------------------------------------------------------------------------ Barlow runs
def barlow_inputs(n, d, seed, ld=None):
    g = torch.Generator().manual_seed(seed)
    zi = torch.randn(n, d, generator=g) * 1.3 + 0.2
    zj = 0.7 * zi + 0.3 * torch.randn(n, d, generator=g)
    if ld is None:
        return zi.cuda(), zj.cuda()
    bi, bj = torch.full((n, ld), float("nan")), torch.full((n, ld), float("nan"))
    bi[:, :d], bj[:, :d] = zi, zj
    return bi.cuda()[:, :d], bj.cuda()[:, :d]


def run_barlow_fwd(C, zi, zj, normalize):
    L, st = c_api(C)
    n, d = zi.shape
    so, stotal = barlow_saved_layout(n, d)
    wo, wtotal = barlow_ws_layout(n, d)
    assert stotal == int(L.ssvb_barlow_saved_bytes(n, d)), f"BarlowSaved restated as {stotal} bytes"
    assert wtotal == int(L.ssvb_barlow_workspace_bytes(n, d)), f"BarlowWs restated as {wtotal} bytes"
    saved, ws = nan_bytes(stotal), nan_bytes(wtotal)
    loss = nan_f32(1)
    C.check(L.ssvb_barlow_fwd(C.ptr(zi), C.ptr(zj), n, d, zi.stride(0), zj.stride(0), int(normalize), ctypes.c_float(LAMBDA),
                              C.ptr(loss), C.ptr(saved), C.ptr(ws), wtotal, st), "ssvb_barlow_fwd")
    torch.cuda.synchronize()
    return dict(n=n, d=d, zi=zi, zj=zj, saved=saved, ws=ws, so=so, wo=wo, loss=loss, normalize=normalize,
                xi=piece(saved, so, "xi", torch.bfloat16, (n, d)), xj=piece(saved, so, "xj", torch.bfloat16, (n, d)),
                dC=piece(saved, so, "dC", torch.bfloat16, (d, d)),
                **{k: piece(saved, so, k, torch.float32, (d,)) for k in ("mean_i", "rstd_i", "mean_j", "rstd_j", "q_i", "q_j")},
                inv_i=piece(saved, so, "inv_i", torch.float32, (n,)), inv_j=piece(saved, so, "inv_j", torch.float32, (n,)))


def run_barlow_bwd(C, r, go, pad=8):
    """ssvb_barlow_bwd after run_barlow_fwd; workspace and outputs NaN-filled, outputs [n x (d + pad)]."""
    L, st = c_api(C)
    n, d = r["n"], r["d"]
    r["ws"].fill_(0xFF)  # the backward reads only `saved`
    bi, bj = nan_f32(n, d + pad), nan_f32(n, d + pad)
    gout = torch.full((1,), go, dtype=torch.float32, device="cuda")
    C.check(L.ssvb_barlow_bwd(C.ptr(r["zi"]), C.ptr(r["zj"]), n, d, r["zi"].stride(0), r["zj"].stride(0), int(r["normalize"]),
                              ctypes.c_float(LAMBDA), C.ptr(gout), C.ptr(r["saved"]), C.ptr(bi), C.ptr(bj), d + pad, d + pad,
                              C.ptr(r["ws"]), r["ws"].numel(), st), "ssvb_barlow_bwd")
    torch.cuda.synchronize()
    for b in (bi, bj):
        assert torch.isfinite(b[:, :d]).all(), "gradient elements never written"
        assert torch.isnan(b[:, d:]).all(), "the backward wrote past column d of a gradient row"
    wo = r["wo"]
    return dict(dzi=bi[:, :d], dzj=bj[:, :d], go=go,
                dti=piece(r["ws"], wo, "dti", torch.float32, (n, d)), dtj=piece(r["ws"], wo, "dtj", torch.float32, (n, d)))


# ------------------------------------------------------------------------------------------------ 1. Barlow forward
def check_barlow_fwd(C, n, d, seed=0):
    """dC per element, the loss, q_i / q_j per column (EPI_BARLOW, bl_rowpart / bl_colpart, barlow_fwd_finish_kernel)."""
    zi, zj = barlow_inputs(n, d, seed)
    r = run_barlow_fwd(C, zi, zj, False)
    plan = barlow_fwd_plan(n, d, num_sms())
    alpha = f32(1.0 / n)
    xi, xj = r["xi"].double(), r["xj"].double()
    assert torch.isfinite(xi).all() and torch.isfinite(xj).all()
    dC = r["dC"].double()
    assert torch.isfinite(dC).all(), "dC elements never written"
    c64 = (xi.T @ xj) * alpha
    rho = absmm(xi.T, xj) * alpha
    eye = torch.eye(d, dtype=torch.bool, device="cuda")
    w2 = torch.where(eye, 2.0, 2.0 * f32(LAMBDA))                            # 2w
    g64 = w2 * torch.where(eye, c64 - 1.0, c64)
    err = ((dC - g64).abs() - 2.0 ** -8 * g64.abs()).clamp(min=0) / (w2 * rho)  # bf16 rounding of dC allowed
    rs, cs, ks = tile_slices(plan, *pick_tile(plan, seed + n))
    cb = c64[rs, cs] - (xi[ks, rs].T @ xj[ks, cs]) * alpha
    gb = w2[rs, cs] * torch.where(eye[rs, cs], cb - 1.0, cb)
    power = (((dC[rs, cs] - gb).abs() - 2.0 ** -8 * gb.abs()).clamp(min=0) / (w2[rs, cs] * rho[rs, cs])).max().item()
    what = f"barlow fwd dC n={n} d={d} units={plan['units']} grid={plan['grid']} nkb={plan['nkb']}"
    check_metric(err, DC_TOL, what, power)
    del err, g64, w2
    # loss against the fp64 loss of the same staged operands
    diag = torch.diagonal(c64)
    l64 = ((diag - 1.0) ** 2).sum() + f32(LAMBDA) * ((c64 * c64).sum() - (diag * diag).sum())
    lerr = abs(r["loss"].item() - l64.item()) / abs(l64.item())
    print(f"barlow fwd loss n={n} d={d}: {r['loss'].item():.8e} vs {l64.item():.8e}, rel {lerr:.3e}")
    assert lerr <= LOSS_TOL, f"loss rel error {lerr:.3e} > {LOSS_TOL:.1e}"
    # q_i[a] = rstd_i[a] sum_b dC[a, b] C[a, b] / (n - 1), q_j[b] likewise over a, with dC AS STORED
    gc, sc = dC * c64, dC.abs() * (c64.abs() + rho)
    inv_nm1 = f32(1.0 / (n - 1))
    ri, rj = r["rstd_i"].double() * inv_nm1, r["rstd_j"].double() * inv_nm1
    qi_ref, qj_ref = gc.sum(1) * ri, gc.sum(0) * rj
    si, sj = sc.sum(1) * ri, sc.sum(0) * rj
    qi, qj = r["q_i"].double(), r["q_j"].double()
    assert torch.isfinite(qi).all() and torch.isfinite(qj).all()
    e_q = torch.stack([(qi - qi_ref).abs() / si, (qj - qj_ref).abs() / sj])  # row 0: q_i, row 1: q_j (column = feature)
    # power: one tile's row partial (bl_rowpart of tile column tn) and one warp's column partial (bl_colpart) missing
    tm, tn = seed % cdiv(d, 128), (seed + 1) % cdiv(d, 256)
    rr, cc = slice(tm * 128, min(d, tm * 128 + 128)), slice(tn * 256, min(d, tn * 256 + 256))
    wr = slice(tm * 128 + 32 * (seed % 4), min(d, tm * 128 + 32 * (seed % 4) + 32))
    p_i = ((qi[rr] - (qi_ref[rr] - gc[rr, cc].sum(1) * ri[rr])).abs() / si[rr]).max().item()
    p_j = ((qj[cc] - (qj_ref[cc] - gc[wr, cc].sum(0) * rj[cc])).abs() / sj[cc]).max().item()
    check_metric(e_q, Q_TOL, f"barlow fwd q_i/q_j n={n} d={d} (row 0: q_i, row 1: q_j)", min(p_i, p_j))
    return r


@pytest.mark.parametrize("n,d", [
    (256, 264),     # ragged M / N: 264 = 256 + 8 (one 8-column tail tile), 3 row tiles with 8 rows in the last
    (300, 4096),    # 512 tiles (~3.5 per CTA), 5 K blocks per tile (the ring phase shifts per tile) with a K tail
    (2048, 8192),   # cfg3: all 67 M dC elements, ~14 tiles per CTA
])
def test_barlow_fwd_elements(C, n, d):
    check_barlow_fwd(C, n, d, seed=n + d)


# ------------------------------------------------------------------------------------------------ 2. Barlow fused backward
@pytest.mark.parametrize("n,d", [
    (200, 264),     # ragged M / N
    (1000, 1000),   # 16 K blocks, ragged N (1000 = 3 x 256 + 232)
    (2000, 3400),   # 448 units (~3 per CTA), 54 K blocks per tile, ragged M / N
])
def test_barlow_bwd_fused_elements(C, n, d):
    """EPI_BARLOW_BWD, DUAL: dzi / dzj per element against the epilogue formula over fp64 dT from the staged operands."""
    seed = n + d
    zi, zj = barlow_inputs(n, d, seed)
    r = run_barlow_fwd(C, zi, zj, False)
    b = run_barlow_bwd(C, r, -0.7)
    # the closed-form epilogue writes the gradients directly: the dT buffers stay untouched
    assert torch.isnan(b["dti"]).all() and torch.isnan(b["dtj"]).all(), "normalize = 0 did not take the fused epilogue"
    plan = barlow_bwd_plan(n, d, num_sms())
    alpha, go = f32(1.0 / n), f32(-0.7)
    dC = r["dC"].double()
    for name, a64, b64, x, s in (("dzi", r["xj"].double(), dC.T, zi, "i"), ("dzj", r["xi"].double(), dC, zj, "j")):
        mean, rstd, q = r["mean_" + s].double(), r["rstd_" + s].double(), r["q_" + s].double()
        t = (a64 @ b64) * alpha
        xc = x.double() - mean
        rho = (absmm(a64, b64) * alpha + xc.abs() * q.abs()) * rstd * abs(go)
        got = b[name].double()
        err = (got - (t - xc * q) * rstd * go).abs() / rho
        rs, cs, ks = tile_slices(plan, *pick_tile(plan, seed + len(s) * ord(s)))
        tb = t[rs, cs] - (a64[rs, ks] @ b64[ks, cs]) * alpha
        power = ((got[rs, cs] - (tb - xc[rs, cs] * q[cs]) * rstd[cs] * go).abs() / rho[rs, cs]).max().item()
        check_metric(err, GEMM_TOL, f"barlow bwd fused {name} n={n} d={d} units={plan['units']} nkb={plan['nkb']}", power)


# ------------------------------------------------------------------------------------------------ 3. un-fused backward
def rel_or_exact(got, ref, scale):
    """|got - ref| / scale; where scale is 0 (a fused stripe of rows beyond n: its staged rows hold zeros) the partial
    must be exactly 0."""
    e = (got - ref).abs() / scale
    return torch.where(scale > 0, e, torch.where(got == ref, 0.0, float("inf")))


def stripe_sums(vals, stripe_of, nstripes):
    out = torch.zeros(nstripes, vals.shape[1], dtype=torch.float64, device=vals.device)
    return out.index_add_(0, stripe_of, vals)


@pytest.mark.parametrize("n,d", [
    (300, 520),     # fused column partials: 12 stripes of 32 rows, ragged M / N
    (2000, 3400),   # fused column partials, 448 DUAL units (~3 per CTA)
    (8320, 136),    # fused_stripes(n) == 0: separate column reduction (col_partials_kernel, 8 stripes)
])
def test_barlow_bwd_unfused_elements(C, n, d):
    """normalize = 1: EPI_STORE_F32 DUAL into the workspace dT buffers (+ fused column partials), then the finish."""
    seed = n + d
    zi, zj = barlow_inputs(n, d, seed)
    r = run_barlow_fwd(C, zi, zj, True)
    b = run_barlow_bwd(C, r, 1.3)
    plan = barlow_bwd_plan(n, d, num_sms())
    alpha, go = f32(1.0 / n), f32(1.3)
    dC = r["dC"].double()
    nfs = fused_stripes(n)
    if nfs:
        nsplit = nfs
        stripe_of = torch.arange(n, device="cuda") // 32
    else:
        nsplit = K_ROW_SPLIT
        stripe_of = torch.arange(n, device="cuda") // cdiv(n, K_ROW_SPLIT)
    colpart = piece(r["ws"], r["wo"], "colpart", torch.float32, (2 * r["wo"]["view_stride"],))
    for v, (name, a64, b64, x, s) in enumerate([("dti", r["xj"].double(), dC.T, zi, "i"),
                                                ("dtj", r["xi"].double(), dC, zj, "j")]):
        got = b[name]
        assert torch.isfinite(got).all(), f"{name}: elements never written"
        gemm_check(got, a64, b64, alpha, plan, seed + v, f"barlow bwd unfused {name} n={n} d={d} units={plan['units']}")
        # column partials per stripe: sum dT and sum dT x~ (fused: x~ = the staged bf16 rows; separate: from fp32 rows)
        inv = r["inv_" + s].double()[:, None]
        mean, rstd = r["mean_" + s].double(), r["rstd_" + s].double()
        xt = r["x" + s].double() if nfs else (x.double() * inv - mean) * rstd
        dt = got.double()
        part = colpart[v * r["wo"]["view_stride"]:][:nsplit * 2 * d].view(nsplit, 2, d).double()
        assert torch.isfinite(part).all(), f"{name}: column partials never written"
        s1, s2 = stripe_sums(dt, stripe_of, nsplit), stripe_sums(dt * xt, stripe_of, nsplit)
        a1, a2 = stripe_sums(dt.abs(), stripe_of, nsplit), stripe_sums((dt * xt).abs(), stripe_of, nsplit)
        e_p = torch.cat([rel_or_exact(part[:, 0], s1, a1), rel_or_exact(part[:, 1], s2, a2)])
        # power: the first row of one stripe missing from that stripe's sums
        st_ = seed % nsplit
        r0 = int((stripe_of == st_).nonzero()[0])
        p1 = (part[st_, 0] - (s1[st_] - dt[r0])).abs() / a1[st_]
        p2 = (part[st_, 1] - (s2[st_] - dt[r0] * xt[r0])).abs() / a2[st_]
        p_p = min(p1.max().item(), p2.max().item())
        check_metric(e_p, PART_TOL, f"barlow bwd column partials {name} stripes={nsplit} (rows: [sum dT; sum dT x~] x stripe)",
                     p_p)
        # finished gradient restated in fp64 from the library's own dT and partials
        m1, m2 = part[:, 0].sum(0) / n, part[:, 1].sum(0) / (n - 1)
        xh = x.double() * inv
        xtl = (xh - mean) * rstd
        g = (dt - m1 - xtl * m2) * rstd * go
        scale = ((dt.abs() + m1.abs() + (xtl * m2).abs()) * rstd * abs(go) * inv).norm(dim=1)
        dot = (g * xh).sum(1, keepdim=True)
        g = (g - dot * xh) * inv
        e_f = (b["dz" + s].double() - g).norm(dim=1) / scale
        print(f"barlow finish dz{s} n={n} d={d}: max row error {e_f.max().item():.3e} (row {int(e_f.argmax())})")
        assert e_f.max().item() <= FINISH_TOL, f"dz{s}: max per-row error {e_f.max().item():.3e} (row {int(e_f.argmax())})"


# ------------------------------------------------------------------------------------------------ 4. distributed xcorr
def check_xcorr(C, world, n_local, d, seed=0):
    """ssvb_barlow_dist_xcorr of every emulated rank: fp32 c_partial (EPI_STORE_F32, both operands MN-major)."""
    L, st = c_api(C)
    zi, zj = barlow_inputs(world * n_local, d, seed)
    so, stotal = barlow_dist_saved_layout(n_local, d)
    assert stotal == int(L.ssvb_barlow_dist_saved_bytes(n_local, d)), f"BarlowDistSaved restated as {stotal} bytes"
    wsb = int(L.ssvb_barlow_dist_workspace_bytes(n_local, d))
    ws = nan_bytes(wsb)
    saved = [nan_bytes(stotal) for _ in range(world)]
    stats_all = nan_f32(world, 2, 2, d)
    sl = [slice(q * n_local, (q + 1) * n_local) for q in range(world)]
    for q in range(world):
        C.check(L.ssvb_barlow_dist_stats(C.ptr(zi[sl[q]]), C.ptr(zj[sl[q]]), n_local, d, d, d, 0, C.ptr(stats_all[q]),
                                         C.ptr(saved[q]), C.ptr(ws), wsb, st), "dist_stats")
    plan = xcorr_plan(n_local, d, num_sms())
    alpha = f32(1.0 / (n_local * world))
    outs = []
    for q in range(world):
        cp = nan_f32(d, d)
        C.check(L.ssvb_barlow_dist_xcorr(C.ptr(zi[sl[q]]), C.ptr(zj[sl[q]]), n_local, d, d, d, 0, C.ptr(stats_all), world,
                                         C.ptr(cp), C.ptr(saved[q]), st), "dist_xcorr")
        torch.cuda.synchronize()
        xi = piece(saved[q], so, "xi", torch.bfloat16, (n_local, d)).double()
        xj = piece(saved[q], so, "xj", torch.bfloat16, (n_local, d)).double()
        assert torch.isfinite(cp).all(), "c_partial elements never written"
        gemm_check(cp, xi.T, xj, alpha, plan, seed + q,
                   f"dist xcorr world={world} rank={q} n_local={n_local} d={d} units={plan['units']}")
        outs.append(cp)
    return outs


@pytest.mark.parametrize("world,n_local,d", [
    (1, 300, 4096),  # 512 units (~3.5 per CTA), 5 K blocks with a K tail
    (3, 100, 520),   # alpha = 1/300, ragged M / N, 2 K blocks
])
def test_dist_xcorr_elements(C, world, n_local, d):
    check_xcorr(C, world, n_local, d, seed=world + n_local)


# ------------------------------------------------------------------------------------------------ 5. column shard
def bf16_rne_bits(x32):
    """fp32 numpy array -> bf16 bit patterns (int16), round to nearest even (finite inputs)."""
    u = x32.astype(np.float32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) & 0xFFFF
    return r.astype(np.uint16).view(np.int16)


def exact_operands(n, d, seed):
    """bf16 [n x d] of multiples of 0.5 in [-2, 2]: every product is a multiple of 0.25 of size <= 4, so every partial
    sum over n <= 4096 rows is a multiple of 0.25 below 2^14, exact in fp32 under any summation order."""
    g = torch.Generator().manual_seed(seed)
    return (torch.randint(-4, 5, (n, d), generator=g).float() * 0.5).to(torch.bfloat16).cuda()


CS_CASES = [(2048, 1032, 264, col0) for col0 in (0, 8, 136, 1032 - 264)] + [(512, 520, 136, 384)]


@pytest.mark.parametrize("n,d,ncols,col0", CS_CASES)
def test_cs_fwd_bit_exact(C, n, d, ncols, col0):
    """ssvb_barlow_cs_fwd (EPI_BARLOW on a column slab, diag_off = col0): with exact accumulators the dC slab is
    bit-identical to the epilogue replicated in fp32.  n is a power of two, so c = acc * fl(1/n) is exact as well and a
    contracted c - 1 (fma) cannot differ from the separate product and difference."""
    L, st = c_api(C)
    assert n & (n - 1) == 0 and n <= 4096
    xa, xb = exact_operands(n, d, seed=col0 + 1), exact_operands(n, d, seed=col0 + 2)
    wsb = int(L.ssvb_barlow_cs_workspace_bytes(n, d, ncols))
    ws = nan_bytes(wsb)
    tail = 4096
    slab = torch.full((d * ncols + tail,), -1, dtype=torch.int16, device="cuda")  # 0xFFFF: bf16 NaN
    C.check(L.ssvb_barlow_cs_fwd(C.ptr(xa), C.ptr(xb), n, d, col0, ncols, ctypes.c_float(LAMBDA), C.ptr(slab), None,
                                 C.ptr(ws), wsb, st), "cs_fwd")
    torch.cuda.synchronize()
    assert (slab[d * ncols:] == -1).all(), "cs_fwd wrote past the end of the dC slab"
    got = slab[:d * ncols].view(d, ncols).cpu().numpy()
    acc = (xa.double().T @ xb[:, col0:col0 + ncols].double()).cpu().numpy()
    assert np.array_equal(acc, acc.astype(np.float32).astype(np.float64)), "accumulator not exact in fp32"
    c = acc.astype(np.float32) * np.float32(1.0 / n)
    diag = (np.arange(d)[:, None] == (np.arange(ncols)[None, :] + col0))
    r = np.where(diag, c - np.float32(1.0), c).astype(np.float32)
    w2 = np.where(diag, np.float32(2.0), np.float32(2.0) * np.float32(LAMBDA)).astype(np.float32)
    want = bf16_rne_bits((w2 * r).astype(np.float32))
    bad = np.argwhere(got != want)
    print(f"cs fwd n={n} d={d} ncols={ncols} col0={col0}: {len(bad)} differing bf16 values")
    assert len(bad) == 0, f"dC slab differs at {len(bad)} elements, first (row, col) {tuple(bad[0])}"


@pytest.mark.parametrize("n,d,ncols,col0", [(2048, 1032, 264, 136), (512, 520, 136, 384)])
def test_cs_bwd_elements(C, n, d, ncols, col0):
    """ssvb_barlow_cs_bwd: dT = Xa~ dC_slab / n (EPI_STORE_F32, B MN-major) then the slab column reduction and finish,
    restated in fp64 (slab_col_partials_kernel / slab_finish_kernel)."""
    L, st = c_api(C)
    xa, xb = exact_operands(n, d, seed=col0 + 1), exact_operands(n, d, seed=col0 + 2)
    wsb = int(L.ssvb_barlow_cs_workspace_bytes(n, d, ncols))
    ws = nan_bytes(wsb)
    slab = torch.empty(d, ncols, dtype=torch.bfloat16, device="cuda")
    C.check(L.ssvb_barlow_cs_fwd(C.ptr(xa), C.ptr(xb), n, d, col0, ncols, ctypes.c_float(LAMBDA), C.ptr(slab), None,
                                 C.ptr(ws), wsb, st), "cs_fwd")
    n_local = 64
    so, stotal = barlow_dist_saved_layout(n_local, d)
    assert stotal == int(L.ssvb_barlow_dist_saved_bytes(n_local, d))
    saved = nan_bytes(stotal)
    rstd = (0.5 + torch.rand(d, generator=torch.Generator().manual_seed(n))).cuda()
    piece(saved, so, "rstd_j", torch.float32, (d,)).copy_(rstd)
    go = f32(-0.9)
    gout = torch.full((1,), go, device="cuda")
    pad = 16
    out = nan_f32(n * ncols + pad)
    ws.fill_(0xFF)
    C.check(L.ssvb_barlow_cs_bwd(C.ptr(xa), C.ptr(xb), C.ptr(slab), n, d, col0, ncols, C.ptr(saved), n_local, 1,
                                 C.ptr(gout), C.ptr(out), C.ptr(ws), wsb, st), "cs_bwd")
    torch.cuda.synchronize()
    assert torch.isnan(out[n * ncols:]).all(), "cs_bwd wrote past the end of the gradient slab"
    got = out[:n * ncols].view(n, ncols).double()
    assert torch.isfinite(got).all()
    plan = gemm_plan(n, ncols, d, 256, num_sms())
    alpha = f32(1.0 / n)
    a64, b64 = xa.double(), slab.double()
    xt = xb[:, col0:col0 + ncols].double()
    rs_ = rstd[col0:col0 + ncols].double()

    def finish(t):
        m1, m2 = t.sum(0) / n, (t * xt).sum(0) / (n - 1)
        return (t - m1 - xt * m2) * rs_ * go

    t = (a64 @ b64) * alpha
    rho_t = absmm(a64, b64) * alpha
    rho = (rho_t + rho_t.mean(0) + xt.abs() * (rho_t * xt.abs()).sum(0) / (n - 1)) * rs_ * abs(go)
    err = (got - finish(t)).abs() / rho
    rs, cs, ks = tile_slices(plan, *pick_tile(plan, n + col0))
    tb = t.clone()
    tb[rs, cs] -= (a64[rs, ks] @ b64[ks, cs]) * alpha
    power = ((got - finish(tb)).abs() / rho).max().item()
    check_metric(err, GEMM_TOL, f"cs bwd n={n} d={d} ncols={ncols} col0={col0}", power)


# ------------------------------------------------------------------------------------------------ 6. SwAV scores
def swav_inputs(nb, nbank, k, d, seed):
    g = torch.Generator().manual_seed(seed)

    def unit(x):
        return x / x.norm(dim=1, keepdim=True)
    z1 = unit(torch.randn(nb, d, generator=g))
    z2 = unit(0.6 * z1 + 0.4 * torch.randn(nb, d, generator=g))
    bank = unit(torch.randn(max(nbank, 1), d, generator=g))[:nbank]
    proto = unit(torch.randn(k, d, generator=g))
    return z1.cuda(), z2.cuda(), bank.cuda().contiguous(), proto.cuda()


def check_swav_scores(C, nb, nbank, k, d, seed=0):
    L, st = c_api(C)
    z1, z2, bank, proto = swav_inputs(nb, nbank, k, d, seed)
    m = swav_dims(nb, nbank, k, d)
    kpad = int(L.ssvb_swav_kpad(k))
    assert kpad == m["kp4"]
    so, stotal = swav_saved_layout(nb, nbank, k, d)
    assert stotal == int(L.ssvb_swav_saved_bytes(nb, nbank, k, d)), f"SwavSaved restated as {stotal} bytes"
    saved = nan_bytes(stotal)
    scores = nan_f32(2 * m["bp"], kpad)
    C.check(L.ssvb_swav_dist_scores(C.ptr(z1), C.ptr(z2), C.ptr(bank) if nbank else None, C.ptr(proto), nb, nbank, k, d,
                                    d, d, d, d, C.ptr(scores), C.ptr(saved), st), "swav_dist_scores")
    torch.cuda.synchronize()
    # Padding columns [k, kpad): the row-store epilogue leaves them alone.  The TMA store (box clipped at column k) was
    # seen on B200 to write them at k = 1001: it stores the last 16-byte piece of a row whole, and the padding then
    # holds the accumulator of the zero-filled prototype rows k .. kpad, exactly 0.0.  The cross-entropy kernels mask
    # the padding per element, so either is harmless; any other value is not.
    padv = scores[:, k:]
    print(f"swav scores k={k} kpad={kpad}: {int((padv == 0).sum())} of {padv.numel()} padding values written as 0.0")
    assert (torch.isnan(padv) | (padv == 0)).all(), "the scores GEMM wrote non-zero values into the padding [k, kpad)"
    got = scores[:, :k]
    assert torch.isfinite(got).all(), "score elements never written"
    z = piece(saved, so, "z", torch.bfloat16, (2 * m["bp"], m["dpad"])).double()
    c = piece(saved, so, "c", torch.bfloat16, (k, m["dpad"])).double()
    plan = scores_plan(nb, nbank, k, d, num_sms())
    gemm_check(got, z, c.T, 1.0, plan, seed, f"swav scores nb={nb} nbank={nbank} k={k} d={d} units={plan['units']}")
    return scores


SCORE_CASES = [
    (512, 3000, 3000, 128),  # cfg4: 660 tiles (~4.5 per CTA)
    (64, 70, 1001, 32),      # k % 4 != 0: padding columns, one K block
    (200, 1000, 1000, 100),  # d % 8 != 0: dpad = 104 > d (zero-padded K tail)
]


@pytest.mark.parametrize("nb,nbank,k,d", SCORE_CASES)
def test_swav_scores_elements(C, nb, nbank, k, d):
    check_swav_scores(C, nb, nbank, k, d, seed=nb + k)


# ------------------------------------------------------------------------------------------------ 7. SwAV backward
def check_swav_bwd(C, nb, nbank, k, d, seed=0, tma_store=True):
    """dz (ds @ C) and dproto (ds^T @ [Z1; Z2]) per element, as the GEMMs leave them in the workspace and as the
    grad_out-scaled outputs; ds is read from `saved` (an input here: the cross-entropy kernel is not under test)."""
    L, st = c_api(C)
    z1, z2, bank, proto = swav_inputs(nb, nbank, k, d, seed)
    m = swav_dims(nb, nbank, k, d)
    bp, dpad = m["bp"], m["dpad"]
    so, stotal = swav_saved_layout(nb, nbank, k, d)
    wo, wtotal = swav_ws_layout(L, nb, nbank, k, d)
    assert stotal == int(L.ssvb_swav_saved_bytes(nb, nbank, k, d)), f"SwavSaved restated as {stotal} bytes"
    assert wtotal == int(L.ssvb_swav_workspace_bytes(nb, nbank, k, d)), f"SwavWs restated as {wtotal} bytes"
    saved, ws = nan_bytes(stotal), nan_bytes(wtotal)
    loss = nan_f32(1)
    bk = C.ptr(bank) if nbank else None
    C.check(L.ssvb_swav_fwd(C.ptr(z1), C.ptr(z2), bk, C.ptr(proto), nb, nbank, k, d, d, d, d, d, ctypes.c_float(0.1),
                            ctypes.c_float(0.05), 3, C.ptr(loss), C.ptr(saved), C.ptr(ws), wtotal, st), "swav_fwd")
    ws.fill_(0xFF)  # the backward reads only `saved`
    pad = 4
    o1, o2, op = nan_f32(nb, d + pad), nan_f32(nb, d + pad), nan_f32(k, d + pad)
    go = f32(1.3)
    gout = torch.full((1,), go, device="cuda")
    C.check(L.ssvb_swav_bwd(C.ptr(z1), C.ptr(z2), bk, C.ptr(proto), nb, nbank, k, d, d, d, d, d, ctypes.c_float(0.1),
                            C.ptr(gout), C.ptr(saved), C.ptr(o1), C.ptr(o2), C.ptr(op), d + pad, d + pad, d + pad,
                            C.ptr(ws), wtotal, st), "swav_bwd")
    torch.cuda.synchronize()
    for o in (o1, o2, op):
        assert torch.isnan(o[:, d:]).all(), "the backward wrote past column d of an output row"
    z = piece(saved, so, "z", torch.bfloat16, (2 * bp, dpad)).double()
    c = piece(saved, so, "c", torch.bfloat16, (k, dpad)).double()
    ds = piece(saved, so, "ds", torch.bfloat16, (2 * bp, m["kp8"]))[:, :k].double()
    assert torch.isfinite(ds).all()
    pz, pc = swav_bwd_plans(nb, nbank, k, d, num_sms(), tma_store)
    dz = piece(ws, wo, "dz", torch.float32, (2 * bp, dpad))
    dc = piece(ws, wo, "dc", torch.float32, (k, dpad))
    for got, a64, b64, plan, name in ((dz, ds, c, pz, "dz"), (dc, ds.T, z, pc, "dproto")):
        assert torch.isfinite(got).all(), f"{name}: elements never written"
        what = (f"swav bwd {name} nb={nb} nbank={nbank} k={k} d={d} tiles={plan['tiles']} splits={plan['splits']} "
                f"kb_per={plan['kb_per']} last={plan['last']}")
        gemm_check(got, a64, b64, 1.0, plan, seed, what)
    # the grad_out-scaled outputs: one fp32 product per element
    for got, ref in ((o1[:, :d], dz[:nb, :d]), (o2[:, :d], dz[bp:bp + nb, :d]), (op[:, :d], dc[:, :d])):
        assert torch.equal(got, ref * go), "grad_out scaling of a GEMM output differs"
    return pz, pc


SWAV_BWD_CASES = [
    (512, 3000, 3000, 128),  # cfg4: dz 55 tiles -> 2 splits (24 + 23 K blocks); dproto 24 tiles -> 6 splits (5 x 19 + 15)
    (64, 70, 1001, 32),      # dz 3 tiles -> 4 splits of 4 blocks; dproto 8 tiles but 5 K blocks -> unsplit
    (300, 350, 1201, 1000),  # dz 88 tiles, dproto 80 tiles (>= 74): both unsplit; 8 column tiles of 128
]


@pytest.mark.parametrize("nb,nbank,k,d", SWAV_BWD_CASES)
def test_swav_bwd_elements(C, nb, nbank, k, d):
    check_swav_bwd(C, nb, nbank, k, d, seed=nb + k)


# ------------------------------------------------------------------------------------------------ plan coverage
FWD_CASES = [(256, 264), (300, 4096), (2048, 8192)]
BWD_CASES = [(200, 264), (1000, 1000), (2000, 3400)]
UNFUSED_CASES = [(300, 520), (2000, 3400), (8320, 136)]
XCORR_CASES = [(1, 300, 4096), (3, 100, 520)]


def test_plan_reaches_every_regime(C):
    """The parameter lists above reach, on this GPU: >= 3 units per CTA in every epilogue mode, a K-block count per
    tile that is not a multiple of the ring depth (4) with several units per CTA, split-K with a short last slice, the
    unsplit case of both SwAV backward GEMMs, and ragged M, N and K tails."""
    sms = num_sms()
    modes = {
        "EPI_BARLOW": [barlow_fwd_plan(n, d, sms) for n, d in FWD_CASES],
        "EPI_BARLOW_BWD": [barlow_bwd_plan(n, d, sms) for n, d in BWD_CASES],
        "DUAL EPI_STORE_F32": [barlow_bwd_plan(n, d, sms) for n, d in UNFUSED_CASES],
        "EPI_STORE_F32": [xcorr_plan(nl, d, sms) for _, nl, d in XCORR_CASES] + [scores_plan(*c, sms) for c in SCORE_CASES],
    }
    swav = [swav_bwd_plans(*c, sms) for c in SWAV_BWD_CASES]
    for mode, plans in modes.items():
        best = max(p["units"] / p["grid"] for p in plans)
        print(f"{mode}: max units per CTA {best:.2f} with {sms} SMs")
        assert any(p["units"] >= 3 * p["grid"] for p in plans), f"{mode}: no case runs >= 3 units on every CTA"
    everything = [p for ps in modes.values() for p in ps] + [p for pair in swav for p in pair]
    assert any(p["splits"] == 1 and p["nkb"] % 4 and p["units"] >= 2 * p["grid"] for p in modes["EPI_BARLOW"])
    assert any(p["splits"] == 1 and p["nkb"] % 4 and p["units"] >= 2 * p["grid"] for p in modes["EPI_BARLOW_BWD"])
    assert any(p["splits"] > 1 and p["last"] < p["kb_per"] for pair in swav for p in pair), "no short last K slice"
    assert any(pz["splits"] > 1 for pz, _ in swav) and any(pc["splits"] > 1 for _, pc in swav), "split-K not reached"
    assert any(pz["splits"] == 1 for pz, _ in swav) and any(pc["splits"] == 1 for _, pc in swav), "unsplit not reached"
    assert any(p["M"] % 128 for p in everything) and any(p["N"] % p["bn"] for p in everything)
    assert any(p["K"] % 64 for p in everything)
    # without the staged TMA-store epilogue (SSVB_GEMM_NO_TMA_STORE) nothing splits
    assert all(p["splits"] == 1 for c in SWAV_BWD_CASES for p in swav_bwd_plans(*c, sms, tma_store=False))


# ------------------------------------------------------------------------------------------------ 8. row-store epilogue
ROWSTORE_CODE = r"""
import importlib.util, sys, torch
sys.path[:0] = [%r, %r]
spec = importlib.util.spec_from_file_location("gemm_elements", %r)
T = importlib.util.module_from_spec(spec)
spec.loader.exec_module(T)
from ssv_b200 import _cabi as C
torch.backends.cuda.matmul.allow_tf32 = False
for n, d in [(256, 264), (300, 4096)]:
    T.check_barlow_fwd(C, n, d, seed=n + d)
for world, n_local, d in T.XCORR_CASES:
    T.check_xcorr(C, world, n_local, d, seed=world + n_local)
for case in T.SCORE_CASES:
    T.check_swav_scores(C, *case, seed=case[0] + case[2])
for case in T.SWAV_BWD_CASES:
    pz, pc = T.check_swav_bwd(C, *case, seed=case[0] + case[2], tma_store=False)
    assert pz["splits"] == 1 and pc["splits"] == 1
# EPI_BARLOW_BWD lives in the staged epilogue only: normalize = 0 now goes through the workspace dT buffers
r = T.run_barlow_fwd(C, *T.barlow_inputs(200, 264, 1), False)
b = T.run_barlow_bwd(C, r, -0.7)
assert torch.isfinite(b["dti"]).all() and torch.isfinite(b["dtj"]).all(), "row-store process took the fused epilogue"
print("rowstore-ok")
"""


def test_row_store_epilogue_elements():
    """SSVB_GEMM_NO_TMA_STORE=1 (read once per process, hence the subprocess): the per-thread row-store epilogue, checked
    with the same functions as above (Barlow forward, xcorr, SwAV scores and backward; no split-K in this mode)."""
    code = ROWSTORE_CODE % (ROOT, PKG, os.path.abspath(__file__))
    env = dict(os.environ, SSVB_GEMM_NO_TMA_STORE="1")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    print(out.stdout[-6000:])
    assert out.returncode == 0 and "rowstore-ok" in out.stdout, out.stdout[-3000:] + out.stderr[-4000:]


# ------------------------------------------------------------------------------------------------ 9. determinism
def bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def test_run_to_run_bitwise(C):
    """Plain-store GEMM outputs are bit-identical over two runs.  Not asserted for the split-K outputs (SwAV dz /
    dproto): the order in which the TMA reduce-add of different CTAs reaches an element is not fixed."""
    L, st = c_api(C)
    zi, zj = barlow_inputs(300, 4096, 11)
    a, b = run_barlow_fwd(C, zi, zj, False), run_barlow_fwd(C, zi, zj, False)
    for key in ("dC", "q_i", "q_j", "loss"):
        assert torch.equal(bits(a[key]), bits(b[key])), key
    zi, zj = barlow_inputs(1000, 1000, 12)
    r1 = run_barlow_fwd(C, zi, zj, False)
    g1 = run_barlow_bwd(C, r1, -0.7)["dzi"].clone()
    g2 = run_barlow_bwd(C, r1, -0.7)["dzi"]
    assert torch.equal(bits(g1), bits(g2)), "dzi"
    s1, s2 = check_swav_scores(C, *SCORE_CASES[0], seed=5), check_swav_scores(C, *SCORE_CASES[0], seed=5)
    k = SCORE_CASES[0][2]
    assert torch.equal(bits(s1[:, :k].contiguous()), bits(s2[:, :k].contiguous())), "scores"
    c1, c2 = check_xcorr(C, 1, 300, 4096, seed=7), check_xcorr(C, 1, 300, 4096, seed=7)
    assert torch.equal(bits(c1[0]), bits(c2[0])), "c_partial"
