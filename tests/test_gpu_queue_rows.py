"""Per-row checks of the queue-axis similarity path: two-pass MoCo, PIRL and the sharded-queue MoCo stages.

These callers run sim_fwd_kernel / sim_bwd_kernel in SIM_MOCO mode in the online-max form: per-chunk (max, sum)
partials, a finalize kernel, and a backward weighted by exp2(c s - lse2).  The whole-tensor checks elsewhere (loss rel
<= 1e-3, gradient rel-L2 <= 1e-2) cannot see one 128-column block of a 65536-entry queue: it moves lse2 by ~3e-3 (log2
units) and the loss by ~2e-4 relative.  These tests drive the C ABI with their own buffers and check every row of every
intermediate against fp64 witnesses built from the same staged bf16 rows:

    staging   ws.queue_bf16 == bf16(queue[:, :d]) bit for bit, zero columns d .. dpad
    forward   lse2_a = log2(exp2(c pos_a) + sum_j exp2(c qh_a . mb_j))     (PIRL: one positive per head)
    backward  dacc_a = sum_j exp2(c qh_a . mb_j - lse2_a) mb_j             (the kernel's own lse2: backward isolated)
    finish    moco_grad_finish_kernel / pirl_grad_kernel restated in fp64 from the saved per-row statistics

Metrics: lse2 absolute for unit rows; for raw rows (normalize=False) divided by max(1, max_j |t_aj|), the fp32 scale of
the largest logit of the row.  Accumulators |dacc_a - wit_a| / rho_a with rho_a = sqrt(sum_j w_aj^2 |mb_j|^2), the scale
of the bf16 rounding of the weights.  Every statistic and accumulator test also removes one 128-column block of the
queue (chosen by the seed) from the witness and asserts that the kernel's metric against that perturbed witness is at
least 10x the tolerance.  Buffers the kernels write are NaN-filled first: a row that is never stored fails as NaN.

Tolerances: measured maxima on one B200 are in profiles/r6_queue_rows.md; each tolerance is about 3x the largest
maximum of its class and at least 10x below the smallest one-block value of that class.
"""
import ctypes
import math

import pytest
import torch

from test_gpu_sim_bwd_rows import (C, LOG2E, MOCO_FUSED_CASES, cdiv, moco_finish_witness,  # noqa: F401
                                   moco_saved_layout, num_sms, plan_chunks_tiles, row_metric, ru, unit_rows)

pytestmark = pytest.mark.gpu

LN2 = math.log(2.0)

# tolerances (profiles/r6_queue_rows.md lists the measured maximum of every case)
LSE_TOL = 2e-5        # lse2 per row, unit rows, absolute: measured <= 2.7e-6 at tau >= 0.07, 7.0e-6 at tau = 0.02
LSE_RAW_TOL = 1e-6    # lse2 per row, raw rows, absolute / max(1, max_j |t_aj|): measured <= 3.2e-7
ACC_TOL = 7e-3        # backward accumulator per row, relative to rho (bf16 weights): measured <= 3.6e-3
FINISH_TOL = 5e-7     # MoCo and PIRL gradient finish restated in fp64 with the fp32 exponent: measured <= 1.4e-7
POS_TOL = 3e-7        # positive logit, |pos - fp64 dot of the staged rows| / (|qh| |kh|): measured <= 1.0e-7
INV_TOL = 4e-7        # 1 / |x| per row, relative: measured <= 1.3e-7
RUN_TO_RUN_TOL = 1e-5  # run-to-run difference of the red.add accumulator, relative to rho: measured <= 2.7e-6 (74 chunks)


# ------------------------------------------------------------------------------------------------ restated layouts
def dpad_of(d):
    return ru(d, 64) if d <= 128 else 256


def queue_fwd_plan(n, k, dpad, sms):
    """moco_plan for sim_fwd_kernel: BN = 256 (dpad <= 128) or 128, at least 512 columns per chunk."""
    bn = 128 if dpad > 128 else 256
    return plan_chunks_tiles(cdiv(n, 128), cdiv(k, bn), 512 // bn, sms)


def queue_bwd_plan(n, k, sms):
    """moco_plan for sim_bwd_kernel (and the fused MoCo forward): 128-column tiles, at least 4 per chunk."""
    return plan_chunks_tiles(cdiv(n, 128), cdiv(k, 128), 4, sms)


def carve(pieces):
    """host_util.h Carver: every piece starts on a 256-byte boundary -> ({name: byte offset}, total bytes)."""
    offs, off = {}, 0
    for name, nbytes in pieces:
        off = ru(off, 256)
        offs[name] = off
        off += nbytes
    return offs, ru(off, 256)


def moco_ws_layout(n, k, dpad, sms):
    """moco.cu moco_ws (two-pass MoCo, PIRL and the sharded stages, n = n_global, k = k_local)."""
    npad = ru(n, 128)
    nch = max(queue_fwd_plan(n, k, dpad, sms)[1], queue_bwd_plan(n, k, sms)[1])
    return carve([("queue_bf16", k * dpad * 2), ("part_m", 4 * nch * npad * 4), ("part_l", 4 * nch * npad * 4),
                  ("block_sums", (cdiv(npad, 8) + 8) * 4), ("counter", 16), ("dacc", npad * dpad * 4)])


PIRL_F32 = ("inv_patch", "inv_img", "pos_patch", "pos_img", "lse_patch", "lse_img", "unused")


def pirl_saved_layout(n, dpad):
    """moco.cu pirl_saved: qhat bf16 [npad x dpad], then seven fp32 [npad] arrays."""
    npad = ru(n, 128)
    return carve([("qhat", npad * dpad * 2)] + [(name, npad * 4) for name in PIRL_F32])


def f32_at(buf, off, count):
    return buf[off:off + count * 4].view(torch.float32).clone()


def bf16_at(buf, off, rows, dpad):
    return buf[off:off + rows * dpad * 2].view(torch.bfloat16).view(rows, dpad).clone()


# ------------------------------------------------------------------------------------------------ witnesses
def logits2(qh, mb, c):
    """c qh mb^T in fp64: the log2-domain logits the forward sees (both operands are the staged bf16 rows)."""
    return c * (qh.double() @ mb.double().T)


def drop_block(k, seed):
    """the 128-column block of a K-row queue that the power checks remove"""
    return (seed * 7 + 3) % cdiv(k, 128)


def lse2_witness(t, pos2=None, drop=None):
    """log2(sum_j exp2(t_aj) [+ exp2(pos2_a)]) in fp64, without the columns of block `drop` when given."""
    if drop is not None:
        t = t.clone()
        t[:, drop * 128:drop * 128 + 128] = -math.inf
    if pos2 is not None:
        t = torch.cat([t, pos2.double()[:, None]], dim=1)
    return torch.logsumexp(t * LN2, dim=1) / LN2


def lse_scale(t, pos2, normalize):
    """1 for unit rows; max(1, max_j |t_aj|) over the row's logits (positive included) for raw rows."""
    if normalize:
        return torch.ones(t.shape[0], dtype=torch.float64, device=t.device)
    s = t.abs().max(dim=1).values
    if pos2 is not None:
        s = torch.maximum(s, pos2.double().abs())
    return s.clamp(min=1.0)


def check_lse(got, t, pos2, normalize, seed, what):
    """per-row lse2 metric and its one-block power check; returns the maximum metric."""
    tol = LSE_TOL if normalize else LSE_RAW_TOL
    scale = lse_scale(t, pos2, normalize)
    assert torch.isfinite(got).all(), f"{what}: non-finite lse2 (a row never stored)"
    err = (got.double() - lse2_witness(t, pos2)).abs() / scale
    power = ((got.double() - lse2_witness(t, pos2, drop_block(t.shape[1], seed))).abs() / scale).max().item()
    worst = err.max().item()
    print(f"{what}: max lse2 metric {worst:.3e} (row {int(err.argmax())}), one block {power:.3e}, tol {tol:.1e}")
    assert worst <= tol, f"{what}: max per-row lse2 error {worst:.3e} > {tol:.1e} (row {int(err.argmax())})"
    assert power >= 10 * tol, f"{what}: one missing queue block moves lse2 only by {power:.3e} (< 10 x {tol:.1e})"
    return worst


def acc_witness(t, rowstat, mb, drop):
    """(sum_j exp2(t_aj - rowstat_a) mb_j, rho_a, the same sum without block `drop`) in fp64."""
    w = torch.exp2(t - rowstat.double()[:, None])
    mbd = mb.double()
    wit = w @ mbd
    rho = ((w * w) @ (mbd * mbd).sum(1)).sqrt()
    blk = slice(drop * 128, drop * 128 + 128)
    return wit, rho, wit - w[:, blk] @ mbd[blk]


def check_acc(got, t, rowstat, mb, seed, what):
    assert torch.isfinite(got).all(), f"{what}: non-finite accumulator entries (a row block or column half never stored)"
    wit, rho, wit_p = acc_witness(t, rowstat, mb, drop_block(t.shape[1], seed))
    err = row_metric(got, wit, rho)
    power = row_metric(got, wit_p, rho).max().item()
    worst = err.max().item()
    print(f"{what}: max acc row metric {worst:.3e} (row {int(err.argmax())}), one block {power:.3e}, tol {ACC_TOL:.1e}")
    assert worst <= ACC_TOL, f"{what}: max per-row accumulator error {worst:.3e} > {ACC_TOL:.1e} (row {int(err.argmax())})"
    assert power >= 10 * ACC_TOL, f"{what}: one missing queue block moves the metric only to {power:.3e}"
    return worst, rho


def check_finish(got_q, got_k, wit, what):
    gq, gk, den_q, den_k = wit
    assert torch.isfinite(got_q).all() and torch.isfinite(got_k).all(), f"{what}: non-finite gradient rows"
    eq = ((got_q.double() - gq).norm(dim=1) / den_q).max().item()
    ek = ((got_k.double() - gk).norm(dim=1) / den_k).max().item()
    print(f"{what}: finish dq {eq:.3e} dk {ek:.3e}, tol {FINISH_TOL:.1e}")
    assert eq <= FINISH_TOL and ek <= FINISH_TOL, f"{what}: gradient finish errors {eq:.3e}, {ek:.3e}"


def check_staging(staged, x, d, what):
    """the staged bf16 rows are bf16(x) bit for bit (round to nearest even), zero columns d .. dpad"""
    ref = x.to(torch.bfloat16)
    assert torch.equal(staged[:, :d].view(torch.int16), ref.view(torch.int16)), f"{what}: staged rows differ from bf16(x)"
    assert (staged[:, d:].view(torch.int16) == 0).all(), f"{what}: padding columns d .. dpad are not zero"


def check_prep(inv, x, normalize, what):
    """pair_prep's 1 / max(|x|, 1e-12) (1 when the rows are used as stored)"""
    if not normalize:
        assert (inv == 1.0).all(), f"{what}: inverse norms of rows used as stored are not 1"
        return
    ref = 1.0 / x.double().norm(dim=1).clamp(min=1e-12)
    err = ((inv.double() - ref).abs() / ref).max().item()
    print(f"{what}: max inverse-norm error {err:.3e}")
    assert err <= INV_TOL, f"{what}: inverse norm error {err:.3e} > {INV_TOL:.1e}"


def check_pos(pos, qh, kh, what):
    """positive logit (unscaled) against the fp64 dot product of the two staged bf16 rows"""
    qd, kd = qh.double(), kh.double()
    err = ((pos.double() - (qd * kd).sum(1)).abs() / (qd.norm(dim=1) * kd.norm(dim=1)).clamp(min=1e-30)).max().item()
    print(f"{what}: max pos error {err:.3e}")
    assert err <= POS_TOL, f"{what}: positive logit error {err:.3e} > {POS_TOL:.1e}"


# ------------------------------------------------------------------------------------------------ inputs
def queue_inputs(n, k, d, tau, normalize, seed, zero_rows=0, planted=0):
    """queries, keys [n x d] and a queue [k x d] on the CPU.  Unit queue rows with normalize; raw rows otherwise, with
    norms spread over 0.5 .. 3 and `planted` late queue rows that are scaled copies of queries of norm 3, so that their
    logit c qh_a . m_j is 160 .. 250 (above 128: exp2 overflows fp32 without the running max, which must rescale the
    partials of the earlier tiles).  Keys are q + 0.7 noise (cosine ~0.8); below tau = 0.05 that positive would take
    the whole softmax (c pos ~60 against ~30 for the largest negative at tau = 0.02) and no queue block could move
    lse2, so there the keys are q + 3 noise (cosine ~0.3)."""
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(n, d, generator=g)
    kk = q + (0.7 if tau >= 0.05 else 3.0) * torch.randn(n, d, generator=g)
    mem = unit_rows(torch.randn(k, d, generator=g))
    if not normalize:
        q = unit_rows(q) * (0.5 + 2.5 * torch.rand(n, 1, generator=g))
        kk = unit_rows(kk) * (0.5 + 2.5 * torch.rand(n, 1, generator=g))
        mem = mem * (0.5 + 2.5 * torch.rand(k, 1, generator=g))
        c = LOG2E / tau
        for i in range(planted):
            a, j = (37 * i + 5) % n, k - 1 - 97 * i
            q[a] = unit_rows(q[a:a + 1])[0] * 3.0
            mem[j] = q[a] * (160.0 + 30.0 * i) / (c * 9.0)
    mem[:zero_rows] = 0.0
    return q, kk, mem


def on_device(x, ld=None):
    """x on the GPU; with `ld`, a view of a NaN-filled [rows x ld] buffer (columns d .. ld are never to be read)."""
    if ld is None:
        return x.cuda()
    buf = torch.full((x.shape[0], ld), float("nan"), device="cuda")
    buf[:, :x.shape[1]] = x.cuda()
    return buf[:, :x.shape[1]]


def bf16_staging(x, dpad):
    """the bf16 shadow of fp32 rows as ssvb_ring_enqueue keeps it: [rows x dpad], zero padded"""
    s = torch.zeros(x.shape[0], dpad, dtype=torch.bfloat16, device=x.device)
    s[:, :x.shape[1]] = x.to(torch.bfloat16)
    return s


# ------------------------------------------------------------------------------------------------ 1. two-pass MoCo
def run_moco2(C, n, k, d, tau, normalize, seed, zero_rows=0, ld_queue=None, shadow=False, planted=0, go=-0.8):
    """ssvb_moco_fwd + ssvb_moco_bwd on the two-pass path with the test's own buffers: saved and workspace NaN-filled
    before the forward, the workspace NaN-filled again before the backward."""
    L = C.lib()
    q, kk, mem = queue_inputs(n, k, d, tau, normalize, seed, zero_rows, planted)
    q, kk, queue = q.cuda(), kk.cuda(), on_device(mem, ld_queue)
    dpad, npad = int(L.ssvb_ntxent_dpad(d)), ru(n, 128)
    assert dpad == dpad_of(d)
    qb = bf16_staging(queue, dpad) if shadow else None
    sb, wsb = int(L.ssvb_moco_saved_bytes(n, k, d)), int(L.ssvb_moco_workspace_bytes(n, k, d))
    offs, total = moco_saved_layout(n, dpad)
    assert total == sb, f"moco saved layout restated as {total} bytes, library says {sb}"
    wo, wtotal = moco_ws_layout(n, k, dpad, num_sms())
    assert wtotal == wsb, f"moco workspace layout restated as {wtotal} bytes, library says {wsb}"
    saved = torch.full((sb,), 0xFF, dtype=torch.uint8, device="cuda")
    ws = torch.full((wsb,), 0xFF, dtype=torch.uint8, device="cuda")
    loss = torch.empty(1, device="cuda")
    st = C.stream_ptr()
    args = (C.ptr(q), C.ptr(kk), C.ptr(queue), C.ptr(qb), int(shadow), n, k, d, d, d, queue.stride(0), int(normalize),
            ctypes.c_float(tau))
    C.check(L.ssvb_moco_fwd(*args, C.ptr(loss), C.ptr(saved), C.ptr(ws), wsb, st), "ssvb_moco_fwd")
    torch.cuda.synchronize()
    staged = qb if shadow else bf16_at(ws, wo["queue_bf16"], k, dpad)
    r = dict(n=n, k=k, d=d, dpad=dpad, tau=tau, c=LOG2E / tau, normalize=normalize, go=go, seed=seed, q=q, kk=kk,
             queue=queue, staged=staged, shadow=shadow, loss=loss.clone(), saved_fwd=saved.clone(),
             qh=bf16_at(saved, offs[0], n, dpad).float(), inv_q=f32_at(saved, offs[1], n), inv_k=f32_at(saved, offs[2], n),
             pos=f32_at(saved, offs[3], n), lse2=f32_at(saved, offs[4], n))
    ws.fill_(0xFF)
    gout = torch.full((1,), go, device="cuda")
    dq, dk = torch.empty(n, d, device="cuda"), torch.empty(n, d, device="cuda")
    C.check(L.ssvb_moco_bwd(*args, C.ptr(gout), C.ptr(saved), C.ptr(dq), C.ptr(dk), d, d, C.ptr(ws), wsb, st),
            "ssvb_moco_bwd")
    torch.cuda.synchronize()
    r.update(dacc=f32_at(ws, wo["dacc"], npad * dpad).view(npad, dpad)[:n], dq=dq, dk=dk)
    return r


# (n, k, d, tau, normalize, zero_rows, ld_queue, shadow, planted)
MOCO2_CASES = [
    (256, 65536, 128, 0.07, True, 0, None, False, 0),   # cfg2, plain tensor queue: forward 64 chunks, backward 74 (ragged)
    (200, 4100, 128, 0.07, True, 0, 136, False, 0),     # n and K ragged; queue a view of a wider NaN-filled buffer
    (300, 4100, 32, 0.1, True, 0, None, False, 0),      # dpad = 64
    (150, 3000, 96, 0.2, True, 0, 100, False, 0),       # d = 96 padded to 128, NaN-filled ld_queue = 100
    (200, 5000, 160, 0.1, True, 0, None, False, 0),     # dpad = 256: 128-column forward tiles, two dhalf launches
    (130, 2000, 256, 0.07, True, 0, None, False, 0),    # d = 256
    (100, 100, 128, 0.07, True, 0, None, False, 0),     # K < 128: one 256-wide tile, second half fully masked; 1 chunk
    (64, 130, 64, 0.1, True, 0, None, False, 0),        # K = 130: a 2-column queue tail, 1 chunk
    (256, 4100, 64, 0.2, True, 37, None, False, 0),     # zero queue rows
    (200, 4100, 128, 0.1, False, 0, None, False, 3),    # raw rows, logits > 128 in late tiles (running-max rescale)
    (256, 16384, 128, 0.02, True, 0, None, True, 0),    # MemoryBank shadow at tau = 0.02: 2 c > 120, two-pass
]


def moco2_id(case):
    n, k, d, tau, normalize, zero_rows, ld, shadow, planted = case
    tag = f"{n}x{k}x{d}-tau{tau}" + ("" if normalize else "-raw") + (f"-zero{zero_rows}" if zero_rows else "")
    return tag + (f"-ld{ld}" if ld else "") + ("-shadow" if shadow else "") + (f"-planted{planted}" if planted else "")


def moco2_run(C, case):
    n, k, d, tau, normalize, zero_rows, ld, shadow, planted = case
    return run_moco2(C, n, k, d, tau, normalize, n + k + d, zero_rows, ld, shadow, planted)


@pytest.mark.parametrize("case", [c for c in MOCO2_CASES if not c[7]], ids=moco2_id)
def test_moco2_queue_staging(C, case):
    r = moco2_run(C, case)
    check_staging(r["staged"], r["queue"], r["d"], moco2_id(case))


@pytest.mark.parametrize("case", MOCO2_CASES, ids=moco2_id)
def test_moco2_fwd_rows(C, case):
    r = moco2_run(C, case)
    what, d, norm = moco2_id(case), r["d"], r["normalize"]
    check_prep(r["inv_q"], r["q"], norm, what + " inv_q")
    check_prep(r["inv_k"], r["kk"], norm, what + " inv_k")
    # the staged queries are bf16(q * inv_q) of the kernel's own inverse norm
    check_staging(r["qh"].to(torch.bfloat16), r["q"] * r["inv_q"][:, None] if norm else r["q"], d, what + " qhat")
    kh = (r["kk"] * r["inv_k"][:, None] if norm else r["kk"]).to(torch.bfloat16).float()
    check_pos(r["pos"], r["qh"][:, :d], kh, what)
    t = logits2(r["qh"], r["staged"].float(), r["c"])
    check_lse(r["lse2"], t, r["c"] * r["pos"].double(), norm, r["seed"], what)


@pytest.mark.parametrize("case", MOCO2_CASES, ids=moco2_id)
def test_moco2_bwd_rows(C, case):
    r = moco2_run(C, case)
    what = moco2_id(case) + f" bwd nchunks={queue_bwd_plan(r['n'], r['k'], num_sms())[1]}"
    t = logits2(r["qh"], r["staged"].float(), r["c"])
    check_acc(r["dacc"], t, r["lse2"], r["staged"].float(), r["seed"], what)
    wit = moco_finish_witness(r["q"], r["kk"], r["inv_q"], r["inv_k"], r["pos"], r["lse2"], r["dacc"], r["tau"], r["go"],
                              r["n"], r["normalize"])
    check_finish(r["dq"], r["dk"], wit, what)


@pytest.mark.parametrize("case", [MOCO2_CASES[0], MOCO2_CASES[4], MOCO2_CASES[7]], ids=moco2_id)
def test_moco2_run_to_run(C, case):
    a, b = moco2_run(C, case), moco2_run(C, case)
    assert torch.equal(a["saved_fwd"], b["saved_fwd"]) and torch.equal(a["loss"], b["loss"]), "forward not bit-stable"
    _, nch = queue_bwd_plan(a["n"], a["k"], num_sms())
    bitwise = torch.equal(a["dacc"], b["dacc"])
    if nch == 1:  # plain stores
        assert bitwise and torch.equal(a["dq"], b["dq"]) and torch.equal(a["dk"], b["dk"])
        return
    # nchunks > 1: float red.add of the chunk partials in arrival order.  Two addends commute exactly (that is why the
    # NT-Xent accumulator at 2 chunks is bit-stable); 74 of them round differently from run to run.
    t = logits2(a["qh"], a["staged"].float(), a["c"])
    _, rho, _ = acc_witness(t, a["lse2"], a["staged"].float(), 0)
    diff = row_metric(a["dacc"], b["dacc"].double(), rho).max().item()
    print(f"run-to-run {moco2_id(case)} nchunks={nch}: bit-identical {bitwise}, max row difference {diff:.3e}")
    assert diff <= RUN_TO_RUN_TOL, f"run-to-run accumulator difference {diff:.3e} > {RUN_TO_RUN_TOL:.1e}"


# ------------------------------------------------------------------------------------------------ 2. PIRL
def pirl_inputs(n, k, d, normalize, seed):
    """img, patch [n x d]; mem_pos [n x d] and mem_neg [k x d] memory-bank rows (unit rows; raw rows with norms spread
    over 0.5 .. 2 when normalize=False, img / patch then of about unit norm)."""
    g = torch.Generator().manual_seed(seed)
    img = torch.randn(n, d, generator=g)
    patch = img + 0.8 * torch.randn(n, d, generator=g)
    mem_pos = unit_rows(img + 0.5 * torch.randn(n, d, generator=g))
    mem_neg = unit_rows(torch.randn(k, d, generator=g))
    if not normalize:
        img, patch = img / math.sqrt(d), patch / math.sqrt(d)
        mem_pos = mem_pos * (0.5 + 1.5 * torch.rand(n, 1, generator=g))
        mem_neg = mem_neg * (0.5 + 1.5 * torch.rand(k, 1, generator=g))
    return img, patch, mem_pos, mem_neg


def run_pirl(C, n, k, d, tau, normalize, seed, w=0.5, go=1.0, ld_in=None, ld_out=None, heads=("patch", "img"),
             sentinel=-7.25):
    L = C.lib()
    img, patch, mem_pos, mem_neg = (on_device(x, ld_in) for x in pirl_inputs(n, k, d, normalize, seed))
    dpad = int(L.ssvb_ntxent_dpad(d))
    sb, wsb = int(L.ssvb_pirl_saved_bytes(n, d)), int(L.ssvb_pirl_workspace_bytes(n, k, d))
    offs, total = pirl_saved_layout(n, dpad)
    assert total == sb, f"pirl saved layout restated as {total} bytes, library says {sb}"
    wo, wtotal = moco_ws_layout(n, k, dpad, num_sms())
    assert wtotal == wsb, f"pirl workspace layout restated as {wtotal} bytes, library says {wsb}"
    saved = torch.full((sb,), 0xFF, dtype=torch.uint8, device="cuda")
    ws = torch.full((wsb,), 0xFF, dtype=torch.uint8, device="cuda")
    loss = torch.empty(1, device="cuda")
    st = C.stream_ptr()
    C.check(L.ssvb_pirl_fwd(C.ptr(img), C.ptr(patch), C.ptr(mem_pos), C.ptr(mem_neg), n, k, d, img.stride(0),
                            patch.stride(0), mem_pos.stride(0), mem_neg.stride(0), int(normalize), ctypes.c_float(tau),
                            ctypes.c_float(w), C.ptr(loss), C.ptr(saved), C.ptr(ws), wsb, st), "ssvb_pirl_fwd")
    ld = ld_out or d
    out = {h: torch.full((n, ld), sentinel, device="cuda") for h in ("patch", "img")}
    dst = {h: (out[h][:, :d] if h in heads else None) for h in ("patch", "img")}
    gout = torch.full((1,), go, device="cuda")
    C.check(L.ssvb_pirl_bwd(C.ptr(img), C.ptr(patch), C.ptr(mem_pos), n, d, img.stride(0), patch.stride(0),
                            mem_pos.stride(0), int(normalize), ctypes.c_float(tau), ctypes.c_float(w), C.ptr(gout),
                            C.ptr(saved), C.ptr(dst["img"]), C.ptr(dst["patch"]), ld, ld, st), "ssvb_pirl_bwd")
    torch.cuda.synchronize()
    r = dict(n=n, k=k, d=d, dpad=dpad, tau=tau, c=LOG2E / tau, normalize=normalize, w=w, go=go, seed=seed, img=img,
             patch=patch, mem_pos=mem_pos, mem_neg=mem_neg, out=out, heads=heads, sentinel=sentinel,
             qh=bf16_at(saved, offs["qhat"], n, dpad).float(), staged=bf16_at(ws, wo["queue_bf16"], k, dpad))
    r.update({name: f32_at(saved, offs[name], n) for name in PIRL_F32})
    return r


# (n, k, d, tau, normalize)
PIRL_CASES = [
    (100, 65536, 128, 0.07, True),   # 128 forward chunks: 512 partials, the tail loop of load_row_partials' callers
    (300, 65536, 128, 0.07, True),   # 43 chunks, ragged
    (100, 4100, 64, 0.07, True),
    (150, 3000, 256, 0.07, True),    # dpad = 256
    (256, 16384, 128, 0.2, False),   # raw rows
]


@pytest.mark.parametrize("n,k,d,tau,normalize", PIRL_CASES)
def test_pirl_fwd_rows(C, n, k, d, tau, normalize):
    seed = n + k + d
    r = run_pirl(C, n, k, d, tau, normalize, seed, w=0.3)
    what = f"pirl {n}x{k}x{d} tau={tau} norm={normalize} nparts={4 * queue_fwd_plan(n, k, r['dpad'], num_sms())[1]}"
    # "query" = mem_pos as stored (never normalised), negatives = mem_neg as stored
    check_staging(r["qh"].to(torch.bfloat16), r["mem_pos"], d, what + " qhat")
    check_staging(r["staged"], r["mem_neg"], d, what + " negatives")
    t = logits2(r["qh"], r["staged"].float(), r["c"])
    for head, inv, pos, lse in (("patch", "inv_patch", "pos_patch", "lse_patch"), ("img", "inv_img", "pos_img", "lse_img")):
        x = r[head]
        check_prep(r[inv], x, normalize, f"{what} {inv}")
        xh = (x * r[inv][:, None] if normalize else x).to(torch.bfloat16).float()
        check_pos(r[pos], r["qh"][:, :d], xh, f"{what} {pos}")
        check_lse(r[lse], t, r["c"] * r[pos].double(), normalize, seed, f"{what} {lse}")


def pirl_grad_witness(r, head):
    """pirl_grad_kernel restated in fp64: coef = (exp2(fp32(pos c - lse2)) - 1) go / (n tau) w_h, g = coef mem_pos,
    projected through the row normalisation of the head's rows; returns (g, |coef mem_pos / |x||)."""
    n, tau = r["n"], r["tau"]
    pos, lse = r["pos_" + head].double(), r["lse_" + head].double()
    c32 = (torch.tensor(LOG2E, dtype=torch.float32) / torch.tensor(tau, dtype=torch.float32)).double()
    arg = (pos * c32 - lse).float()
    w32 = torch.tensor(r["w"], dtype=torch.float32)
    wh = float(w32 if head == "patch" else 1.0 - w32)  # the kernel's fp32 w and 1 - w
    coef = ((torch.exp2(arg) - 1.0).double() * (r["go"] / (n * tau)) * wh)[:, None]
    g = coef * r["mem_pos"].double()
    x = r[head].double()
    iv = r["inv_" + head].double()[:, None] if r["normalize"] else torch.ones(n, 1, dtype=torch.float64, device="cuda")
    den = (g * iv).norm(dim=1).clamp(min=1e-30)
    if r["normalize"]:
        xh = x * iv
        g = (g - (g * xh).sum(1, keepdim=True) * xh) * iv
    return g, den


@pytest.mark.parametrize("n,k,d,tau,normalize,w,go,ld_in,ld_out,heads", [
    (100, 4100, 64, 0.07, True, 0.3, 1.0, 72, 68, ("patch", "img")),
    (150, 3000, 256, 0.2, True, 0.7, -1.3, 260, 264, ("patch", "img")),   # second float4 of each lane
    (300, 2000, 36, 0.07, False, 0.6, 2.0, 40, 44, ("patch", "img")),     # raw rows, first float4 partial
    (200, 1000, 128, 0.1, True, 0.25, -0.6, 132, 136, ("patch",)),        # d_img = NULL
    (200, 1000, 128, 0.1, False, 0.25, -0.6, 132, 136, ("img",)),         # d_patch = NULL
])
def test_pirl_grad_rows(C, n, k, d, tau, normalize, w, go, ld_in, ld_out, heads):
    r = run_pirl(C, n, k, d, tau, normalize, n + d, w=w, go=go, ld_in=ld_in, ld_out=ld_out, heads=heads)
    for head in ("patch", "img"):
        buf = r["out"][head]
        if head not in heads:
            assert (buf == r["sentinel"]).all(), f"d_{head} is NULL but its buffer was written"
            continue
        assert (buf[:, d:] == r["sentinel"]).all(), f"pirl_grad_kernel wrote d_{head} past column d"
        g, den = pirl_grad_witness(r, head)
        got = buf[:, :d].double()
        assert torch.isfinite(got).all()
        err = ((got - g).norm(dim=1) / den).max().item()
        print(f"pirl grad n={n} d={d} norm={normalize} w={w} go={go} d_{head}: max row error {err:.3e}")
        assert err <= FINISH_TOL, f"d_{head}: max per-row error {err:.3e} > {FINISH_TOL:.1e}"


# ------------------------------------------------------------------------------------------------ 3. sharded queue
def run_moco_dist(C, world, n, k, d, tau, normalize, seed, shadow=False, go=1.3):
    """prep -> shard_fwd -> finalize -> shard_bwd -> finish for `world` ranks emulated in one process (all-gather =
    shared buffers, reduce-scatter = sum of the partial accumulators).  Every output buffer is NaN-filled first and
    every shard call gets a NaN-filled workspace."""
    L = C.lib()
    ng, kl = n * world, k // world
    assert kl * world == k
    q, kk, mem = queue_inputs(ng, k, d, tau, normalize, seed, zero_rows=5)
    Q, K, M = q.cuda(), kk.cuda(), mem.cuda()
    npad, dpad = int(L.ssvb_moco_dist_npad(ng)), int(L.ssvb_ntxent_dpad(d))
    assert npad == ru(ng, 128)
    st = C.stream_ptr()
    qhat_all = torch.full((npad, dpad), float("nan"), dtype=torch.bfloat16, device="cuda")
    rowstat = torch.full((world, 3, n), float("nan"), device="cuda")
    for r in range(world):
        C.check(L.ssvb_moco_dist_prep(C.ptr(Q[r * n:]), C.ptr(K[r * n:]), n, d, d, d, int(normalize), world, r,
                                      C.ptr(qhat_all), C.ptr(rowstat[r]), st), "prep")
    wsb = int(L.ssvb_moco_dist_workspace_bytes(ng, kl, d))
    wo, wtotal = moco_ws_layout(ng, kl, dpad, num_sms())
    assert wtotal == wsb, f"sharded workspace layout restated as {wtotal} bytes, library says {wsb}"
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    shards = [M[r * kl:(r + 1) * kl] for r in range(world)]
    shadows = [bf16_staging(s, dpad) for s in shards] if shadow else [None] * world
    # part_local per rank: [m (n_global) | l (n_global) | pos (n_local)]
    part_all = torch.full((world, 2 * ng + n), float("nan"), device="cuda")
    staged = []
    for r in range(world):
        ws.fill_(0xFF)
        C.check(L.ssvb_moco_dist_shard_fwd(C.ptr(qhat_all), ng, C.ptr(shards[r]), C.ptr(shadows[r]), kl, d, d, tau,
                                           C.ptr(rowstat[r]), n, C.ptr(part_all[r]), C.ptr(ws), wsb, st), "shard_fwd")
        torch.cuda.synchronize()
        staged.append(shadows[r] if shadow else bf16_at(ws, wo["queue_bf16"], kl, dpad))
    lse2_all = torch.full((npad,), float("nan"), device="cuda")
    loss = torch.empty((), device="cuda")
    ws.fill_(0xFF)
    C.check(L.ssvb_moco_dist_finalize(C.ptr(part_all), world, n, tau, C.ptr(lse2_all), C.ptr(loss), C.ptr(ws), wsb, st),
            "finalize")
    dacc_parts = []
    for r in range(world):
        part = torch.full((npad, dpad), float("nan"), device="cuda")
        ws.fill_(0xFF)
        C.check(L.ssvb_moco_dist_shard_bwd(C.ptr(qhat_all), ng, C.ptr(shards[r]), C.ptr(shadows[r]), kl, d, d, tau,
                                           C.ptr(lse2_all), C.ptr(part), C.ptr(ws), wsb, st), "shard_bwd")
        dacc_parts.append(part[:ng])
    dacc = torch.zeros(ng, dpad, device="cuda")
    for p in dacc_parts:
        dacc += p
    gout = torch.full((1,), go, device="cuda")
    dq, dk = torch.empty(ng, d, device="cuda"), torch.empty(ng, d, device="cuda")
    for r in range(world):
        sl = slice(r * n, (r + 1) * n)
        C.check(L.ssvb_moco_dist_finish(C.ptr(Q[sl]), C.ptr(K[sl]), n, ng, d, d, d, int(normalize), tau,
                                        C.ptr(rowstat[r]), C.ptr(lse2_all[sl]), C.ptr(dacc[sl]), C.ptr(gout),
                                        C.ptr(dq[sl]), C.ptr(dk[sl]), d, d, st), "finish")
    torch.cuda.synchronize()
    return dict(world=world, n=n, ng=ng, kl=kl, d=d, dpad=dpad, tau=tau, c=LOG2E / tau, normalize=normalize, go=go,
                seed=seed, Q=Q, K=K, shards=shards, qhat_all=qhat_all, qh=qhat_all[:ng].float(), rowstat=rowstat, part_all=part_all,
                staged=staged, lse2=lse2_all[:ng], dacc_parts=dacc_parts, dacc=dacc, dq=dq, dk=dk)


# (world, n_local, K, d, tau, normalize, shadow)
DIST_CASES = [
    (4, 64, 8192, 128, 0.07, True, False),
    (2, 50, 1000, 64, 0.2, True, False),     # shards of 500 rows (ragged tiles), 1 chunk
    (8, 32, 65536, 128, 0.07, True, False),  # shards of 8192 rows
    (3, 100, 3000, 256, 0.1, True, False),   # dpad = 256
    (2, 64, 4096, 128, 0.2, False, False),   # raw rows
    (4, 64, 8192, 128, 0.07, True, True),    # each shard's bf16 staging passed as the shadow
]


def dist_id(case):
    world, n, k, d, tau, normalize, shadow = case
    return f"w{world}-{n}x{k}x{d}-tau{tau}" + ("" if normalize else "-raw") + ("-shadow" if shadow else "")


def dist_run(C, case):
    world, n, k, d, tau, normalize, shadow = case
    return run_moco_dist(C, world, n, k, d, tau, normalize, seed=10 * world + n + d, shadow=shadow)


def test_dist_prep_rows(C):
    """prep writes its rank's slot of qhat_all (bf16 of the normalised rows), zero padding rows, and rowstat_local"""
    r = dist_run(C, DIST_CASES[1])
    ng, n, d = r["ng"], r["n"], r["d"]
    inv_q, inv_k = r["rowstat"][:, 0].reshape(-1), r["rowstat"][:, 1].reshape(-1)
    check_prep(inv_q, r["Q"], True, "dist prep inv_q")
    check_prep(inv_k, r["K"], True, "dist prep inv_k")
    check_staging(r["qh"].to(torch.bfloat16), r["Q"] * inv_q[:, None], d, "dist prep qhat_all")
    check_pos(r["rowstat"][:, 2].reshape(-1), r["qh"][:, :d], (r["K"] * inv_k[:, None]).to(torch.bfloat16).float(),
              "dist prep pos")
    assert ng % 128 != 0 and (r["qhat_all"][ng:].view(torch.int16) == 0).all(), "padding rows of qhat_all not zeroed"


@pytest.mark.parametrize("case", DIST_CASES, ids=dist_id)
def test_dist_shard_fwd_rows(C, case):
    r = dist_run(C, case)
    ng, n = r["ng"], r["n"]
    for s in range(r["world"]):
        what = f"{dist_id(case)} shard {s}"
        if not case[6]:
            check_staging(r["staged"][s], r["shards"][s], r["d"], what)
        part = r["part_all"][s]
        assert torch.equal(part[2 * ng:], r["rowstat"][s, 2]), f"{what}: pos block is not rank {s}'s positive logits"
        got = part[:ng].double() + torch.log2(part[ng:2 * ng].double())
        t = logits2(r["qh"], r["staged"][s].float(), r["c"])
        check_lse(got, t, None, r["normalize"], r["seed"] + s, what)


@pytest.mark.parametrize("case", DIST_CASES, ids=dist_id)
def test_dist_finalize_rows(C, case):
    r = dist_run(C, case)
    t = logits2(r["qh"], torch.cat(r["staged"]).float(), r["c"])
    pos2 = r["c"] * r["rowstat"][:, 2].reshape(-1).double()
    check_lse(r["lse2"], t, pos2, r["normalize"], r["seed"], f"{dist_id(case)} finalize")


@pytest.mark.parametrize("case", DIST_CASES, ids=dist_id)
def test_dist_shard_bwd_rows(C, case):
    r = dist_run(C, case)
    nch = queue_bwd_plan(r["ng"], r["kl"], num_sms())[1]
    for s in range(r["world"]):
        mb = r["staged"][s].float()
        t = logits2(r["qh"], mb, r["c"])
        check_acc(r["dacc_parts"][s], t, r["lse2"], mb, r["seed"] + s, f"{dist_id(case)} shard {s} nchunks={nch}")


@pytest.mark.parametrize("case", DIST_CASES, ids=dist_id)
def test_dist_finish_rows(C, case):
    r = dist_run(C, case)
    rs = r["rowstat"]
    wit = moco_finish_witness(r["Q"], r["K"], rs[:, 0].reshape(-1), rs[:, 1].reshape(-1), rs[:, 2].reshape(-1),
                              r["lse2"], r["dacc"], r["tau"], r["go"], r["ng"], r["normalize"])
    check_finish(r["dq"], r["dk"], wit, f"{dist_id(case)} finish")


# ------------------------------------------------------------------------------------------------ 0. regimes
def test_queue_cases_reach_every_regime(C):
    """the case tables above reach every chunking / padding regime of the queue-axis kernels on this GPU"""
    sms = num_sms()
    fused = [(c[0], c[1], c[2]) for c in MOCO_FUSED_CASES]
    shapes = [(c[0], c[1], c[2]) for c in MOCO2_CASES] + [(c[0], c[1], c[2]) for c in PIRL_CASES]
    shapes += [(c[0] * c[1], c[2] // c[0], c[3]) for c in DIST_CASES]  # (n_global, k_local, d)
    fwd = [queue_fwd_plan(n, k, dpad_of(d), sms) for n, k, d in shapes]
    bwd = [queue_bwd_plan(n, k, sms) for n, k, _ in shapes]
    tiles_f = [cdiv(k, 128 if dpad_of(d) > 128 else 256) for _, k, d in shapes]
    tiles_b = [cdiv(k, 128) for _, k, _ in shapes]
    assert any(nch == 1 for _, nch in fwd) and any(nch > 1 for _, nch in fwd), fwd
    assert any(nch == 1 for _, nch in bwd) and any(nch > 1 for _, nch in bwd), bwd
    assert any(nch > 1 and ct % tpc for (tpc, nch), ct in zip(fwd, tiles_f)), "no ragged last forward chunk"
    assert any(nch > 1 and ct % tpc for (tpc, nch), ct in zip(bwd, tiles_b)), "no ragged last backward chunk"
    assert any(4 * queue_fwd_plan(n, k, dpad_of(d), sms)[1] > 384 for n, k, d, _, _ in PIRL_CASES), "PIRL partials"
    assert any(4 * queue_bwd_plan(n, k, sms)[1] > 384 for n, k, _ in fused), "fused MoCo partials"
    assert {dpad_of(d) for _, _, d in shapes} >= {64, 128, 256}
    assert any(k % 128 for _, k, _ in shapes) and any(k < 128 for _, k, _ in shapes)
    assert any(n % 128 for n, _, _ in shapes)
