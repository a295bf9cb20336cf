#!/usr/bin/env python
"""bench.py — BASELINE.json's metric: NT-Xent fwd+bwd samples/s (and fraction of the tensor roofline)
at global batch 32768 x 128-d, tau = 0.5, normalize = True, on 1/2/4/8 B200.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our CUDA path
    python bench.py --dump-outputs DIR [...]                        # ... and write its last step's outputs to DIR
    python bench.py --impl reference [...]                          # CPU arm (oracle port, host cores)
    torchrun --nproc-per-node N bench.py --gpus N ...               # N > 1: one rank per GPU, NCCL

One "step" = one forward + backward of SimclrLoss over the global batch (strong scaling: the global batch
is fixed, rank r owns 32768/N rows per view; SURVEY.md §8e).  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "self-supervised-vision_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

N_GLOBAL = 32768          # images per step ("B=32768"): M = 65536 embedding rows
DIM = 128
TAU = 0.5
METRIC = "ntxent_fwd_bwd_samples_per_s"
WORKLOAD = "SimCLR global-batch NT-Xent 32768x128-d (M=65536 rows), tau=0.5, normalize=True (BASELINE configs[4])"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            pk = json.load(f)
        return {"bf16_tflops": pk.get("bf16_tflops", 1590.0), "bf16_tflops_sustained": pk.get("bf16_tflops_sustained"),
                "hbm_gbs": pk.get("hbm_gbs", 6650.0), "source": "measured"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


# ----------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    """`nvidia-smi -lms 20` in the background, started early (it needs a few hundred ms before its first sample);
    `mark()` stamps the start of the region of interest and `stop()` keeps the samples taken from then on (warm-up +
    timed region), so idle samples from set-up do not dilute the clocks-under-load figure."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.t_mark = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "20", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def mark(self):
        import datetime
        self.t_mark = datetime.datetime.now()

    def stop(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f")
                rows.append((ts, float(parts[2]), float(parts[3]), [nm for nm, v in zip(names, parts[5:9]) if v.lower() == "active"]))
            except ValueError:
                continue
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if self.t_mark is not None:
            inside = [r for r in rows if r[0] >= self.t_mark - datetime.timedelta(milliseconds=20)]
            rows = inside if len(inside) >= 3 else rows[-10:]   # a very short region: the last samples before the stop
        if rows:
            clocks = [r[1] for r in rows]
            reasons = sorted({nm for r in rows for nm in r[3]})
            # median over the upper half of the samples == "under load" (idle gaps between steps drop out)
            top = sorted(clocks)[len(clocks) // 2:]
            out.update(sm_mhz=statistics.median(top), sm_max_mhz=rows[-1][2], reasons=reasons, samples=len(clocks))
        return out


# ----------------------------------------------------------------------------------------- CPU arm
def cpu_sample(rows=4096, reps=1):
    from oracle import cpu_port
    r = cpu_port.time_ntxent_sample(N_GLOBAL, DIM, TAU, rows=rows, reps=reps, threads=os.cpu_count())
    return r


REF_SAMPLE_N = 4096   # the reference's classes materialise ~14 N^2 floats: N = 32768 needs > 150 GB (SURVEY.md §3.2)


def reference_step_fn(n):
    """One fwd+bwd of the UNMODIFIED reference SimclrLoss (utils/losses.py:8-46) at per-view batch n on the host
    cores, or None when no staged copy of the reference exists (oracle/make_ref.py -> baseline/_ref)."""
    import torch
    from oracle import ref_loader
    R = ref_loader.load()
    if R is None:
        return None
    torch.set_num_threads(os.cpu_count())
    g = torch.Generator().manual_seed(0)
    zi = torch.randn(n, DIM, generator=g).requires_grad_(True)
    zj = torch.randn(n, DIM, generator=g).requires_grad_(True)
    fn = R.losses.SimclrLoss(True, TAU)

    def step():
        zi.grad = None
        zj.grad = None
        loss = fn(zi, zj)
        loss.backward()
        return float(loss)
    return step


def extrapolate(n_sample, sec):
    """fwd+bwd time grows with N^2 beyond cache (SURVEY.md §6: 365 ms / 1.365 s at N = 2048 / 4096), so
    samples/s at N_GLOBAL = (n_sample / sec) * n_sample / N_GLOBAL."""
    return (n_sample / sec) * n_sample / N_GLOBAL


def cpu_baseline_leg():
    """cpu_baseline of our arm (rank 0, N = 1): the reference's own classes when staged, beside the slab port."""
    import torch
    out = {}
    port = cpu_sample(rows=4096, reps=2)
    port_d = {"value": port["samples_per_s"], "unit": "samples/s", "cores": port["threads"], "kind": "port",
              "sample": (f"{port['reps']} row slabs of {port['rows']} of the {port['m']} similarity rows x all columns "
                         f"(each {port['rows']}/{port['m']} of the full job), torch CPU fp32 closed form fwd+bwd, "
                         f"{port['seconds']:.2f} s per slab")}
    series = []
    for n, reps in ((1024, 3), (4096, 3), (8192, 1)):
        step = reference_step_fn(n)
        if step is None:
            break
        step()
        t0 = time.perf_counter()
        for _ in range(reps):
            step()
        sec = (time.perf_counter() - t0) / reps
        series.append({"n": n, "seconds": sec, "samples_per_s": n / sec, "extrapolated_to_32768": extrapolate(n, sec)})
    if series:
        last = series[-1]
        out = {"value": last["extrapolated_to_32768"], "unit": "samples/s", "cores": torch.get_num_threads(),
               "kind": "reference", "extrapolated": True,
               "sample": (f"the reference's own SimclrLoss(True, {TAU}) fwd+bwd (utils/losses.py:8-46, unmodified, "
                          f"baseline/_ref) at N = {last['n']} ({last['seconds']:.2f} s), extrapolated ~N^2 to N = {N_GLOBAL} "
                          f"because the reference needs > 150 GB of N x N intermediates there"),
               "series": series, "port": port_d}
    else:
        out = dict(port_d)
        out["note"] = "no staged reference (baseline/_ref): oracle port only"
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import cpu_port
    torch.set_num_threads(os.cpu_count())
    m = 2 * N_GLOBAL
    step = reference_step_fn(REF_SAMPLE_N)
    if step is not None:
        kind = "reference"
        sample = (f"each step = one fwd+bwd of the reference's own SimclrLoss(True, {TAU}) (utils/losses.py:8-46, "
                  f"unmodified copy in baseline/_ref) at N = {REF_SAMPLE_N} on the host cores; value extrapolated ~N^2 to "
                  f"N = {N_GLOBAL} (the reference cannot run that size: > 150 GB of N x N intermediates)")
        to_value = lambda dt: extrapolate(REF_SAMPLE_N, dt)  # noqa: E731
    else:
        kind = "port"
        rows = 4096
        g = torch.Generator().manual_seed(0)
        zi = torch.randn(N_GLOBAL, DIM, generator=g)
        zj = torch.randn(N_GLOBAL, DIM, generator=g)

        def step():
            zhat = torch.nn.functional.normalize(torch.cat([zi, zj]), dim=-1)
            loss_sum, d_rows, d_cols = cpu_port.ntxent_row_slab(zhat, N_GLOBAL, 0, rows, TAU)
            d_cols[:rows] += d_rows
            return float(loss_sum)
        sample = (f"row slab: {rows} of the {m} similarity rows x all {m} columns per step (= {rows}/{m} of the full "
                  f"6*M^2*d job), torch CPU fp32, fwd + both gradient GEMMs (no staged reference found)")
        to_value = lambda dt: (N_GLOBAL * rows / m) / dt  # noqa: E731

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    value = to_value(dt)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": N_GLOBAL, "dim": DIM},
            "cpu_baseline": {"value": value, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": kind,
                             "extrapolated": kind == "reference", "sample": sample},
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------- parity witness
def parity_witness(zi, zj, dzi, loss_value, world, rank, dist_mod, rows=4096, tau=TAU, dzj=None):
    """Loss and gradient of the global batch from a chunked fp32 closed form on the GPU (plain torch.matmul, TF32
    off; reference math utils/losses.py:15-46 restated as in SURVEY.md §8 a1), compared with what the kernels
    produced: the global loss, and the gradient of this rank's first `rows` rows of view i.  Runs once, outside the
    timed region; max over ranks."""
    import torch
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = zi.device
    n_local = zi.shape[0]
    with torch.no_grad():
        if world > 1:
            gi = [torch.empty_like(zi) for _ in range(world)]
            gj = [torch.empty_like(zj) for _ in range(world)]
            dist_mod.all_gather(gi, zi.detach().contiguous())
            dist_mod.all_gather(gj, zj.detach().contiguous())
            zgi, zgj = torch.cat(gi), torch.cat(gj)
        else:
            zgi, zgj = zi.detach(), zj.detach()
        n = zgi.shape[0]
        m = 2 * n
        z = torch.cat([zgi, zgj])
        nrm = z.norm(dim=1, keepdim=True).clamp_min(1e-12)
        zh = z / nrm
        lse = torch.empty(m, device=dev)
        for c0 in range(0, m, rows):
            s = zh[c0:c0 + rows] @ zh.t() / tau
            idx = torch.arange(c0, min(c0 + rows, m), device=dev)
            s[idx - c0, idx] = float("-inf")
            lse[c0:c0 + rows] = torch.logsumexp(s, dim=1)
        pos = (zh[:n] * zh[n:]).sum(1) / tau
        loss_w = (lse.double().sum() - 2.0 * pos.double().sum()) / m
        r0 = rank * n_local
        rr = min(rows, n_local)
        idx = torch.arange(r0, r0 + rr, device=dev)
        s = zh[idx] @ zh.t() / tau
        w = torch.exp(s - lse[idx, None]) + torch.exp(s - lse[None, :])
        w[torch.arange(rr, device=dev), idx] = 0.0
        g = (w @ zh - 2.0 * zh[idx + n]) / (m * tau)
        g = (g - (g * zh[idx]).sum(1, keepdim=True) * zh[idx]) / nrm[idx]
        loss_rel = abs(float(loss_value) - float(loss_w)) / abs(float(loss_w))
        grad_rel = float((dzi[:rr].double() - g.double()).norm() / g.double().norm())
        if dzj is not None:   # the same rows of view j (global rows n + idx)
            s = zh[idx + n] @ zh.t() / tau
            w = torch.exp(s - lse[idx + n, None]) + torch.exp(s - lse[None, :])
            w[torch.arange(rr, device=dev), idx + n] = 0.0
            g = (w @ zh - 2.0 * zh[idx]) / (m * tau)
            g = (g - (g * zh[idx + n]).sum(1, keepdim=True) * zh[idx + n]) / nrm[idx + n]
            grad_rel = max(grad_rel, float((dzj[:rr].double() - g.double()).norm() / g.double().norm()))
        t = torch.tensor([loss_rel, grad_rel], dtype=torch.float64, device=dev)
        if world > 1:
            dist_mod.all_reduce(t, op=dist_mod.ReduceOp.MAX)
    return {"loss_rel": t[0].item(), "grad_rel_l2": t[1].item(), "loss": float(loss_value), "witness_loss": float(loss_w),
            "grad_rows_checked_per_rank": rr, "tolerance": {"loss_rel": 1e-3, "grad_rel_l2": 1e-2},
            "witness": "chunked fp32 closed form on the GPU (torch.matmul, TF32 off) over the gathered global batch; "
                       "max over ranks"}


def dump_outputs(out_dir, arrays):
    """Writes each tensor as out_dir/<name>.npy in float32, so that two builds run with the same arguments (hence the
    same seeded inputs) can be compared output by output.  At one GPU that is the loss and both 32768 x 128 gradients:
    32 MiB in all."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


# ----------------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    import ssv_b200
    from ssv_b200 import _cabi
    from ssv_b200.dist import DistributedSimclrLoss

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus N>1 must be launched with torchrun (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # nvidia-smi needs a few hundred ms before its first sample: start it now so that it is sampling every 20 ms by the
    # time the warm-up and the timed region run (the timed region of the default run lasts only ~60 ms)
    sampler = ClockSampler(local_rank)
    sampler.start()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _cabi.lib()
    _cabi.check(L.ssvb_device_check(), "ssvb_device_check")

    n_local = N_GLOBAL // world
    m = 2 * N_GLOBAL
    # synthetic embeddings (SURVEY.md §8d cfg5): rank r rows seeded 100+2r / 101+2r, made on the host
    gi = torch.Generator().manual_seed(100 + 2 * rank)
    gj = torch.Generator().manual_seed(101 + 2 * rank)
    h_zi = torch.randn(n_local, DIM, generator=gi).pin_memory()
    h_zj = torch.randn(n_local, DIM, generator=gj).pin_memory()
    zi = h_zi.to(dev).requires_grad_(True)
    zj = h_zj.to(dev).requires_grad_(True)
    loss_fn = ssv_b200.SimclrLoss(True, TAU) if world == 1 else DistributedSimclrLoss(True, TAU)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2
    last = {}

    def step_resident():
        zi.grad = None
        zj.grad = None
        loss = loss_fn(zi, zj)
        loss.backward()
        last["loss"] = loss
        return loss

    # e2e: what a training loop does — the next step's inputs travel host->device on a side stream (pinned memory,
    # double-buffered) while the current step computes.  EVERY step's H2D copy is issued inside a timed region (the
    # copy for step t+1 is enqueued right after step t's start event), and every step ends with the D2H read of its
    # loss and a stream synchronize, like `loss.item()` in the reference loop (models/simclr.py:95).
    copy_stream = torch.cuda.Stream(device=dev)
    d_in = [(torch.empty(n_local, DIM, device=dev), torch.empty(n_local, DIM, device=dev)) for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    h_loss = torch.empty((), dtype=torch.float32).pin_memory()
    st = {"t": 0}

    def issue_copy(slot, first_use):
        with torch.cuda.stream(copy_stream):
            if not first_use:
                copy_stream.wait_event(consumed[slot])  # the step that read this buffer pair has finished with it
            d_in[slot][0].copy_(h_zi, non_blocking=True)
            d_in[slot][1].copy_(h_zj, non_blocking=True)
            copied[slot].record(copy_stream)

    def step_e2e():
        t = st["t"]
        slot = t & 1
        if t == 0:
            issue_copy(slot, True)          # the very first step waits for its own copy
        issue_copy(slot ^ 1, t == 0)        # inputs of step t+1: overlap with this step's kernels
        torch.cuda.current_stream().wait_event(copied[slot])
        a = d_in[slot][0].detach().requires_grad_(True)
        b = d_in[slot][1].detach().requires_grad_(True)
        loss = loss_fn(a, b)
        loss.backward()
        h_loss.copy_(loss.detach(), non_blocking=True)
        consumed[slot].record()
        torch.cuda.current_stream().synchronize()  # the caller reads the loss (loss.item() in the reference loop)
        st["t"] = t + 1
        return float(h_loss)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, profile=False):
        for _ in range(warmup):
            fn()
        barrier()
        evs = []
        if profile:
            L.ssvb_launch_count(1)
            L.ssvb_profile_enable(1)
        for _ in range(steps):
            flush.zero_()  # evict L2 between timed iterations (not timed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        barrier()
        launches = L.ssvb_launch_count(0) if profile else 0
        prof = {}
        if profile:
            for kind, name in ((0, "sim_fwd"), (1, "sim_bwd")):
                ms, cnt = ctypes.c_double(0), ctypes.c_longlong(0)
                L.ssvb_profile_summary(kind, ctypes.cast(ctypes.pointer(ms), ctypes.c_void_p),
                                       ctypes.cast(ctypes.pointer(cnt), ctypes.c_void_p))
                prof[name] = (ms.value, cnt.value)
            L.ssvb_profile_enable(0)
        total_ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item() / steps, launches, prof

    sampler.mark()
    ms_step, launches, prof = timed(step_resident, args.steps, args.warmup, profile=True)
    clocks = sampler.stop()
    # what the last timed step handed its caller; the steps below allocate fresh gradients and leave these untouched
    outputs = {"loss": last["loss"], "dzi": zi.grad, "dzj": zj.grad}
    ms_e2e, _, _ = timed(step_e2e, args.steps, max(3, args.warmup // 2))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)

    # correctness evidence carried by the bench line itself (every N): one more step, outside the timed regions
    zi.grad = None
    zj.grad = None
    loss_chk = loss_fn(zi, zj)
    loss_chk.backward()
    torch.cuda.synchronize()
    parity = parity_witness(zi, zj, zi.grad, loss_chk.item(), world, rank, dist)
    parity_ok = parity["loss_rel"] <= 1e-3 and parity["grad_rel_l2"] <= 1e-2

    peaks = load_peaks()
    value = N_GLOBAL / (ms_step * 1e-3)
    e2e_value = N_GLOBAL / (ms_e2e * 1e-3)
    # algorithmic FLOPs (SURVEY.md §8d): 6*M^2*d per step over all ranks; the dominant kernel (sim_bwd_kernel,
    # recompute S + dZ GEMM) carries 4*(M/world)*M*d per launch, sim_fwd_kernel 2*(M/world)*M*d.
    bwd_ms = prof["sim_bwd"][0] / max(prof["sim_bwd"][1], 1)
    fwd_ms = prof["sim_fwd"][0] / max(prof["sim_fwd"][1], 1)
    bwd_flops = 4.0 * (m / world) * m * DIM
    fwd_flops = 2.0 * (m / world) * m * DIM
    achieved = bwd_flops / (bwd_ms * 1e-3) / 1e12
    # denominator: the burst cuBLAS figure, unless the clock record shows the power cap biting during the timed
    # region (a long back-to-back run) - then the sustained figure is the like-for-like one (B200_PROFILING.md)
    capped = "sw_power_cap" in clocks.get("reasons", []) and peaks.get("bf16_tflops_sustained")
    peak = peaks["bf16_tflops_sustained"] if capped else peaks["bf16_tflops"]
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if world == 1 and os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("sim_bwd_kernel")  # bytes per launch from the committed ncu capture
    roofline = {"bound": "tensor", "kernel": "sim_bwd_kernel<KB=2, SIM_NTX_FIXED, OPF16=1>", "achieved": achieved, "peak": peak,
                "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this "
                                  "kernel at this shape (profiles/traffic.json), not measured in this run",
                "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": f"{peaks['source']} {'sustained (sw_power_cap active)' if capped else 'burst'} bf16 "
                               f"(MEASURED_PEAKS.json)",
                "frac_of_burst": achieved / peaks["bf16_tflops"],
                "kernel_ms": bwd_ms, "flops_per_launch": bwd_flops,
                "fwd_kernel": {"name": "sim_fwd_kernel<KB=2, SIM_NTX_FIXED, OPF16=1>", "ms": fwd_ms,
                               "achieved": fwd_flops / (fwd_ms * 1e-3) / 1e12,
                               "frac": fwd_flops / (fwd_ms * 1e-3) / 1e12 / peak},
                "step": {"flops": 6.0 * m * m * DIM, "achieved": 6.0 * m * m * DIM / (ms_step * 1e-3) / 1e12 / world,
                         "frac": 6.0 * m * m * DIM / (ms_step * 1e-3) / 1e12 / world / peak},
                "frac_of_sustained": (achieved / peaks["bf16_tflops_sustained"]) if peaks.get("bf16_tflops_sustained") else None}

    line = None
    if rank == 0:
        cpu = None
        per_config = None
        if world == 1 and not args.no_cpu:
            cpu = cpu_baseline_leg()
        if world == 1 and not args.no_per_config:
            # every BASELINE config (and the other §8 rows) beside its CPU arm and the reference run eagerly on this B200
            import bench_losses
            del flush
            torch.cuda.empty_cache()
            per_config = bench_losses.run_all(dev, reps=10, cpu=not args.no_cpu, ref_gpu=True,
                                              only=("cfg1", "cfg2", "cfg3", "cfg4", "swav", "rowdot128", "rowdot1024",
                                                    "relic512", "relic4096", "ntx8192"))
        line = {"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f16", "data": "synthetic",
                "dtype_detail": "fp16 tensor-core operands (unit-norm rows scaled by sqrt(log2(e)/tau); bf16 for raw "
                                "inputs), fp32 accumulation / statistics / loss / gradients",
                "config": {"workload": WORKLOAD, "global_batch": N_GLOBAL, "dim": DIM, "rows_per_rank": 2 * n_local,
                           "parallelism": f"row-sharded x{world}, all-gather zhat + lse", "l2": "flushed (256 MiB write) between timed iterations",
                           "per_config_l2": "flushed between repetitions by a 256 MiB write followed by a 256 MiB read "
                                            "(cold and clean lines, bench_losses.l2_flush)"},
                "roofline": roofline, "cpu_baseline": cpu,
                "e2e": {"value": e2e_value, "unit": "samples/s", "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": 2 * n_local * DIM * 4 * world, "d2h_bytes_per_step": 4 * world,
                        "pipeline": "H2D of step t+1 (pinned, side stream, double-buffered) overlaps the kernels of step t; "
                                    "every copy is issued inside a timed step; each step ends with the loss D2H + sync"},
                "gpu_launches": int(launches), "clocks": clocks, "parity": parity, "parity_ok": parity_ok,
                "per_config": per_config}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not parity_ok:
        raise SystemExit(f"parity check failed: {parity}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-per-config", action="store_true", help="skip the per_config array (the other BASELINE configs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss and the gradients of the last timed step (rank 0's "
                         "rows) as DIR/loss.npy, DIR/dzi.npy, DIR/dzj.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
