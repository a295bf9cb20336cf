"""bench.py on the B200: --dump-outputs writes what the timed path returned in its last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs(tmp_path):
    out_dir = tmp_path / "out"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--no-cpu",
                          "--no-per-config", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2 and d["parity_ok"]
    assert sorted(os.listdir(out_dir)) == ["dzi.npy", "dzj.npy", "loss.npy"]
    assert sum(os.path.getsize(out_dir / f) for f in os.listdir(out_dir)) <= 64 * 2 ** 20
    loss, dzi, dzj = (np.load(out_dir / f"{name}.npy") for name in ("loss", "dzi", "dzj"))
    assert loss.shape == () and loss.dtype == np.float32
    assert dzi.shape == dzj.shape == (32768, 128) and dzi.dtype == dzj.dtype == np.float32
    # the same seeded inputs as the step bench.py checks after the timed regions: the same loss
    assert abs(float(loss) - d["parity"]["loss"]) <= 1e-6 * abs(d["parity"]["loss"])

    # the dumped gradients against the closed form on bench.py's inputs (rank 0 of one GPU: seeds 100 / 101)
    from bench import parity_witness
    zi = torch.randn(32768, 128, generator=torch.Generator().manual_seed(100)).cuda()
    zj = torch.randn(32768, 128, generator=torch.Generator().manual_seed(101)).cuda()
    par = parity_witness(zi, zj, torch.from_numpy(dzi).cuda(), float(loss), 1, 0, None, dzj=torch.from_numpy(dzj).cuda())
    assert par["loss_rel"] <= 1e-3 and par["grad_rel_l2"] <= 1e-2, par
