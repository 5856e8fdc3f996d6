"""bench.py on the GPU: `--dump-outputs` writes what the timed fused call returned in its last step, computed on the
seeded bench inputs, so two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    import torch
    import smnngp_b200 as sm
    from oracle import nngp_oracle as orc
    from tests.synth import pixel_data, DEFAULT_HP as hp
    n, d = 2000, 784
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--rows", str(n), "--steps", "2",
                        "--warmup", "1", "--no-cpu-baseline", "--no-grad", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    assert line["steps"] == 2 and line["warmup"] == 1
    out, info = np.load(tmp_path / "out.npy"), np.load(tmp_path / "info.npy")
    assert out.dtype == np.float64 and out.shape == (4,) and info.tolist() == [0.0]
    assert out[1] == line["loss"]
    # the same seeded inputs in this process give the same outputs, and the loss is the oracle's
    x, y, *_ = pixel_data(n, d, seed=10)
    again, _ = sm.device.lml(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), spec=sm.StackSpec(3, "relu", "mlp"),
                             hp=sm.make_hp(device="cuda", **hp), kind="student_t")
    assert np.all(np.abs(again.cpu().numpy() - out) <= 1e-12 * np.abs(out)), (again, out)
    ref = orc.spr_loss(x, y, num_hiddens=3, act="relu", arch="mlp", w_std=hp["w_std"], b_std=hp["b_std"],
                       last_w_std=hp["last_w_std"], eps=hp["eps"], kind="student_t", a=hp["alpha"], b=hp["beta"])
    assert abs(out[1] - ref) <= 1e-8 * abs(ref)
