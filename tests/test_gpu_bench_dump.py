"""bench.py --dump-outputs on the GPU: the files hold what the last timed headline step computed (a trainer driven through the
same warm-up and timed episodes holds the same bytes), every file is float32 / float64, and a second run with the same
arguments writes the same bytes."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

from tests.conftest import ROOT
from tests.helpers import host

pytestmark = pytest.mark.gpu
ARGS = ["--gpus", "1", "--steps", "2", "--warmup", "3", "--repeats", "1", "--envs-per-gpu", "64", "--skip-cpu-baseline",
        "--skip-kernel-rooflines", "--skip-configs"]


def run_bench(out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *ARGS, "--dump-outputs", str(out)], capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    import torch

    import bench

    line = run_bench(tmp_path / "a")
    assert line["steps"] == 2 and line["warmup"] == 3
    run_bench(tmp_path / "b")
    names = sorted(f[:-4] for f in os.listdir(tmp_path / "a"))
    assert names == sorted(f[:-4] for f in os.listdir(tmp_path / "b"))
    dumped = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in names}
    for n, a in dumped.items():
        assert a.dtype in (np.float32, np.float64), n
        assert np.array_equal(a, np.load(tmp_path / "b" / f"{n}.npy")), n
    # the bench's trainer after its 3 warm-up episodes and one timed block of 2
    ctx = types.SimpleNamespace(dev=torch.device("cuda", 0), rank=0, world=1)
    tr = bench.make_trainer(ctx, 64, 2, fused=True)
    for _ in range(3 + 2):
        tr.train_episode()
    torch.cuda.synchronize()
    want = {"critic_loss": tr.loss_out[0], "actor_loss": tr.loss_out[1], "actor_params": tr.actor_params,
            "critic_params": tr.critic_params, "ep_return": tr.ep_return, "obs": tr.obs, "reward": tr.reward, "act": tr.act,
            "partner_pred": tr.partner_pred}
    assert set(names) == set(want) | {"env_index"}
    for n, t in want.items():
        assert np.array_equal(dumped[n], host(t).astype(dumped[n].dtype)), n
    assert np.array_equal(dumped["env_index"], np.arange(64))
