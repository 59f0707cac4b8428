"""bench.py contract checks that need no GPU: the reference arm (the unmodified reference loop from oracle/_ref on the host CPU,
or the oracle port when the staged copy is absent) prints one JSON line with the agreed keys."""
import json
import os
import subprocess
import sys
import types

from tests.conftest import ROOT


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--cpu-envs", "64"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "agent-steps/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("agent-steps/sec") and line["value"] > 0 and line["steps"] == 2
    from oracle import ref_runner
    have_ref = ref_runner.find_reference()[0] is not None
    assert line["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    assert line["cpu_baseline"]["cores"] >= 1 and "sample" in line["cpu_baseline"] and line["warmup"] == 1
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_other_ranks_exit_silently():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_samples_envs_within_the_byte_budget(tmp_path, monkeypatch):
    """Above the budget the per-env arrays keep the same fixed, seeded envs in every file and on every call."""
    import numpy as np
    import torch

    import bench

    E, N, T = 5000, 2, 30
    g = torch.Generator().manual_seed(0)
    tr = types.SimpleNamespace(E=E, env_offset=0, loss_out=torch.rand(2, N, generator=g),
                               actor_params=torch.rand(N, 105, generator=g), critic_params=torch.rand(N, 147, generator=g),
                               ep_return=torch.rand(E, dtype=torch.float64, generator=g), obs=torch.rand(T + 1, E, 6, generator=g),
                               reward=torch.rand(T, E, generator=g), act=torch.randint(0, 3, (T + 1, E, N), dtype=torch.uint8, generator=g),
                               partner_pred=torch.randint(0, 3, (T + 1, E, N), dtype=torch.uint8, generator=g))
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    for d in ("a", "b"):
        os.makedirs(tmp_path / d)
        bench.dump_outputs(tr, str(tmp_path / d))
    out = {f[:-4]: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert all(np.array_equal(a, np.load(tmp_path / "b" / f"{n}.npy")) for n, a in out.items())
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(os.path.getsize(tmp_path / "a" / f"{n}.npy") for n in out) <= 1 << 20
    keep = out["env_index"].astype(np.int64)
    assert 0 < len(keep) < E and np.all(np.diff(keep) > 0)
    assert np.array_equal(out["obs"], tr.obs.numpy()[:, keep]) and np.array_equal(out["ep_return"], tr.ep_return.numpy()[keep])
    assert np.array_equal(out["act"], tr.act.numpy()[:, keep].astype(np.float32))
    assert np.array_equal(out["critic_loss"], tr.loss_out[0].numpy()) and np.array_equal(out["critic_params"], tr.critic_params.numpy())


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "--dump-outputs needs --impl ours" in r.stderr


def test_our_arm_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
