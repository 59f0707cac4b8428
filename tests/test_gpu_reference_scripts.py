"""SURVEY.md §8 f1 / b1: the reference's own scripts, UNMODIFIED, executed on the GPU against the drop-in modules.

tests/reference_script_driver.py exec's oracle/_ref/ia2c.py and oracle/_ref/a2c_org_test.py (staged by
oracle/make_ref.py, sha256-verified; loop length set by in-memory substitution as oracle/gen_golden.py did) in a
fresh interpreter whose path resolves ``Org``, ``ac_nets``, ``belief_filter`` and ``gymnasium`` to
ia2c_b200/compat(+compat_gym).  The golden run's sampled actions and np.random draws are replayed; everything the
script then computes must match the tapes recorded from the unmodified reference on the CPU:
env states / observations / rewards and beliefs bit-exact, losses / gradients / parameters within 1e-5."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.conftest import GOLDEN, ROOT
from tests.helpers import rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-5


def run_driver(script, golden_name, tmp_path):
    out = str(tmp_path / "out.npz")
    env = dict(os.environ)
    env.pop("PYTHONPATH", None)
    r = subprocess.run([sys.executable, "-P", os.path.join(ROOT, "tests", "reference_script_driver.py"), script,
                        os.path.join(GOLDEN, golden_name), out], capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=900)
    if r.returncode == 3 and "NO_REFERENCE" in r.stdout:
        pytest.skip("oracle/_ref not staged (IA2C_REFERENCE=<checkout of thinclab/IA2C> python -m oracle.make_ref)")
    assert r.returncode == 0 and "REFERENCE_SCRIPT_DONE" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
    return np.load(out, allow_pickle=False), r.stdout


def test_unmodified_ia2c_py_runs_on_the_gpu_and_matches_the_reference_tape(golden, tmp_path):
    g = golden("ia2c_E10.npz")
    o, stdout = run_driver("ia2c.py", "ia2c_E10.npz", tmp_path)
    episodes, T = int(g["meta_episodes"]), int(g["meta_T"])
    # same construction order + same torch / numpy seeds -> the script drew the reference's initial parameters and models
    for n in ("crit1", "crit2", "act1", "act2"):
        assert np.array_equal(o[f"{n}/init"][0], g[f"{n}/init"][0]), n
    for f in ("bf0", "bf1"):
        assert np.array_equal(o[f"{f}/filterAction"][0], g[f"{f}/filterAction"][0])
    # bit-exact: env observations (float32 [E,6]), rewards (float64), truncation, reset observations, episode returns
    assert o["env/obs"].dtype == np.float32 and o["env/reward"].dtype == np.float64
    assert np.array_equal(o["env/obs"], g["env/obs"]) and np.array_equal(o["env/reward"], g["env/reward"])
    assert np.array_equal(o["env/truncated"], g["env/truncated"]) and np.array_equal(o["env/reset_obs"], g["env/reset_obs"])
    assert np.array_equal(o["reward_lst"], g["reward_lst"])
    assert o["env/obs"].shape[0] == episodes * T
    # bit-exact: rounded posteriors and predicted actions of both filters, every call
    for f in ("bf0", "bf1"):
        assert np.array_equal(o[f"{f}/bprime"], g[f"{f}/bprime"]) and np.array_equal(o[f"{f}/ap"], g[f"{f}/ap"])
    # <= 1e-5: targets, advantages, losses, gradients (the actors' running sums, Q2), post-Adam parameters
    for c, a in (("crit1", "act1"), ("crit2", "act2")):
        assert o[f"{c}/target_requires_grad"].all()          # residual-gradient target (Q8)
        assert not o[f"{a}/adv_requires_grad"].any()         # gradient-free advantage in ia2c.py (Q7)
        for ep in range(episodes):
            assert np.array_equal(o[f"{c}/upd_obs"][ep], g[f"{c}/upd_obs"][ep])
            assert rel_err(o[f"{c}/upd_target"][ep], g[f"{c}/upd_target"][ep]) < RTOL
            assert rel_err(o[f"{c}/upd_loss"][ep], g[f"{c}/upd_loss"][ep]) < RTOL
            assert rel_err(o[f"{c}/upd_grad"][ep], g[f"{c}/upd_grad"][ep]) < RTOL
            assert rel_err(o[f"{c}/upd_params"][ep], g[f"{c}/upd_params"][ep]) < RTOL
            assert rel_err(o[f"{a}/upd_adv"][ep], g[f"{a}/upd_adv"][ep]) < RTOL
            assert rel_err(o[f"{a}/upd_loss"][ep], g[f"{a}/upd_loss"][ep]) < RTOL
            assert rel_err(o[f"{a}/upd_grad"][ep], g[f"{a}/upd_grad"][ep]) < RTOL
            assert rel_err(o[f"{a}/upd_params"][ep], g[f"{a}/upd_params"][ep]) < RTOL
    assert rel_err(o["critic_loss_window"], g["critic_loss_window"]) < RTOL
    assert rel_err(o["actor_loss_window"], g["actor_loss_window"]) < RTOL
    # the script's own progress line (ia2c.py:133-134) for episode 0: mean return and the four loss windows
    ours, theirs = stdout.splitlines()[0].split(), str(g["stdout"]).splitlines()[0].split()
    assert ours[0] == theirs[0] == "0" and rel_err([float(x) for x in ours[1:6]], [float(x) for x in theirs[1:6]]) < RTOL


def test_unmodified_a2c_org_test_py_runs_on_the_gpu_and_matches_the_reference_tape(golden, tmp_path):
    g = golden("a2c_org.npz")
    o, _ = run_driver("a2c_org_test.py", "a2c_org.npz", tmp_path)
    updates, T = int(g["meta_updates"]), int(g["meta_T"])
    assert np.array_equal(o["main1/init"][0], g["main1/init"][0]) and np.array_equal(o["act1/init"][0], g["act1/init"][0])
    # bit-exact: the single Org instance's state, fp64 reward and in-place observation over the whole 400-step walk
    assert o["org/state"].shape[0] == updates * T
    assert np.array_equal(o["org/state"], g["org/state"]) and np.array_equal(o["org/reward"], g["org/reward"])
    assert np.array_equal(o["org/obs"], g["org/obs"])
    assert o["act1/adv_requires_grad"].all()                  # differentiable advantage Q_cur - V (Q7)
    for u in range(updates):
        assert np.array_equal(o["main1/upd_obs"][u], g["main1/upd_obs"][u])          # ep_states == ep_next_states (Q4)
        assert np.array_equal(o["main1/upd_target"][u], g["main1/upd_target"][u])    # target == reward (Q5)
        for n in ("main1", "act1"):
            assert rel_err(o[f"{n}/upd_loss"][u], g[f"{n}/upd_loss"][u]) < RTOL, (n, u)
            assert rel_err(o[f"{n}/upd_grad"][u], g[f"{n}/upd_grad"][u]) < RTOL, (n, u)
            assert rel_err(o[f"{n}/upd_params"][u], g[f"{n}/upd_params"][u]) < RTOL, (n, u)
        assert rel_err(o["act1/upd_adv"][u], g["act1/upd_adv"][u]) < RTOL
    assert rel_err(o["critic_loss_window"], g["critic_loss_window"]) < RTOL
    assert rel_err(o["actor_loss_window"], g["actor_loss_window"]) < RTOL
