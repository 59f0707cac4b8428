"""CPU-side checks of the evaluation entry point: the ctypes mirror of ia2c_eval_desc has the C layout, the policy workspace
is sized as documented, and ia2c_evaluate / evaluate_actors refuse what they do not support before any device work."""
import ctypes as C
import os
import subprocess

import pytest

from tests.conftest import ROOT

HEADER = os.path.join(ROOT, "include", "ia2c_b200.h")
INVALID = -1


def test_eval_desc_layout_matches_c(tmp_path):
    from ia2c_b200 import _lib
    fields = [f[0] for f in _lib.EvalDesc._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu", sizeof(ia2c_eval_desc));' % HEADER
    for f in fields:
        prog += 'printf(" %%zu", offsetof(ia2c_eval_desc, %s));' % f
    prog += 'printf(" %d %d %d %d", IA2C_EVAL_MAX_RUNS, IA2C_EVAL_MAX_AGENTS, IA2C_EVAL_MAX_STEPS, IA2C_ABI_VERSION);return 0;}\n'
    c = tmp_path / "layout.c"
    c.write_text(prog)
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(c), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.EvalDesc)
    assert out[1:-4] == [getattr(_lib.EvalDesc, f).offset for f in fields]
    assert out[-4:] == [_lib.EVAL_MAX_RUNS, _lib.EVAL_MAX_AGENTS, _lib.EVAL_MAX_STEPS, _lib.ABI_VERSION]


def _desc(R=3, N=5, E=37, K=2, T=30):
    """A descriptor whose pointers are non-NULL but point nowhere: every refusal below must come before the first device
    access."""
    from ia2c_b200 import _lib
    lib = _lib.load()
    d = _lib.EvalDesc()
    d.R, d.N, d.E, d.episodes, d.T, d.max_episode_steps = R, N, E, K, T, 30
    fake = 0x1000
    d.actor_params = d.policy = d.returns = d.action_counts = fake
    d.policy_floats = R * N * 27
    return lib, d


@pytest.mark.parametrize("case, message", [
    ("null descriptor", "null descriptor"),
    ("null actor_params", "null actor_params"),
    ("null policy", "null actor_params"),
    ("null returns", "null actor_params"),
    ("null counts", "null actor_params"),
    ("R=0", "R=0"),
    ("R too large", "R=65536"),
    ("N=1", "N=1"),
    ("N=1024", "N=1024"),
    ("R*N too large", "IA2C_MAX_RUN_NETS"),
    ("E=0", "E=0"),
    ("episodes=0", "episodes=0"),
    ("T=0", "T=0"),
    ("T too large", "T=65536"),
    ("negative time limit", "max_episode_steps=-1"),
    ("grid", "do not fit"),
    ("episode0 overflow", "2^32"),
    ("greedy with envs", "greedy needs"),
    ("greedy with tape", "no uniform tape"),
    ("small workspace", "policy workspace"),
])
def test_evaluate_refuses_without_touching_a_device(case, message):
    from ia2c_b200 import _lib
    lib, d = _desc()
    if case == "null descriptor":
        assert lib.ia2c_evaluate(None, None) == INVALID
        assert message in lib.ia2c_last_error().decode()
        return
    if case.startswith("null "):
        setattr(d, {"actor_params": "actor_params", "policy": "policy", "returns": "returns", "counts": "action_counts"}[case[5:]], None)
    elif case == "R=0":
        d.R = 0
    elif case == "R too large":
        d.R, d.N = _lib.EVAL_MAX_RUNS + 1, 2
    elif case == "N=1":
        d.N = 1
    elif case == "N=1024":
        d.N = 1024
    elif case == "R*N too large":
        d.R, d.N = 100, 1000
    elif case == "E=0":
        d.E = 0
    elif case == "episodes=0":
        d.episodes = 0
    elif case == "T=0":
        d.T = 0
    elif case == "T too large":
        d.T = _lib.EVAL_MAX_STEPS + 1
    elif case == "negative time limit":
        d.max_episode_steps = -1
    elif case == "grid":
        d.E, d.episodes = 1 << 40, 1 << 20
    elif case == "episode0 overflow":
        d.episode0 = (1 << 32) - 1
    elif case == "greedy with envs":
        d.greedy = 1
    elif case == "greedy with tape":
        d.greedy, d.E, d.episodes, d.inj_u_action = 1, 1, 1, 0x1000
    elif case == "small workspace":
        d.policy_floats = int(lib.ia2c_eval_policy_floats(C.byref(d))) - 1
    assert lib.ia2c_evaluate(C.byref(d), None) == INVALID
    assert message in lib.ia2c_last_error().decode(), lib.ia2c_last_error().decode()


def test_policy_floats_sizing():
    lib, d = _desc(R=3, N=5)
    assert int(lib.ia2c_eval_policy_floats(C.byref(d))) == 3 * 5 * 9 * 3
    d.R, d.N = 128, 2
    assert int(lib.ia2c_eval_policy_floats(C.byref(d))) == 128 * 2 * 27
    d.R = 0
    assert int(lib.ia2c_eval_policy_floats(C.byref(d))) == 0
    assert int(lib.ia2c_eval_policy_floats(None)) == 0


@pytest.mark.parametrize("kwargs, match", [
    (dict(R=0), "runs=0"),
    (dict(N=1), "n_agents=1"),
    (dict(N=1024), "n_agents=1024"),
    (dict(R=100, N=1000), "runs \\* n_agents"),
    (dict(envs=0), "envs=0"),
    (dict(episodes=0), "episodes=0"),
    (dict(T=70000), "T=70000"),
    (dict(max_episode_steps=-3), "max_episode_steps=-3"),
    (dict(seed=-1), "seed=-1"),
    (dict(seed=1 << 64), "seed="),
    (dict(episode0=(1 << 32) - 1, episodes=2), "2\\*\\*32"),
    (dict(greedy=True), "greedy"),
    (dict(greedy=True, envs=1, episodes=1, u_action=[0.5]), "greedy"),
])
def test_evaluate_actors_refuses_before_any_device_work(kwargs, match):
    from ia2c_b200.evaluate import evaluate_actors
    args = dict(actor_params=None, R=2, N=3, envs=4, episodes=1, T=30, max_episode_steps=30, greedy=False, seed=0, episode0=0,
                device="cuda")
    args.update(kwargs)
    with pytest.raises(ValueError, match=match):
        evaluate_actors(**args)
