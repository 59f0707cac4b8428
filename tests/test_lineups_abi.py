"""CPU-side checks of the cross-play entry point: the ctypes mirror of ia2c_lineup_desc has the C layout, and
ia2c_evaluate_lineups / evaluate_lineups / cross_play refuse what they do not support before any device work."""
import ctypes as C
import os
import subprocess
import types

import numpy as np
import pytest

from tests.conftest import ROOT

HEADER = os.path.join(ROOT, "include", "ia2c_b200.h")
INVALID = -1


def test_lineup_desc_layout_matches_c(tmp_path):
    from ia2c_b200 import _lib
    fields = [f[0] for f in _lib.LineupDesc._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu", sizeof(ia2c_lineup_desc));' % HEADER
    for f in fields:
        prog += 'printf(" %%zu", offsetof(ia2c_lineup_desc, %s));' % f
    prog += 'printf(" %d %d", IA2C_EVAL_MAX_LINEUPS, IA2C_ABI_VERSION);return 0;}\n'
    c = tmp_path / "layout.c"
    c.write_text(prog)
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(c), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.LineupDesc)
    assert out[1:-2] == [getattr(_lib.LineupDesc, f).offset for f in fields]
    assert out[-2:] == [_lib.EVAL_MAX_LINEUPS, _lib.ABI_VERSION]
    assert _lib.EVAL_MAX_LINEUPS >= 1024 * 1024


def _desc(nets=6, N=3, P=4, E=37, K=2, T=30):
    """A descriptor whose pointers are non-NULL but point nowhere: every refusal below must come before the first device
    access."""
    from ia2c_b200 import _lib
    lib = _lib.load()
    d = _lib.LineupDesc()
    d.nets, d.N, d.P, d.E, d.episodes, d.T, d.max_episode_steps = nets, N, P, E, K, T, 30
    fake = 0x1000
    d.actor_params = d.lineups = d.policy = d.returns = d.action_counts = d.return_sum = d.return_m2 = fake
    d.policy_floats = nets * 27
    return lib, d


POINTERS = ("actor_params", "lineups", "policy", "returns", "action_counts", "return_sum", "return_m2")


@pytest.mark.parametrize("case, message", [
    ("null descriptor", "null descriptor"),
    *[(f"null {p}", "null actor_params") for p in POINTERS],
    ("N=1", "N=1"),
    ("N=1024", "N=1024"),
    ("nets=0", "nets=0"),
    ("P=0", "P=0"),
    ("P too large", "P=1048577"),
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
def test_evaluate_lineups_refuses_without_touching_a_device(case, message):
    from ia2c_b200 import _lib
    lib, d = _desc()
    if case == "null descriptor":
        assert lib.ia2c_evaluate_lineups(None, None) == INVALID
        assert message in lib.ia2c_last_error().decode()
        return
    if case.startswith("null "):
        setattr(d, case[5:], None)
    elif case == "N=1":
        d.N = 1
    elif case == "N=1024":
        d.N = 1024
    elif case == "nets=0":
        d.nets = 0
    elif case == "P=0":
        d.P = 0
    elif case == "P too large":
        d.P = _lib.EVAL_MAX_LINEUPS + 1
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
        d.policy_floats = d.nets * 27 - 1
    assert lib.ia2c_evaluate_lineups(C.byref(d), None) == INVALID
    assert message in lib.ia2c_last_error().decode(), lib.ia2c_last_error().decode()


class _Pool:
    """Stands in for the pool tensor: evaluate_lineups reads its shape on the host before any device work."""
    ndim = 2

    def __init__(self, nets):
        self.shape = (nets, 105)


@pytest.mark.parametrize("kwargs, match", [
    (dict(lineups=[[0, 6]]), r"lineups\[0, 1\] = 6 outside"),
    (dict(lineups=[[0, 1], [-1, 2]]), r"lineups\[1, 0\] = -1 outside"),
    (dict(lineups=[[0, 1, 2]]), "lineups must be"),
    (dict(lineups=[0, 1]), "lineups must be"),
    (dict(lineups=np.zeros((0, 2), dtype=np.int32)), "lineups must be"),
    (dict(lineups=[[0.0, 1.0]]), "lineups must be"),
    (dict(n_agents=1, lineups=[[0]]), "n_agents=1"),
    (dict(envs=0), "envs=0"),
    (dict(episodes=0), "episodes=0"),
    (dict(T=70000), "T=70000"),
    (dict(max_episode_steps=-3), "max_episode_steps=-3"),
    (dict(seed=-1), "seed=-1"),
    (dict(episode0=(1 << 32) - 1, episodes=2), "2\\*\\*32"),
    (dict(greedy=True), "greedy"),
])
def test_evaluate_lineups_refuses_before_any_device_work(kwargs, match):
    from ia2c_b200.evaluate import evaluate_lineups
    args = dict(actor_params=_Pool(6), n_agents=2, lineups=[[0, 1], [2, 3]], envs=4, episodes=1, T=30, max_episode_steps=30,
                greedy=False, seed=0, episode0=0, device="cuda")
    args.update(kwargs)
    with pytest.raises(ValueError, match=match):
        evaluate_lineups(**args)


def _source(cls, N=2, T=30, mes=30, device="cuda:0", R=3, E=10):
    """A trainer or batch with only the attributes cross_play reads before any device work (no GPU here)."""
    s = object.__new__(cls)
    s.N, s.T, s.device, s.R, s.E, s.E_total = N, T, device, R, E, E
    s.desc = types.SimpleNamespace(max_episode_steps=mes)
    return s


@pytest.mark.parametrize("change, match", [
    (dict(N=3), "must share"),
    (dict(T=20), "must share"),
    (dict(mes=10), "must share"),
    (dict(device="cuda:1"), "must share"),
])
def test_cross_play_refuses_mismatched_sources(change, match):
    from ia2c_b200.evaluate import cross_play
    from ia2c_b200.runs import IA2CRuns
    from ia2c_b200.trainer import IA2CTrainer
    with pytest.raises(ValueError, match=match):
        cross_play([_source(IA2CRuns), _source(IA2CTrainer, **change)])


@pytest.mark.parametrize("split", [0, 4, -1])
def test_cross_play_refuses_a_split_outside_the_seats(split):
    from ia2c_b200.evaluate import cross_play
    from ia2c_b200.runs import IA2CRuns
    with pytest.raises(ValueError, match=f"split={split}"):
        cross_play(_source(IA2CRuns, N=4), split=split)


def test_cross_play_refuses_other_sources_and_too_many_runs():
    from ia2c_b200.evaluate import cross_play
    from ia2c_b200.runs import IA2CRuns
    with pytest.raises(ValueError, match="a source must be"):
        cross_play([_source(IA2CRuns), "runs"])
    with pytest.raises(ValueError, match="no sources"):
        cross_play([])
    with pytest.raises(ValueError, match="1025 runs"):
        cross_play([_source(IA2CRuns, R=1000), _source(IA2CRuns, R=25)])
