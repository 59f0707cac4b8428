"""CPU-side checks of the PBT entry point: the ctypes mirror of ia2c_pbt_desc has the C layout, the symbols are exported, the
workspace query, and every refusal of ia2c_pbt_step and IA2CRuns.exploit_explore happens before any device work."""
import ctypes as C
import os
import subprocess
from types import SimpleNamespace

import pytest

from tests.conftest import ROOT

HEADER = os.path.join(ROOT, "include", "ia2c_b200.h")
INVALID, UNSUPPORTED = -1, -3


def test_pbt_desc_layout_matches_c(tmp_path):
    from ia2c_b200 import _lib
    fields = [f[0] for f in _lib.PbtDesc._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu", sizeof(ia2c_pbt_desc));' % HEADER
    for f in fields:
        prog += 'printf(" %%zu", offsetof(ia2c_pbt_desc, %s));' % f
    prog += 'printf(" %d %d %d %d", IA2C_PBT_LR_ACTOR, IA2C_PBT_LR_CRITIC, IA2C_PBT_BETA, IA2C_ABI_VERSION);return 0;}\n'
    c = tmp_path / "layout.c"
    c.write_text(prog)
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(c), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.PbtDesc)
    assert out[1:-4] == [getattr(_lib.PbtDesc, f).offset for f in fields]
    assert out[-4:-1] == [_lib.PBT_LR_ACTOR, _lib.PBT_LR_CRITIC, _lib.PBT_BETA]
    assert out[-1] == _lib.ABI_VERSION == 6


def test_pbt_symbols_are_exported():
    from ia2c_b200 import _lib
    lib = _lib.load()
    for name in ("ia2c_pbt_step", "ia2c_pbt_workspace_bytes"):
        assert hasattr(lib, name) and name in _lib.SIGNATURES


def test_workspace_query():
    from ia2c_b200 import _lib
    lib = _lib.load()
    assert [lib.ia2c_pbt_workspace_bytes(r) for r in (1, 2, 128, 32767)] == [4, 8, 512, 131068]
    assert lib.ia2c_pbt_workspace_bytes(0) == 0 and lib.ia2c_pbt_workspace_bytes(-3) == 0


def _descs(R=8, N=2, cap=4):
    """Descriptors whose pointers are non-NULL but point nowhere: every refusal below must come before the first device
    access."""
    from ia2c_b200 import _lib
    lib = _lib.load()
    fake = 0x1000
    d = _lib.EpisodeDesc()
    d.E, d.E_total, d.env_offset, d.N, d.T, d.M = 10, 10, 0, N, 30, 5
    for k in ("actor_params", "critic_params", "actor_m", "actor_v", "critic_m", "critic_v", "actor_step", "critic_step",
              "actor_grad_accum", "filter_action"):
        setattr(d, k, fake)
    r = _lib.RunsDesc()
    r.runs, r.seed = R, fake
    h = _lib.HistoryDesc()
    h.capacity, h.return_sum = cap, fake
    p = _lib.PbtDesc()
    p.window, p.slot, p.q, p.perturb, p.factor_lo, p.factor_hi = 2, 1, 2, 7, 0.8, 1.2
    for k in ("lr_actor", "lr_critic", "gamma", "beta", "log_fitness", "log_rank", "log_donor", "log_lr_actor", "log_lr_critic",
              "log_gamma", "log_beta", "workspace"):
        setattr(p, k, fake)
    p.workspace_bytes = 4 * R
    return lib, d, r, h, p


# the ten per-net buffers of the episode descriptor, the ring's return_sum, then the PBT descriptor's arrays
NULLS = ["actor_params", "critic_params", "actor_m", "actor_v", "critic_m", "critic_v", "actor_step", "critic_step",
         "actor_grad_accum", "filter_action", "return_sum", "lr_actor", "lr_critic", "gamma", "beta", "log_fitness", "log_rank",
         "log_donor", "log_lr_actor", "log_lr_critic", "log_gamma", "log_beta", "workspace"]


@pytest.mark.parametrize("case, status, message", [
    ("null episode descriptor", INVALID, "null episode, runs, history or pbt descriptor"),
    ("null runs descriptor", INVALID, "null episode, runs, history or pbt descriptor"),
    ("null history descriptor", INVALID, "null episode, runs, history or pbt descriptor"),
    ("null pbt descriptor", INVALID, "null episode, runs, history or pbt descriptor"),
    *[("null " + k, INVALID, "null") for k in NULLS],
    ("runs=0", INVALID, "runs=0"),
    ("N=0", INVALID, "N=0"),
    ("runs*N too large", INVALID, "IA2C_MAX_RUN_NETS"),
    ("capacity=1", INVALID, "capacity=1"),
    ("window=0", INVALID, "window=0"),
    ("window=capacity", INVALID, "window=4"),
    ("slot=-1", INVALID, "slot=-1"),
    ("slot=capacity", INVALID, "slot=4"),
    ("q=-1", INVALID, "q=-1"),
    ("2q > R", INVALID, "q=5"),
    ("perturb gamma bit", INVALID, "perturb=0x8"),
    ("factor 0", INVALID, "factors"),
    ("factor < 0", INVALID, "factors"),
    ("factor inf", INVALID, "factors"),
    ("factor nan", INVALID, "factors"),
    ("small workspace", INVALID, "workspace of 31 bytes"),
    ("env_offset", UNSUPPORTED, "one GPU"),
    ("E_total", UNSUPPORTED, "one GPU"),
])
def test_pbt_step_refuses_without_touching_a_device(case, status, message):
    lib, d, r, h, p = _descs()
    refs = [C.byref(d), C.byref(r), C.byref(h), C.byref(p)]
    if case.endswith(" descriptor"):
        refs[["null episode descriptor", "null runs descriptor", "null history descriptor", "null pbt descriptor"].index(case)] = None
    elif case.startswith("null "):
        field = case[5:]
        setattr(d if field in NULLS[:10] else (h if field == "return_sum" else p), field, None)
    elif case == "runs=0":
        r.runs = 0
    elif case == "N=0":
        d.N = 0
    elif case == "runs*N too large":
        r.runs = 65535 // 2 + 1
        p.workspace_bytes = 4 * r.runs
    elif case == "capacity=1":
        h.capacity, p.window, p.slot = 1, 1, 0
    elif case == "window=0":
        p.window = 0
    elif case == "window=capacity":
        p.window = 4
    elif case == "slot=-1":
        p.slot = -1
    elif case == "slot=capacity":
        p.slot = 4
    elif case == "q=-1":
        p.q = -1
    elif case == "2q > R":
        p.q = 5
    elif case == "perturb gamma bit":
        p.perturb = 8
    elif case.startswith("factor"):
        p.factor_hi = {"factor 0": 0.0, "factor < 0": -1.2, "factor inf": float("inf"), "factor nan": float("nan")}[case]
    elif case == "small workspace":
        p.workspace_bytes = 31
    elif case == "env_offset":
        d.env_offset = 10
    elif case == "E_total":
        d.E_total = 20
    assert lib.ia2c_pbt_step(*refs, None) == status
    assert message in lib.ia2c_last_error().decode(), lib.ia2c_last_error().decode()


def _batch(R=8, head=10, capacity=64, mark=0, ring=True):
    """An IA2CRuns built without __init__ (there is no device here), with a stand-in history ring."""
    from ia2c_b200.runs import IA2CRuns
    obj = IA2CRuns.__new__(IA2CRuns)
    obj.R = R
    obj._history = SimpleNamespace(head=head, capacity=capacity) if ring else None
    obj._pbt_mark = mark
    return obj


@pytest.mark.parametrize("kw, setup, message", [
    (dict(window=0), {}, "window=0"),
    (dict(window=64), {}, "window=64"),
    (dict(window=3), dict(capacity=4, head=10), None),
    (dict(window=4), dict(capacity=4, head=10), "window=4"),
    (dict(window=8), dict(ring=False), "no history ring"),
    (dict(window=8), dict(head=7), "only 7 episodes"),
    (dict(window=8), dict(head=20, mark=13), "only 7 episodes"),
    (dict(window=8, fraction=0.51), {}, "fraction=0.51"),
    (dict(window=8, fraction=-0.1), {}, "fraction=-0.1"),
    (dict(window=8, fraction=float("nan")), {}, "fraction=nan"),
    (dict(window=8, perturb=("lr_actor", "gamma")), {}, "gamma is inherited"),
    (dict(window=8, perturb=("lr",)), {}, "unknown hyper-parameter 'lr'"),
    (dict(window=8, perturb="beta2"), {}, "unknown hyper-parameter 'beta2'"),
    (dict(window=8, factors=(0.8, 0.0)), {}, "factors"),
    (dict(window=8, factors=(-0.8, 1.2)), {}, "factors"),
    (dict(window=8, factors=(0.8, float("inf"))), {}, "factors"),
    (dict(window=8, factors=(0.8,)), {}, "factors"),
    (dict(window=8, seed=-1), {}, "seed=-1"),
    (dict(window=8, seed=1 << 64), {}, "seed="),
])
def test_exploit_explore_refuses_before_device_work(kw, setup, message):
    obj = _batch(**setup)
    args = dict(fraction=0.25, perturb=("lr_actor", "lr_critic", "beta"), factors=(0.8, 1.2), seed=0)
    args.update(kw)
    window = args.pop("window")
    if message is None:   # accepted by the checks: window 3 of a 4-slot ring
        assert obj._pbt_args(window, **args) == (3, 2, 7, (0.8, 1.2), 0)
        return
    with pytest.raises(ValueError, match=message.replace("(", r"\(").replace(")", r"\)")):
        obj.exploit_explore(window, **args)
    assert obj._pbt_log is None and obj._pbt_generation == 0


def test_q_is_floor_of_fraction_times_runs():
    for R, fraction, q in ((8, 0.25, 2), (7, 0.5, 3), (10, 0.3, 3), (3, 0.25, 0), (1, 0.5, 0), (128, 0.5, 64)):
        assert _batch(R=R)._pbt_args(8, fraction, (), (1.0, 1.0), 0)[1] == q


def test_empty_pbt_history_has_the_documented_shapes():
    obj = _batch(R=5)
    out = obj.pbt_history()
    assert out["generation"].shape == out["episode"].shape == (0,)
    for k, dt in (("fitness", "float64"), ("rank", "int32"), ("donor", "int32"), ("lr_actor", "float64"),
                  ("lr_critic", "float64"), ("beta", "float32"), ("gamma", "float32")):
        assert out[k].shape == (0, 5) and out[k].dtype == dt, k


def test_pbt_log_capacity_is_a_class_attribute():
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    assert IA2CRuns.PBT_LOG_CAPACITY == IA2CRunsMany.PBT_LOG_CAPACITY == 16
