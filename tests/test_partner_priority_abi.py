"""CPU-side checks of prioritized partners per env: the ctypes mirror of ia2c_partner_priority_desc has the C layout, the
symbols are exported, every refusal of the prioritized twins, ia2c_record_partner_returns, ia2c_prioritize_partners and of
the Python interface happens before any device work, and the two new kernels read nothing before their
griddepcontrol.wait."""
import ctypes as C
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.conftest import ROOT
from tests.test_env_partners_abi import CASES, STANDALONE_ONLY, _descs, _pool, _trainer

HEADER = os.path.join(ROOT, "include", "ia2c_b200.h")
INVALID, UNSUPPORTED = -1, -3
ENTRIES = ("ia2c_rollout_env_partners_prioritized", "ia2c_train_episode_env_partners_prioritized", "ia2c_record_partner_returns",
           "ia2c_prioritize_partners")
FAKE = 0x1000


def test_partner_priority_desc_layout_matches_c(tmp_path):
    from ia2c_b200 import _lib
    fields = [f[0] for f in _lib.PartnerPriorityDesc._fields_]
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu", sizeof(ia2c_partner_priority_desc));'
            % HEADER)
    for f in fields:
        prog += 'printf(" %%zu", offsetof(ia2c_partner_priority_desc, %s));' % f
    prog += 'printf(" %d %d", IA2C_ABI_VERSION, IA2C_PARTNER_PRIORITY_MAX_CELLS);return 0;}\n'
    c = tmp_path / "layout.c"
    c.write_text(prog)
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(c), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.PartnerPriorityDesc)
    assert out[1:-2] == [getattr(_lib.PartnerPriorityDesc, f).offset for f in fields]
    assert fields == ["count", "sum", "table", "R", "Q"]
    assert out[-2] == _lib.ABI_VERSION == 6
    assert out[-1] == _lib.PARTNER_PRIORITY_MAX_CELLS == 1 << 24


def test_partner_priority_symbols_are_exported_and_declared():
    from ia2c_b200 import _lib
    lib = _lib.load()
    header = open(HEADER).read()
    for name in ENTRIES:
        assert hasattr(lib, name) and name in _lib.SIGNATURES
        assert re.search(r"\bint %s\(" % name, header), name


def _prio(R=4, Q=3):
    from ia2c_b200 import _lib
    w = _lib.PartnerPriorityDesc()
    w.count, w.sum, w.table, w.R, w.Q = FAKE, FAKE, FAKE, R, Q
    return w


@pytest.mark.parametrize("case, status, message", CASES)
@pytest.mark.parametrize("entry", ["train_batch", "train_standalone", "rollout"])
def test_prioritized_twins_refuse_what_the_uniform_entries_refuse(case, status, message, entry):
    """The per-env mode's refusals, through the prioritized twins with a valid priority descriptor."""
    from ia2c_b200 import _lib
    lib, d, r, p = _descs()
    batch = entry == "train_batch"
    if not batch and case in ("null seed", "runs=0", "runs*N too large"):
        pytest.skip("a standalone run has no runs descriptor")
    if batch and case in STANDALONE_ONLY:
        pytest.skip("a batch always runs the fused or the whole-episode rollout")
    w = _prio(R=r.runs if batch else 1, Q=p.Q)
    dref, pref = C.byref(d), C.byref(p)
    if case == "null episode descriptor":
        dref = None
    elif case == "null partner descriptor":
        pref = None
    elif case == "null seed":
        r.seed = None
    elif case.startswith("null policy"):
        d.N, d.flags, p.policy = 16, _lib.FLAG_ACTOR_COLUMNS, None
    elif case.startswith("null "):
        setattr(p, case[5:], None)
    elif case == "runs=0":
        r.runs = 0
    elif case == "N=1":
        d.N = 1
    elif case == "runs*N too large":
        r.runs = 65535 // 3 + 1
    elif case in ("S=0", "S=N"):
        p.S = 0 if case == "S=0" else 3
    elif case == "P=0":
        p.P = 0
    elif case == "Q=0":
        p.Q = 0
    elif case == "Q too large":
        p.Q = (1 << 20) + 1
    elif case == "env_offset":
        d.env_offset = 10
    elif case == "E_total":
        d.E_total = 20
    elif case == "injected actions":
        d.inj_actions = FAKE
    elif case == "N > 256":
        d.N, d.flags = 300, _lib.FLAG_ACTOR_COLUMNS
    elif case == "M without a fused instantiation":
        d.M, d.flags = 4, 0 if not batch else d.flags
    elif case == "fused_rollout off":
        d.flags = 0
    elif case in ("ROLLOUT_PER_STEP", "BELIEF_PER_STEP"):
        d.N, d.flags = 16, getattr(_lib, "FLAG_" + case)
    elif case == "no whole-episode belief kernel":
        d.N, d.M, d.flags = 16, 7, 0
    if entry == "rollout":
        rc = lib.ia2c_rollout_env_partners_prioritized(dref, pref, C.byref(w), None)
    else:
        rc = lib.ia2c_train_episode_env_partners_prioritized(dref, C.byref(r) if batch else None, pref, C.byref(w), None)
    assert rc == status
    assert message in lib.ia2c_last_error().decode(), lib.ia2c_last_error().decode()


PRIO_CASES = [
    ("null priority descriptor", "null priority descriptor"),
    ("null count", "null count, sum or table"),
    ("null sum", "null count, sum or table"),
    ("null table", "null count, sum or table"),
    ("R=0", "R=0"),
    ("Q=0", "Q=0"),
    ("Q too large", "Q=1048577"),
    ("R*Q too large", "IA2C_PARTNER_PRIORITY_MAX_CELLS"),
]


def _break_prio(w, case):
    if case.startswith("null ") and case != "null priority descriptor":
        setattr(w, case[5:], None)
    elif case == "R=0":
        w.R = 0
    elif case == "Q=0":
        w.Q = 0
    elif case == "Q too large":
        w.Q = (1 << 20) + 1
    elif case == "R*Q too large":
        w.R, w.Q = 17, 1 << 20
    return None if case == "null priority descriptor" else C.byref(w)


@pytest.mark.parametrize("case, message", PRIO_CASES + [("R != runs", "priority R=3, but 4 runs"),
                                                        ("Q != pool Q", "priority Q=2, but the pool has Q=3")])
@pytest.mark.parametrize("entry", ["train_batch", "train_standalone", "rollout"])
def test_prioritized_twins_refuse_bad_priority_descriptors(case, message, entry):
    lib, d, r, p = _descs()
    batch = entry == "train_batch"
    w = _prio(R=r.runs if batch else 1, Q=p.Q)
    if case == "R != runs":
        if not batch:
            pytest.skip("a standalone run is R = 1; covered by the batch")
        w.R = 3
    elif case == "Q != pool Q":
        w.Q = 2
    wref = _break_prio(w, case)
    if entry == "rollout":
        rc = lib.ia2c_rollout_env_partners_prioritized(C.byref(d), C.byref(p), wref, None)
    else:
        rc = lib.ia2c_train_episode_env_partners_prioritized(C.byref(d), C.byref(r) if batch else None, C.byref(p), wref, None)
    assert rc == INVALID
    assert message in lib.ia2c_last_error().decode(), lib.ia2c_last_error().decode()


@pytest.mark.parametrize("case, status, message", [(c, INVALID, m) for c, m in PRIO_CASES] + [
    ("null episode descriptor", INVALID, "null episode descriptor"),
    ("null ep_return", INVALID, "null ep_return or env_team"),
    ("null env_team", INVALID, "null ep_return or env_team"),
    ("E=0", INVALID, "E=0"),
    ("env_offset", UNSUPPORTED, "one GPU"),
    ("E_total", UNSUPPORTED, "one GPU"),
])
def test_record_partner_returns_refuses_without_touching_a_device(case, status, message):
    lib, d, _, _ = _descs()
    d.ep_return = FAKE
    team, dref = FAKE, C.byref(d)
    w = _prio()
    wref = _break_prio(w, case) if case in dict(PRIO_CASES) else C.byref(w)
    if case == "null episode descriptor":
        dref = None
    elif case == "null ep_return":
        d.ep_return = None
    elif case == "null env_team":
        team = None
    elif case == "E=0":
        d.E = d.E_total = 0
    elif case == "env_offset":
        d.env_offset = 10
    elif case == "E_total":
        d.E_total = 20
    assert lib.ia2c_record_partner_returns(dref, team, wref, None) == status
    assert message in lib.ia2c_last_error().decode(), lib.ia2c_last_error().decode()


@pytest.mark.parametrize("case, power, floor, message", [(c, 2, 0.1, m) for c, m in PRIO_CASES] + [
    ("power", -1, 0.1, "power=-1"), ("power", 17, 0.1, "power=17"), ("floor", 2, -0.5, "floor=-0.5"),
    ("floor", 2, 1.5, "floor=1.5"), ("floor", 2, float("nan"), "floor=nan"), ("floor", 2, float("inf"), "floor=inf")])
def test_prioritize_partners_refuses_without_touching_a_device(case, power, floor, message):
    from ia2c_b200 import _lib
    lib = _lib.load()
    w = _prio()
    wref = _break_prio(w, case) if case in dict(PRIO_CASES) else C.byref(w)
    assert lib.ia2c_prioritize_partners(wref, power, floor, 1, None) == INVALID
    assert message in lib.ia2c_last_error().decode(), lib.ia2c_last_error().decode()


def test_prioritized_without_per_env_is_refused():
    tr = _trainer()
    with pytest.raises(ValueError, match="per_env=True"):
        tr.set_partners(_pool(), prioritized=True)
    assert tr.partners is None and not tr.partners_prioritized


def test_prioritized_mode_is_refused_where_per_env_is():
    from ia2c_b200 import _lib
    tr = _trainer(3, 5, 0)   # fused_rollout=False
    with pytest.raises(_lib.IA2CError, match="per-step rollout"):
        tr.set_partners(_pool(), per_env=True, prioritized=True)
    assert tr.partners is None and not tr.partners_prioritized
    with pytest.raises(_lib.IA2CError, match="one GPU"):
        _trainer(world=2).set_partners(_pool(), per_env=True, prioritized=True)


def test_prioritized_statistics_above_the_cap_are_refused():
    from ia2c_b200 import _lib
    from ia2c_b200.runs import IA2CRuns
    runs = IA2CRuns.__new__(IA2CRuns)
    runs.R, runs.N, runs.device, runs.runs_desc = 17, 3, torch.device("cuda:0"), _lib.RunsDesc()
    pool = _pool()
    pool.Q = 1 << 20
    with pytest.raises(ValueError, match="PARTNER_PRIORITY_MAX_CELLS"):
        runs.set_partners(pool, per_env=True, prioritized=True)
    assert runs.partners is None and not runs.partners_prioritized


@pytest.mark.parametrize("call", ["prioritize_partners", "partner_returns", "partner_weights"])
@pytest.mark.parametrize("mode", ["none", "per_episode", "per_env"])
def test_priority_calls_are_refused_outside_the_mode(call, mode):
    from ia2c_b200 import _lib
    tr = _trainer()
    if mode != "none":
        tr._partners, tr._env_partners = _pool(), mode == "per_env"
    with pytest.raises(_lib.IA2CError, match="prioritized=True"):
        getattr(tr, call)()


@pytest.mark.parametrize("power, floor", [(-1, 0.1), (17, 0.1), (2.5, 0.1), (True, 0.1), (2, -0.1), (2, 1.01), (2, float("nan"))])
def test_prioritize_partners_refuses_bad_arguments(power, floor):
    tr = _trainer()
    tr._priority = {"desc": None}
    with pytest.raises(ValueError):
        tr.prioritize_partners(power=power, floor=floor)


def test_set_partners_none_and_a_new_pool_drop_the_statistics():
    tr = _trainer()
    tr._partners, tr._env_partners, tr._priority = _pool(), True, {"desc": None}
    tr.set_partners(None)
    assert tr._priority is None and not tr.partners_prioritized


def test_checkpoints_carry_the_statistics_and_older_ones_load_uniform():
    calls = []
    tr = _trainer()
    tr.set_partners = lambda pool, per_env=False, **kw: calls.append((per_env, kw.get("prioritized", False)))
    pool = _pool()
    pool.state = lambda: {}
    tr._partners, tr._env_partners = pool, True
    z = lambda *s: torch.zeros(s, dtype=torch.int64)
    tr._priority = dict(count=z(1, 3), sum=z(1, 3), table=z(1, 4))
    sd = tr._partner_state({})
    assert sd["partners_per_env"] is True and set(sd["partner_priority"]) == {"count", "sum", "table"}
    assert sd["partner_priority"]["table"].shape == (1, 4)
    tr._load_partner_state({"partners": None})
    assert calls == [(False, False)]
    bad = {"partners": {"teams": z(3, 1)}, "partners_per_env": True, "partner_priority": dict(count=z(1, 2), sum=z(1, 2), table=z(1, 3))}
    with pytest.raises(ValueError, match="partner_priority"):
        tr._load_partner_state(bad)
    assert calls == [(False, False)]


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not installed")
def test_priority_kernels_wait_before_they_read():
    """partner_returns_kernel and partner_priority_kernel release their successor (PREEXIT) and load nothing before
    griddepcontrol.wait (ACQBULK); tools/pdl_hoist_check.py lists no early load for them."""
    from ia2c_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("library not built")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "pdl_hoist_check.py"), _lib.LIB_PATH], capture_output=True,
                         text=True, check=True).stdout
    for name in ("partner_returns_kernel", "partner_priority_kernel"):
        line = next(ln for ln in out.splitlines() if ln.startswith(name + ":"))
        assert line.endswith(", 0 global loads before it"), line
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    for chunk in sass.split("Function : ")[1:]:
        name, body = chunk.split("\n", 1)
        if "partner_returns_kernel" in name or "partner_priority_kernel" in name:
            ops = [ln for ln in body.split("Fatbin", 1)[0].splitlines() if re.search(r"/\*[0-9a-f]{4}\*/", ln)]
            wait = next(i for i, ln in enumerate(ops) if "ACQBULK" in ln)
            assert any("PREEXIT" in ln for ln in ops[:wait]), name
            assert not [ln for ln in ops[:wait] if re.search(r"\b(LDG|STG|ATOMG|RED)", ln)], name
