"""CPU-side checks of frozen-partner seating: the ctypes mirror of ia2c_partner_desc has the C layout, the symbol is exported,
the kernel waits before its first load and store, and every refusal of ia2c_seat_partners, PartnerPool and set_partners
happens before any device work."""
import ctypes as C
import os
import re
import shutil
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from tests.conftest import ROOT

HEADER = os.path.join(ROOT, "include", "ia2c_b200.h")
INVALID, UNSUPPORTED = -1, -3


def test_partner_desc_layout_matches_c(tmp_path):
    from ia2c_b200 import _lib
    fields = [f[0] for f in _lib.PartnerDesc._fields_]
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu", sizeof(ia2c_partner_desc));'
            % HEADER)
    for f in fields:
        prog += 'printf(" %%zu", offsetof(ia2c_partner_desc, %s));' % f
    prog += 'printf(" %d %d", IA2C_PARTNER_MAX_TEAMS, IA2C_ABI_VERSION);return 0;}\n'
    c = tmp_path / "layout.c"
    c.write_text(prog)
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(c), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.PartnerDesc)
    assert out[1:-2] == [getattr(_lib.PartnerDesc, f).offset for f in fields]
    assert out[-2] == _lib.PARTNER_MAX_TEAMS
    assert out[-1] == _lib.ABI_VERSION == 6


def test_seat_partners_is_exported():
    from ia2c_b200 import _lib
    lib = _lib.load()
    assert hasattr(lib, "ia2c_seat_partners") and "ia2c_seat_partners" in _lib.SIGNATURES


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not installed")
def test_seat_kernel_waits_before_its_first_load_and_store():
    """The kernel overwrites rows the previous episode's Adam step writes: no load or store may precede griddepcontrol.wait
    (SASS ACQBULK), and the early release (PREEXIT) comes first."""
    from ia2c_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("library not built")
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    body = [b for b in sass.split("Function : ")[1:] if "partner_seat_kernel" in b.split("\n", 1)[0]]
    assert len(body) == 1
    ops = [ln for ln in body[0].split("Fatbin", 1)[0].splitlines() if re.search(r"/\*[0-9a-f]{4}\*/", ln)]
    wait = next(i for i, ln in enumerate(ops) if "ACQBULK" in ln)
    assert any("PREEXIT" in ln for ln in ops[:wait])
    assert not [ln for ln in ops[:wait] if re.search(r"\b(LDG|STG|LD|ST|ATOM|RED)\b", ln)], ops[:wait]


def _descs(R=4, N=3):
    """Descriptors whose pointers are non-NULL but point nowhere: every refusal below must come before the first device
    access."""
    from ia2c_b200 import _lib
    lib = _lib.load()
    fake = 0x1000
    d = _lib.EpisodeDesc()
    d.E, d.E_total, d.env_offset, d.N, d.T, d.M = 10, 10, 0, N, 30, 5
    d.actor_params = fake
    r = _lib.RunsDesc()
    r.runs, r.seed = R, fake
    p = _lib.PartnerDesc()
    p.rows, p.P, p.seats, p.S, p.teams, p.Q, p.episode, p.log_team = fake, 5, fake, 1, fake, 3, 0, fake
    return lib, d, r, p


@pytest.mark.parametrize("case, status, message", [
    ("null episode descriptor", INVALID, "null episode or partner descriptor"),
    ("null partner descriptor", INVALID, "null episode or partner descriptor"),
    ("null actor_params", INVALID, "null actor_params"),
    ("null rows", INVALID, "null rows"),
    ("null seats", INVALID, "null rows"),
    ("null teams", INVALID, "null rows"),
    ("null log_team", INVALID, "null rows"),
    ("null seed", INVALID, "null seed"),
    ("runs=0", INVALID, "runs=0"),
    ("N=1", INVALID, "N=1"),
    ("runs*N too large", INVALID, "IA2C_MAX_RUN_NETS"),
    ("S=0", INVALID, "S=0"),
    ("S=N", INVALID, "S=3"),
    ("P=0", INVALID, "P=0"),
    ("Q=0", INVALID, "Q=0"),
    ("Q too large", INVALID, "Q=1048577"),
    ("env_offset", UNSUPPORTED, "one GPU"),
    ("E_total", UNSUPPORTED, "one GPU"),
])
@pytest.mark.parametrize("batch", [True, False])
def test_seat_partners_refuses_without_touching_a_device(case, status, message, batch):
    lib, d, r, p = _descs()
    if not batch and case in ("null seed", "runs=0", "runs*N too large"):
        pytest.skip("a standalone run has no runs descriptor")
    refs = [C.byref(d), C.byref(r) if batch else None, C.byref(p)]
    if case == "null episode descriptor":
        refs[0] = None
    elif case == "null partner descriptor":
        refs[2] = None
    elif case == "null actor_params":
        d.actor_params = None
    elif case == "null seed":
        r.seed = None
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
    assert lib.ia2c_seat_partners(*refs, None) == status
    assert message in lib.ia2c_last_error().decode(), lib.ia2c_last_error().decode()


ROWS = np.zeros((4, 105), dtype=np.float32)


@pytest.mark.parametrize("kw, message", [
    (dict(rows=ROWS.astype(np.float64)), "rows must be float32"),
    (dict(rows=ROWS[:, :100]), "rows must have shape"),
    (dict(rows=ROWS[:0]), "rows must have shape"),
    (dict(rows=ROWS.tolist()), "rows must be float32"),
    (dict(n_agents=1), "n_agents=1"),
    (dict(seats=[1, 1], teams=[[0, 1]]), "repeat a seat"),
    (dict(seats=[3]), r"outside \[0, 3\)"),
    (dict(seats=[-1]), "outside"),
    (dict(seats=np.zeros(0, dtype=np.int32), teams=np.zeros((1, 0), dtype=np.int32)), "seats must be a list of 1 .. n_agents - 1"),
    (dict(seats=[0, 1, 2], teams=[[0, 1, 2]]), "seats must be a list of 1 .. n_agents - 1"),
    (dict(seats=[1.0]), "seats must be an integer array"),
    (dict(teams=[[4]]), r"teams\[0, 0\] = 4 outside the pool's rows \[0, 4\)"),
    (dict(teams=[[0], [-1]]), r"teams\[1, 0\] = -1"),
    (dict(teams=[[0, 1]]), r"teams must have shape \[Q, 1\]"),
    (dict(teams=np.zeros((0, 1), dtype=np.int32)), "teams must have shape"),
    (dict(teams=[[0.0]]), "teams must be an integer array"),
])
def test_pool_refuses_before_device_work(kw, message):
    from ia2c_b200.partners import PartnerPool
    args = dict(rows=ROWS, teams=[[0], [3]], seats=[2], n_agents=3)
    args.update(kw)
    with pytest.raises(ValueError, match=message):
        PartnerPool(**args)


def _pool(N=3, device="cuda:0"):
    """A PartnerPool built without __init__ (there is no device here)."""
    from ia2c_b200.partners import PartnerPool
    pool = PartnerPool.__new__(PartnerPool)
    pool.N, pool.device = N, torch.device(device)
    return pool


def _trainer(cls_name, N=3, world=1, device="cuda:0"):
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    from ia2c_b200.trainer import IA2CTrainer
    cls = dict(IA2CTrainer=IA2CTrainer, IA2CRuns=IA2CRuns, IA2CRunsMany=IA2CRunsMany)[cls_name]
    obj = cls.__new__(cls)
    obj.N, obj.device, obj.world = N, torch.device(device), world
    return obj


@pytest.mark.parametrize("cls_name", ["IA2CTrainer", "IA2CRuns", "IA2CRunsMany"])
@pytest.mark.parametrize("pool_kw, message", [
    (dict(N=4), "the pool is for n_agents=4, this trainer has 3"),
    (dict(device="cuda:1"), "the pool lives on cuda:1, this trainer on cuda:0"),
])
def test_set_partners_refuses_a_mismatched_pool(cls_name, pool_kw, message):
    obj = _trainer(cls_name)
    with pytest.raises(ValueError, match=message):
        obj.set_partners(_pool(**pool_kw))
    assert obj.partners is None


def test_set_partners_refuses_other_objects_and_accepts_none():
    obj = _trainer("IA2CRuns")
    with pytest.raises(ValueError, match="expected a PartnerPool or None"):
        obj.set_partners(SimpleNamespace(N=3, device=torch.device("cuda:0")))
    obj.set_partners(None)
    assert obj.partners is None


def test_set_partners_refuses_more_than_one_gpu():
    from ia2c_b200 import _lib
    obj = _trainer("IA2CTrainer", world=2)
    with pytest.raises(_lib.IA2CError, match="one GPU"):
        obj.set_partners(_pool())


@pytest.mark.parametrize("call", ["train_episode_host", "train_episodes_host"])
def test_host_tape_calls_refuse_while_a_pool_is_set(call):
    from ia2c_b200 import _lib
    obj = _trainer("IA2CTrainer")
    obj._partners = _pool()
    with pytest.raises(_lib.IA2CError, match=f"{call} does not seat partners"):
        getattr(obj, call)(*((None, None) if call == "train_episode_host" else ([],)))


@pytest.mark.parametrize("split, message", [(0, "split=0 outside 1..2"), (3, "split=3 outside 1..2")])
def test_from_sources_refuses_a_split_without_both_kinds_of_seat(split, message):
    from ia2c_b200.partners import PartnerPool
    with pytest.raises(ValueError, match=message):
        PartnerPool.from_sources(_trainer("IA2CRuns"), split=split)


def test_from_sources_refuses_mixed_sources():
    from ia2c_b200.partners import PartnerPool
    with pytest.raises(ValueError, match="must share"):
        PartnerPool.from_sources([_trainer("IA2CRuns"), _trainer("IA2CRuns", N=4)])
    with pytest.raises(ValueError, match="must share"):
        PartnerPool.from_sources([_trainer("IA2CTrainer"), _trainer("IA2CRuns", device="cuda:1")])
    with pytest.raises(ValueError, match="a source must be"):
        PartnerPool.from_sources([object()])
    with pytest.raises(ValueError, match="no sources"):
        PartnerPool.from_sources([])


def test_empty_partner_history_has_the_documented_shapes():
    from ia2c_b200 import _lib
    runs = _trainer("IA2CRuns")
    runs.R, runs.runs_desc = 5, _lib.RunsDesc()
    out = runs.partner_history()
    assert out["episode"].shape == (0,) and out["team"].shape == (0, 5) and out["team"].dtype == np.int32
    tr = _trainer("IA2CTrainer")
    assert tr.partner_history()["team"].shape == (0,)


def test_partner_log_capacity_is_a_class_attribute():
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    from ia2c_b200.trainer import IA2CTrainer
    assert IA2CTrainer.PARTNER_LOG_CAPACITY == IA2CRuns.PARTNER_LOG_CAPACITY == IA2CRunsMany.PARTNER_LOG_CAPACITY == 64
