"""CPU-side checks of the history entry point: the ctypes mirror of ia2c_history_desc has the C layout, the symbol is exported,
and ia2c_record_episode / train_episodes refuse what they do not support before any device work."""
import ctypes as C
import os
import subprocess

import pytest

from tests.conftest import ROOT

HEADER = os.path.join(ROOT, "include", "ia2c_b200.h")
INVALID, UNSUPPORTED = -1, -3


def test_history_desc_layout_matches_c(tmp_path):
    from ia2c_b200 import _lib
    fields = [f[0] for f in _lib.HistoryDesc._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu", sizeof(ia2c_history_desc));' % HEADER
    for f in fields:
        prog += 'printf(" %%zu", offsetof(ia2c_history_desc, %s));' % f
    prog += 'printf(" %d", IA2C_ABI_VERSION);return 0;}\n'
    c = tmp_path / "layout.c"
    c.write_text(prog)
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(c), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.HistoryDesc)
    assert out[1:-1] == [getattr(_lib.HistoryDesc, f).offset for f in fields]
    assert out[-1] == _lib.ABI_VERSION == 6


def test_record_symbol_is_exported():
    from ia2c_b200 import _lib
    lib = _lib.load()
    assert hasattr(lib, "ia2c_record_episode") and "ia2c_record_episode" in _lib.SIGNATURES


def _descs(E=37, N=5, T=30, cap=4):
    """Descriptors whose pointers are non-NULL but point nowhere: every refusal below must come before the first device
    access."""
    from ia2c_b200 import _lib
    lib = _lib.load()
    d = _lib.EpisodeDesc()
    d.E, d.E_total, d.env_offset, d.N, d.T, d.M = E, E, 0, N, T, 5
    fake = 0x1000
    d.act = d.partner_true = d.partner_pred = d.ep_return = d.loss_out = fake
    h = _lib.HistoryDesc()
    h.capacity = cap
    h.return_sum = h.loss = h.action_counts = h.partner_hits = fake
    return lib, d, h


@pytest.mark.parametrize("case, status, message", [
    ("null episode descriptor", INVALID, "null episode or history descriptor"),
    ("null history descriptor", INVALID, "null episode or history descriptor"),
    ("null act", INVALID, "null act"),
    ("null partner_true", INVALID, "null act"),
    ("null partner_pred", INVALID, "null act"),
    ("null ep_return", INVALID, "null act"),
    ("null loss_out", INVALID, "null act"),
    ("null return_sum", INVALID, "null return_sum"),
    ("null loss", INVALID, "null return_sum"),
    ("null action_counts", INVALID, "null return_sum"),
    ("null partner_hits", INVALID, "null return_sum"),
    ("runs=0", INVALID, "runs=0"),
    ("runs*N too large", INVALID, "IA2C_MAX_RUN_NETS"),
    ("capacity=1", INVALID, "capacity=1"),
    ("slot=-1", INVALID, "slot=-1"),
    ("slot=capacity", INVALID, "slot=4"),
    ("env_offset", UNSUPPORTED, "one GPU"),
    ("E_total", UNSUPPORTED, "one GPU"),
    ("T*E too large", INVALID, "2^32"),
])
def test_record_refuses_without_touching_a_device(case, status, message):
    lib, d, h = _descs()
    runs, slot = 3, 1
    dp, hp = C.byref(d), C.byref(h)
    if case == "null episode descriptor":
        dp = None
    elif case == "null history descriptor":
        hp = None
    elif case.startswith("null "):
        field = case[5:]
        setattr(d if field in ("act", "partner_true", "partner_pred", "ep_return", "loss_out") else h, field, None)
    elif case == "runs=0":
        runs = 0
    elif case == "runs*N too large":
        runs = 65535 // 5 + 1
    elif case == "capacity=1":
        h.capacity, slot = 1, 0
    elif case == "slot=-1":
        slot = -1
    elif case == "slot=capacity":
        slot = 4
    elif case == "env_offset":
        d.env_offset = 37
    elif case == "E_total":
        d.E_total = 74
    elif case == "T*E too large":
        d.E, d.E_total, d.T = 1 << 27, 1 << 27, 32
    assert lib.ia2c_record_episode(dp, runs, hp, slot, None) == status
    assert message in lib.ia2c_last_error().decode(), lib.ia2c_last_error().decode()


def test_trainer_train_episodes_refuses_multi_gpu_before_device_work():
    """IA2CTrainer.train_episodes at world > 1 raises before touching the ring or the device (the object is built without
    __init__: there is no device here)."""
    from ia2c_b200 import _lib
    from ia2c_b200.trainer import IA2CTrainer
    tr = IA2CTrainer.__new__(IA2CTrainer)
    tr.world = 2
    with pytest.raises(_lib.IA2CError, match="one GPU"):
        tr.train_episodes(3)
    assert tr._history is None
    with pytest.raises(ValueError, match="n=-1"):
        tr.train_episodes(-1)


def test_history_capacity_is_a_class_attribute():
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    from ia2c_b200.trainer import IA2CTrainer
    assert IA2CTrainer.HISTORY_CAPACITY == IA2CRuns.HISTORY_CAPACITY == IA2CRunsMany.HISTORY_CAPACITY == 64


def test_empty_history_arrays_have_the_documented_shapes():
    from ia2c_b200.history import history_arrays
    out = history_arrays([], 3, 5, 10, 30)
    assert out["episode"].shape == (0,) and out["return_sum"].shape == (0, 3) and out["mean_return"].shape == (0, 3)
    assert out["critic_loss"].shape == out["actor_loss"].shape == out["partner_accuracy"].shape == (0, 3, 5)
    assert out["action_counts"].shape == out["action_freq"].shape == (0, 3, 5, 3)
