"""CPU-side checks of the native A2C trainer's entry point: the ctypes mirror of ia2c_a2c_desc has the C layout, and
ia2c_a2c_train_update refuses what it cannot run before it makes any CUDA call (its pointers here point nowhere)."""
import ctypes as C
import os
import subprocess

import pytest

from tests.conftest import ROOT

HEADER = os.path.join(ROOT, "include", "ia2c_b200.h")
INVALID = -1


def test_a2c_desc_layout_matches_c(tmp_path):
    from ia2c_b200 import _lib
    fields = [f[0] for f in _lib.A2CDesc._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu", sizeof(ia2c_a2c_desc));' % HEADER
    for f in fields:
        prog += 'printf(" %%zu", offsetof(ia2c_a2c_desc, %s));' % f
    prog += 'printf(" %d %d %d", IA2C_A2C_MAX_RUNS, IA2C_A2C_MAX_ENVS, IA2C_A2C_MAX_STEPS);return 0;}\n'
    c = tmp_path / "layout.c"
    c.write_text(prog)
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(c), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.A2CDesc)
    assert out[1:-3] == [getattr(_lib.A2CDesc, f).offset for f in fields]
    assert out[-3:] == [_lib.A2C_MAX_RUNS, _lib.A2C_MAX_ENVS, _lib.A2C_MAX_STEPS]


def _desc(R=4, E=37, T=100):
    from ia2c_b200 import _lib
    lib = _lib.load()
    d = _lib.A2CDesc()
    d.E, d.R, d.T = E, R, T
    fake = 0x1000
    for name, _ in _lib.A2CDesc._fields_:
        if name not in ("E", "R", "T", "update", "beta", "lr_actor", "lr_critic", "lr_actor_run", "lr_critic_run", "beta_run",
                        "inj_actions", "partials_floats"):
            setattr(d, name, fake)
    d.partials_floats = 1 << 40
    return lib, d


@pytest.mark.parametrize("case, message", [
    ("null desc", "null descriptor"),
    ("R=0", "R=0"),
    ("R too large", "R=65536"),
    ("E=0", "E=0"),
    ("R*E too large", "R * E"),
    ("T=0", "T=0"),
    ("T too large", "T=65535"),
    ("null seed", "null seed"),
    ("null params", "null network"),
    ("null env", "null env"),
    ("null trajectory", "null trajectory"),
    ("small workspace", "partials"),
])
def test_train_update_refuses_without_touching_a_device(case, message):
    from ia2c_b200 import _lib
    lib, d = _desc()
    arg = C.byref(d)
    if case == "null desc":
        arg = None
    elif case == "R=0":
        d.R = 0
    elif case == "R too large":
        d.R = _lib.A2C_MAX_RUNS + 1
    elif case == "E=0":
        d.E = 0
    elif case == "R*E too large":
        d.R, d.E = 2, _lib.A2C_MAX_ENVS
    elif case == "T=0":
        d.T = 0
    elif case == "T too large":
        d.T = _lib.A2C_MAX_STEPS + 1
    elif case == "null seed":
        d.seed = None
    elif case == "null params":
        d.critic_m = None
    elif case == "null env":
        d.pending_action = None
    elif case == "null trajectory":
        d.reward = None
    elif case == "small workspace":
        d.partials_floats = int(lib.ia2c_a2c_partials_floats(C.byref(d))) - 1
    assert lib.ia2c_a2c_train_update(arg, None) == INVALID
    assert message in lib.ia2c_last_error().decode()


def test_partials_cover_one_row_per_block_of_32_envs_per_run():
    lib, d = _desc(R=3, E=37)
    assert int(lib.ia2c_a2c_partials_floats(C.byref(d))) == 3 * 2 * 148
    d.R, d.E = 1, 1
    assert int(lib.ia2c_a2c_partials_floats(C.byref(d))) == 148
    d.R = 0
    assert int(lib.ia2c_a2c_partials_floats(C.byref(d))) == 0


def test_python_refusals_before_any_device_work():
    from ia2c_b200.a2c import A2COrgTrainer
    with pytest.raises(ValueError, match="at least one run"):
        A2COrgTrainer(1, seeds=[])
    with pytest.raises(ValueError, match="one value per run"):
        A2COrgTrainer(1, seeds=[1, 2, 3], lr_actor=[1e-4, 2e-4])
    with pytest.raises(ValueError, match="finite"):
        A2COrgTrainer(1, seeds=[1], beta=float("nan"))
    with pytest.raises(ValueError, match="num_envs"):
        A2COrgTrainer(0)
    with pytest.raises(ValueError, match="steps_per_update"):
        A2COrgTrainer(1, steps_per_update=0)
    with pytest.raises(ValueError, match="seeds must lie"):
        A2COrgTrainer(1, seeds=-1)
    with pytest.raises(ValueError, match="one \\(actor, critic\\) pair per run"):
        A2COrgTrainer(1, seeds=[0, 1], init=[(None, None)])
    with pytest.raises(ValueError, match="147 parameters"):
        A2COrgTrainer(1, seeds=[0], init=[([0.0] * 5, [0.0] * 147)])
