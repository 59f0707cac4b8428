"""CPU-side checks of the batched-runs entry point: the ctypes mirror of ia2c_runs_desc has the C layout, and
ia2c_train_episode_runs refuses what it does not support before it makes any CUDA call."""
import ctypes as C
import os
import subprocess

import pytest

from tests.conftest import ROOT

HEADER = os.path.join(ROOT, "include", "ia2c_b200.h")


def test_runs_desc_layout_matches_c(tmp_path):
    from ia2c_b200 import _lib
    fields = [f[0] for f in _lib.RunsDesc._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu", sizeof(ia2c_runs_desc));' % HEADER
    for f in fields:
        prog += 'printf(" %%zu", offsetof(ia2c_runs_desc, %s));' % f
    prog += 'printf(" %d", IA2C_MAX_RUN_NETS);return 0;}\n'
    c = tmp_path / "layout.c"
    c.write_text(prog)
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(c), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.RunsDesc)
    assert out[1:-1] == [getattr(_lib.RunsDesc, f).offset for f in fields]
    assert out[-1] == _lib.MAX_RUN_NETS


def _descs(N=2, M=5, E=10, T=30, runs=4):
    """A descriptor whose buffer pointers are non-NULL but point nowhere: every refusal below must come before the first
    device access."""
    from ia2c_b200 import _lib
    lib = _lib.load()
    d = _lib.EpisodeDesc()
    d.E, d.E_total, d.env_offset, d.N, d.T, d.M, d.max_episode_steps = E, E, 0, N, T, M, T
    d.flags = _lib.FLAG_FUSED_ROLLOUT | _lib.FLAG_FUSED_CRITIC | _lib.FLAG_ACTOR_COLUMNS
    fake = 0x1000
    for name, _ in _lib.EpisodeDesc._fields_[14:38]:
        setattr(d, name, fake)
    d.partials, d.partials_floats = fake, 1 << 40
    r = _lib.RunsDesc()
    r.runs, r.seed = runs, fake
    return lib, d, r


INVALID, UNSUPPORTED = -1, -3


@pytest.mark.parametrize("case, status, message", [
    ("runs=0", INVALID, "runs=0"),
    ("runs*N too large", INVALID, "IA2C_MAX_RUN_NETS"),
    ("null seed", INVALID, "null seed"),
    ("N=9", UNSUPPORTED, "N=9"),
    ("N=3 M=3", UNSUPPORTED, "N=3 M=3"),
    ("env_offset", UNSUPPORTED, "env_offset"),
    ("E_total", UNSUPPORTED, "E_total"),
    ("replay tape", UNSUPPORTED, "replay"),
    ("parity dump", UNSUPPORTED, "dumps"),
    ("skip adam", UNSUPPORTED, "flags"),
    ("small workspace", INVALID, "partials"),
])
def test_train_episode_runs_refuses_without_touching_a_device(case, status, message):
    from ia2c_b200 import _lib
    lib, d, r = _descs()
    if case == "runs=0":
        r.runs = 0
    elif case == "runs*N too large":
        r.runs = _lib.MAX_RUN_NETS // 2 + 1
    elif case == "null seed":
        r.seed = None
    elif case == "N=9":
        d.N = 9
    elif case == "N=3 M=3":
        d.N, d.M = 3, 3
    elif case == "env_offset":
        d.env_offset = 10
    elif case == "E_total":
        d.E_total = 2 * d.E
    elif case == "replay tape":
        d.inj_u_action = 0x1000
    elif case == "parity dump":
        d.belief_dump = 0x1000
    elif case == "skip adam":
        d.flags |= _lib.FLAG_SKIP_ADAM
    elif case == "small workspace":
        d.partials_floats = int(lib.ia2c_runs_partials_floats(C.byref(d), r.runs)) - 1
    assert lib.ia2c_train_episode_runs(C.byref(d), C.byref(r), None) == status
    assert message in lib.ia2c_last_error().decode()


def test_runs_partials_scale_with_the_batch():
    lib, d, _ = _descs(E=37)
    one = int(lib.ia2c_episode_partials_floats(C.byref(d)))
    assert one > 0
    assert int(lib.ia2c_runs_partials_floats(C.byref(d), 1)) == one
    assert int(lib.ia2c_runs_partials_floats(C.byref(d), 64)) == 64 * one
    assert int(lib.ia2c_runs_partials_floats(C.byref(d), 0)) == 0


def test_python_refusals_before_any_device_work():
    from ia2c_b200.runs import IA2CRuns
    with pytest.raises(ValueError, match="fused path"):
        IA2CRuns(10, [1, 2], n_agents=9)
    with pytest.raises(ValueError, match="fused path"):
        IA2CRuns(10, [1, 2], n_agents=3, n_models=3)
    with pytest.raises(ValueError, match="one value per run"):
        IA2CRuns(10, [1, 2, 3], lr_actor=[1e-4, 2e-4])
    with pytest.raises(ValueError, match="at least one run"):
        IA2CRuns(10, [])
    with pytest.raises(ValueError, match="above the limit"):
        IA2CRuns(10, range(40000), n_agents=2)
    with pytest.raises(ValueError, match="finite"):
        IA2CRuns(10, [1], gamma=float("nan"))
