"""CPU-side checks of the batched Org-N entry point (9 <= N <= 256): ia2c_train_episode_runs_many refuses what it does not
support before it makes any CUDA call, its workspace is the one ia2c_runs_partials_floats sizes, and IA2CRunsMany raises
before any device work."""
import ctypes as C

import pytest

from tests.test_runs_abi import _descs

INVALID, UNSUPPORTED = -1, -3


def _many(N=16, M=5, E=10, runs=4):
    from ia2c_b200 import _lib
    lib, d, r = _descs(N=N, M=M, E=E, runs=runs)
    d.flags = _lib.FLAG_ACTOR_COLUMNS
    return lib, d, r


def test_abi_version():
    from ia2c_b200 import _lib
    assert _lib.ABI_VERSION == 6
    assert _lib.load().ia2c_abi_version() == 6


@pytest.mark.parametrize("case, status, message", [
    ("N=8", UNSUPPORTED, "ia2c_train_episode_runs"),
    ("N=2", UNSUPPORTED, "N <= 8"),
    ("N=257", UNSUPPORTED, "N=257"),
    ("env_offset", UNSUPPORTED, "env_offset"),
    ("E_total", UNSUPPORTED, "E_total"),
    ("replay actions", UNSUPPORTED, "replay"),
    ("replay uniforms", UNSUPPORTED, "replay"),
    ("replay beliefs", UNSUPPORTED, "replay"),
    ("belief dump", UNSUPPORTED, "dumps"),
    ("target dump", UNSUPPORTED, "dumps"),
    ("fused flags", UNSUPPORTED, "flags"),
    ("no flags", UNSUPPORTED, "flags"),
    ("skip adam", UNSUPPORTED, "flags"),
    ("runs=0", INVALID, "runs=0"),
    ("runs*N too large", INVALID, "IA2C_MAX_RUN_NETS"),
    ("null seed", INVALID, "null seed"),
    ("M=1", INVALID, "M=1"),
    ("M=7", INVALID, "M=7"),
    ("null params", INVALID, "null network"),
    ("null records", INVALID, "null env/belief"),
    ("null optimiser", INVALID, "null optimiser"),
    ("small workspace", INVALID, "partials"),
])
def test_train_episode_runs_many_refuses_without_touching_a_device(case, status, message):
    from ia2c_b200 import _lib
    lib, d, r = _many()
    if case == "N=8":
        d.N = 8
    elif case == "N=2":
        d.N = 2
    elif case == "N=257":
        d.N = 257
    elif case == "env_offset":
        d.env_offset = 10
    elif case == "E_total":
        d.E_total = 2 * d.E
    elif case == "replay actions":
        d.inj_actions = 0x1000
    elif case == "replay uniforms":
        d.inj_u_action = 0x1000
    elif case == "replay beliefs":
        d.inj_u_belief = 0x1000
    elif case == "belief dump":
        d.belief_dump = 0x1000
    elif case == "target dump":
        d.target_dump = 0x1000
    elif case == "fused flags":
        d.flags = _lib.FLAG_FUSED_ROLLOUT | _lib.FLAG_FUSED_CRITIC | _lib.FLAG_ACTOR_COLUMNS
    elif case == "no flags":
        d.flags = 0
    elif case == "skip adam":
        d.flags |= _lib.FLAG_SKIP_ADAM
    elif case == "runs=0":
        r.runs = 0
    elif case == "runs*N too large":
        r.runs = _lib.MAX_RUN_NETS // d.N + 1
    elif case == "null seed":
        r.seed = None
    elif case == "M=1":
        d.M = 1
    elif case == "M=7":
        d.M = 7
    elif case == "null params":
        d.actor_params = None
    elif case == "null records":
        d.belief_records = None
    elif case == "null optimiser":
        d.actor_m = None
    elif case == "small workspace":
        d.partials_floats = int(lib.ia2c_runs_partials_floats(C.byref(d), r.runs)) - 1
    assert lib.ia2c_train_episode_runs_many(C.byref(d), C.byref(r), None) == status
    assert message in lib.ia2c_last_error().decode()


def test_n8_refusal_points_to_the_fused_entry_point():
    lib, d, r = _many()
    d.N = 8
    assert lib.ia2c_train_episode_runs_many(C.byref(d), C.byref(r), None) == UNSUPPORTED
    assert "ia2c_train_episode_runs" in lib.ia2c_last_error().decode()


@pytest.mark.parametrize("N, E", [(9, 37), (16, 10), (64, 1024), (256, 10)])
def test_workspace_is_runs_partials_floats(N, E):
    """The batch's workspace is R x the standalone size (which covers the grad_blocks(E) partial rows per net that the six
    launches write), and one float less is refused as too small.  A workspace of exactly that size is what IA2CRunsMany
    allocates, so the GPU tests exercise its acceptance."""
    lib, d, r = _many(N=N, E=E)
    one = int(lib.ia2c_episode_partials_floats(C.byref(d)))
    assert one > 0
    assert int(lib.ia2c_runs_partials_floats(C.byref(d), 8)) == 8 * one
    d.partials_floats = int(lib.ia2c_runs_partials_floats(C.byref(d), r.runs)) - 1
    assert lib.ia2c_train_episode_runs_many(C.byref(d), C.byref(r), None) == INVALID
    assert "partials workspace too small" in lib.ia2c_last_error().decode()


@pytest.mark.parametrize("N", [2, 8, 257])
def test_python_refuses_agent_counts_outside_9_to_256(N):
    from ia2c_b200.runs import IA2CRunsMany
    with pytest.raises(ValueError, match="IA2CRuns" if N <= 8 else "256"):
        IA2CRunsMany(10, [1, 2], n_agents=N)


def test_python_refusals_before_any_device_work():
    from ia2c_b200 import _lib
    from ia2c_b200.runs import IA2CRunsMany
    with pytest.raises(ValueError, match="one value per run"):
        IA2CRunsMany(10, [1, 2, 3], n_agents=16, lr_actor=[1e-4, 2e-4])
    with pytest.raises(ValueError, match="one value per run"):
        IA2CRunsMany(10, [1, 2], n_agents=16, gamma=[0.9, 0.9, 0.9])
    with pytest.raises(ValueError, match="above the limit"):
        IA2CRunsMany(10, range(_lib.MAX_RUN_NETS // 256 + 1), n_agents=256)
    with pytest.raises(ValueError, match="n_models"):
        IA2CRunsMany(10, [1, 2], n_agents=16, n_models=7)
    with pytest.raises(ValueError, match="at least one run"):
        IA2CRunsMany(10, [], n_agents=16)


def test_exported_from_the_package():
    import ia2c_b200
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    assert ia2c_b200.IA2CRunsMany is IA2CRunsMany and issubclass(IA2CRunsMany, IA2CRuns)
