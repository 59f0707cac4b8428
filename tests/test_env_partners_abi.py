"""CPU-side checks of frozen partners per env: the ctypes mirror of ia2c_env_partner_desc has the C layout, the symbols are
exported, every refusal of ia2c_rollout_env_partners / ia2c_train_episode_env_partners / ia2c_partner_policy and of
set_partners(per_env=True) happens before any device work, the stream-7 draw of the oracle is the documented Philox block,
uniform over teams, and the PARTNERS instantiations of the rollout kernels read nothing before their griddepcontrol.wait."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch
from scipy import stats

from oracle import env_partners as EP
from oracle import partners as PT
from oracle import philox
from tests.conftest import ROOT

HEADER = os.path.join(ROOT, "include", "ia2c_b200.h")
INVALID, UNSUPPORTED = -1, -3
ENTRIES = ("ia2c_partner_policy", "ia2c_rollout_env_partners", "ia2c_train_episode_env_partners")


def test_env_partner_desc_layout_matches_c(tmp_path):
    from ia2c_b200 import _lib
    fields = [f[0] for f in _lib.EnvPartnerDesc._fields_]
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu", sizeof(ia2c_env_partner_desc));'
            % HEADER)
    for f in fields:
        prog += 'printf(" %%zu", offsetof(ia2c_env_partner_desc, %s));' % f
    prog += 'printf(" %d", IA2C_ABI_VERSION);return 0;}\n'
    c = tmp_path / "layout.c"
    c.write_text(prog)
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(c), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.EnvPartnerDesc)
    assert out[1:-1] == [getattr(_lib.EnvPartnerDesc, f).offset for f in fields]
    assert fields == ["rows", "P", "policy", "seats", "S", "teams", "Q", "log_env_team"]
    assert out[-1] == _lib.ABI_VERSION == 6


def test_env_partner_symbols_are_exported_and_declared():
    from ia2c_b200 import _lib
    lib = _lib.load()
    header = open(HEADER).read()
    for name in ENTRIES:
        assert hasattr(lib, name) and name in _lib.SIGNATURES
        assert re.search(r"\bint %s\(" % name, header), name


def _descs(R=4, N=3, M=5):
    """Descriptors whose pointers are non-NULL but point nowhere: every refusal below must come before the first device
    access."""
    from ia2c_b200 import _lib
    lib = _lib.load()
    fake = 0x1000
    d = _lib.EpisodeDesc()
    d.E, d.E_total, d.env_offset, d.N, d.T, d.M = 10, 10, 0, N, 30, M
    d.flags = _lib.FLAG_FUSED_ROLLOUT | _lib.FLAG_FUSED_CRITIC
    r = _lib.RunsDesc()
    r.runs, r.seed = R, fake
    p = _lib.EnvPartnerDesc()
    p.rows, p.P, p.policy, p.seats, p.S, p.teams, p.Q, p.log_env_team = fake, 5, fake, fake, 1, fake, 3, fake
    return lib, d, r, p


CASES = [
    ("null episode descriptor", INVALID, "null episode or partner descriptor"),
    ("null partner descriptor", INVALID, "null episode or partner descriptor"),
    ("null rows", INVALID, "null rows"),
    ("null seats", INVALID, "null rows"),
    ("null teams", INVALID, "null rows"),
    ("null log_env_team", INVALID, "null rows"),
    ("null seed", INVALID, "null seed"),
    ("runs=0", INVALID, "runs=0"),
    ("N=1", INVALID, "N=1"),
    ("runs*N too large", INVALID, "IA2C_MAX_RUN_NETS"),
    ("S=0", INVALID, "S=0"),
    ("S=N", INVALID, "S=3"),
    ("P=0", INVALID, "P=0"),
    ("Q=0", INVALID, "Q=0"),
    ("Q too large", INVALID, "Q=1048577"),
    ("null policy at N > 8", INVALID, "null policy table"),
    ("env_offset", UNSUPPORTED, "one GPU"),
    ("E_total", UNSUPPORTED, "one GPU"),
    ("injected actions", UNSUPPORTED, "inj_actions"),
    ("N > 256", UNSUPPORTED, "N above 256"),
    ("M without a fused instantiation", UNSUPPORTED, "no fused rollout instantiation"),
    ("fused_rollout off", UNSUPPORTED, "without IA2C_FLAG_FUSED_ROLLOUT"),
    ("ROLLOUT_PER_STEP", UNSUPPORTED, "per-step rollout"),
    ("BELIEF_PER_STEP", UNSUPPORTED, "per-step rollout"),
    ("no whole-episode belief kernel", UNSUPPORTED, "per-step rollout"),
]
STANDALONE_ONLY = ("fused_rollout off", "ROLLOUT_PER_STEP", "BELIEF_PER_STEP", "no whole-episode belief kernel")


@pytest.mark.parametrize("case, status, message", CASES)
@pytest.mark.parametrize("entry", ["train_batch", "train_standalone", "rollout"])
def test_env_partner_entries_refuse_without_touching_a_device(case, status, message, entry):
    from ia2c_b200 import _lib
    lib, d, r, p = _descs()
    batch = entry == "train_batch"
    if not batch and case in ("null seed", "runs=0", "runs*N too large"):
        pytest.skip("a standalone run has no runs descriptor")
    if batch and case in STANDALONE_ONLY:
        pytest.skip("a batch always runs the fused or the whole-episode rollout")
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
        d.inj_actions = 0x1000
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
        rc = lib.ia2c_rollout_env_partners(dref, pref, None)
    else:
        rc = lib.ia2c_train_episode_env_partners(dref, C.byref(r) if batch else None, pref, None)
    assert rc == status
    assert message in lib.ia2c_last_error().decode(), lib.ia2c_last_error().decode()


@pytest.mark.parametrize("rows, P, policy, message", [(None, 4, 0x1000, "null rows or policy"), (0x1000, 4, None, "null rows or policy"),
                                                      (0x1000, 0, 0x1000, "P=0")])
def test_partner_policy_refuses_without_touching_a_device(rows, P, policy, message):
    from ia2c_b200 import _lib
    lib = _lib.load()
    assert lib.ia2c_partner_policy(rows, P, policy, None) == INVALID
    assert message in lib.ia2c_last_error().decode()


def _pool(N=3, device="cuda:0"):
    """A PartnerPool built without __init__ (there is no device here)."""
    from ia2c_b200.partners import PartnerPool
    pool = PartnerPool.__new__(PartnerPool)
    pool.N, pool.device = N, torch.device(device)
    return pool


def _trainer(N=3, M=5, flags=None, world=1):
    from ia2c_b200 import _lib
    from ia2c_b200.trainer import IA2CTrainer
    obj = IA2CTrainer.__new__(IA2CTrainer)
    obj.N, obj.M, obj.device, obj.world, obj.lib = N, M, torch.device("cuda:0"), world, _lib.load()
    obj.desc = _lib.EpisodeDesc()
    obj.desc.flags = (_lib.FLAG_FUSED_ROLLOUT | _lib.FLAG_FUSED_CRITIC) if flags is None else flags
    return obj


@pytest.mark.parametrize("N, M, flags, message", [
    (3, 5, 0, "per-step rollout"),                                   # fused_rollout=False
    (300, 5, 16, "above 256"),
    (16, 5, 16 | 64, "per-step rollout"),                            # rollout_kernel="step"
    (16, 5, 16 | 32, "per-step rollout"),                            # belief_kernel="step"
    (16, 7, 16, "per-step rollout"),                                 # no whole-episode belief kernel
])
def test_set_partners_per_env_refuses_paths_without_per_env_kernels(N, M, flags, message):
    from ia2c_b200 import _lib
    tr = _trainer(N, M, flags)
    with pytest.raises(_lib.IA2CError, match=message):
        tr.set_partners(_pool(N), per_env=True)
    assert tr.partners is None and not tr.partners_per_env


def test_set_partners_per_env_refuses_more_than_one_gpu_and_mismatched_pools():
    from ia2c_b200 import _lib
    with pytest.raises(_lib.IA2CError, match="one GPU"):
        _trainer(world=2).set_partners(_pool(), per_env=True)
    with pytest.raises(ValueError, match="the pool is for n_agents=4"):
        _trainer().set_partners(_pool(N=4), per_env=True)


def test_per_env_mode_refuses_the_host_tape_calls_the_timed_episode_and_injected_actions():
    from ia2c_b200 import _lib
    tr = _trainer()
    tr._partners, tr._env_partners = _pool(), True
    with pytest.raises(_lib.IA2CError, match="train_episode_host does not seat partners"):
        tr.train_episode_host(None, None)
    with pytest.raises(_lib.IA2CError, match="train_episodes_host does not seat partners"):
        tr.train_episodes_host([])
    with pytest.raises(_lib.IA2CError, match="train_episode_timed does not play partners per env"):
        tr.train_episode_timed()
    tr.inj_actions = torch.zeros(1)
    with pytest.raises(_lib.IA2CError, match="injected actions"):
        tr._play_env_partners(lambda p: 0, "ia2c_train_episode_env_partners")


def test_set_partners_none_leaves_per_env_mode():
    tr = _trainer()
    tr._partners, tr._env_partners = _pool(), True
    tr.set_partners(None)
    assert tr.partners is None and not tr.partners_per_env


def test_empty_env_partner_history_has_the_documented_shapes():
    from ia2c_b200 import _lib
    from ia2c_b200.runs import IA2CRuns
    runs = IA2CRuns.__new__(IA2CRuns)
    runs.R, runs.E, runs.runs_desc = 5, 7, _lib.RunsDesc()
    out = runs.env_partner_history()
    assert out["episode"].shape == (0,) and out["env_team"].shape == (0, 5, 7) and out["env_team"].dtype == np.int32
    tr = _trainer()
    tr.E = 9
    assert tr.env_partner_history()["env_team"].shape == (0, 9)


def test_checkpoints_carry_the_mode_and_older_ones_load_per_episode():
    calls = []
    tr = _trainer()
    tr.set_partners = lambda pool, per_env=False: calls.append(per_env)
    assert tr._partner_state({}) == {}
    tr._load_partner_state({})
    tr._partners, tr._env_partners = _pool(), True
    tr._partners.state = lambda: {}
    assert tr._partner_state({})["partners_per_env"] is True
    assert calls == [False]


def test_env_teams_are_the_documented_stream_7_block():
    seed, episode, E, Q = 0x1234_5678_9ABC_DEF0, 7, 1000, 37
    teams = EP.env_teams(seed, episode, E, Q)
    for e in (0, 1, 999):
        x = philox.philox4x32(np.uint32(e), np.uint32(0), np.uint32(7 << 16), np.uint32(episode), seed & 0xFFFFFFFF, seed >> 32)[0]
        assert teams[e] == (int(x) * Q) >> 32
    words = np.stack(philox.draw(seed, 7, episode, 0, np.arange(E, dtype=np.uint64)))
    assert len({tuple(w) for w in words.T}) == E                       # distinct counters per env: distinct blocks
    assert not np.array_equal(EP.env_teams(seed, episode + 1, E, Q), teams)
    assert PT.team(seed, episode, Q) != teams[0] or PT.words(seed, episode) != tuple(int(w) for w in words[:, 0])   # stream 6 is another stream
    assert np.array_equal(EP.env_teams(seed, episode, E, 1), np.zeros(E))


def test_env_teams_are_uniform():
    Q, E = 16, 64000
    teams = np.concatenate([EP.env_teams(seed, 3, E // 4, Q) for seed in (1, 2, 3, 4)])
    counts = np.bincount(teams, minlength=Q)
    assert teams.min() >= 0 and teams.max() < Q
    assert stats.chisquare(counts).pvalue > 1e-4


def test_env_actors_play_the_team_rows_with_the_guard():
    rng = np.random.RandomState(0)
    N, E, P = 4, 300, 6
    actor = rng.normal(size=(N, 105)).astype(np.float32)
    rows = rng.normal(size=(P, 105)).astype(np.float32)
    teams = np.array([[0, 1], [2, 3], [4, 5], [1, 0]], dtype=np.int32)
    seats = np.array([3, 1], dtype=np.int32)
    actors, log = EP.env_actors(actor, (rows, teams, seats), 9, 2, E)
    assert np.array_equal(log, EP.env_teams(9, 2, E, 4))
    for e in range(E):
        want = actor.copy()
        want[seats] = rows[teams[log[e]]]
        assert np.array_equal(actors[e], want)
    bad = teams.copy()
    bad[2, 1] = P
    actors, log = EP.env_actors(actor, (rows, bad, seats), 9, 2, E)
    hit = EP.env_teams(9, 2, E, 4) == 2
    assert hit.any() and (log[hit] == -1).all() and (log[~hit] >= 0).all()
    assert np.array_equal(actors[hit], np.repeat(actor[None], hit.sum(), 0))
    _, log = EP.env_actors(actor, (rows, teams, np.array([3, 4], dtype=np.int32)), 9, 2, E)
    assert (log == -1).all()
    actors, _ = EP.env_actors(actor, (rows, teams, np.array([1, 1], dtype=np.int32)), 9, 2, E)   # a repeated seat: lowest j wins
    assert all(np.array_equal(actors[e, 1], rows[teams[EP.env_teams(9, 2, E, 4)[e], 0]]) for e in range(E))


def test_env_probs_of_own_rows_are_the_rollouts_probs_and_follow_each_envs_rows():
    from oracle import loops as L
    from ia2c_b200.trainer import reference_init
    N, M, E, T = 3, 5, 40, 6
    actor, critic, fa = reference_init(N, M, seed=2)
    rng = np.random.RandomState(1)
    u_act, u_bel = rng.rand(T + 1, E, N).astype(np.float32), rng.rand(T + 1, E, N, N - 1)
    st = L.IA2CState(actor=actor.astype(np.float64), critic=critic.astype(np.float64), filter_action=fa, T=T, max_episode_steps=T)
    traj = L.ia2c_rollout(st, E, u_act=u_act, u_belief=u_bel)
    own = np.repeat(actor[None], E, 0)
    assert np.array_equal(EP.env_probs(own, traj["obs"]), traj["probs"])
    other = own.copy()
    other[::2, 1] = rng.normal(size=105).astype(np.float32)   # every other env: another row in seat 1
    probs = EP.env_probs(other, traj["obs"])
    from oracle import nets as NN
    want = NN.forward(other[0, 1].astype(np.float64), traj["obs"][:, 0], 6, 3, softmax=True)
    assert np.array_equal(probs[:, 0, 1], want) and np.array_equal(probs[:, 1], traj["probs"][:, 1])


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not installed")
def test_partner_instantiations_wait_before_they_read():
    """The PARTNERS instantiations read the pool, seats, teams and table after griddepcontrol.wait (SASS ACQBULK): before it
    they load exactly what their unpartnered twins load there (the fused kernel's filter tables), never through the read-only
    path (tests/test_pdl_hoist.py's rule), and the table kernel loads nothing before it and releases its successor (PREEXIT)
    first."""
    from ia2c_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("library not built")
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    bodies = {}
    for chunk in sass.split("Function : ")[1:]:
        name, body = chunk.split("\n", 1)
        bodies[name.strip()] = [ln for ln in body.split("Fatbin", 1)[0].splitlines() if re.search(r"/\*[0-9a-f]{4}\*/", ln)]
    partners = re.compile(r"(rollout_fused_kernel|rollout_many_kernel)I(L[ib]\d+E)*Lb1EEE")   # last template argument PARTNERS = true
    new = {n: b for n, b in bodies.items() if "partner_policy_kernel" in n or partners.search(n)}
    assert len(new) == 1 + 24 + 2, sorted(new)
    def early_loads(ops):
        wait = next(i for i, ln in enumerate(ops) if "ACQBULK" in ln)
        return [ln.split("/*")[2].split(";")[0].strip() for ln in ops[:wait] if re.search(r"\bLDG", ln)]

    for name, ops in new.items():
        early = early_loads(ops)
        assert not [ln for ln in early if "CONSTANT" in ln], name
        twin = None if "partner_policy_kernel" in name else re.sub(r"Lb1EEE", "Lb0EEE", name, count=1)
        assert len(early) == (len(early_loads(bodies[twin])) if twin else 0), name
    ops = new[next(n for n in new if "partner_policy_kernel" in n)]
    assert any("PREEXIT" in ln for ln in ops[:next(i for i, ln in enumerate(ops) if "ACQBULK" in ln)])
