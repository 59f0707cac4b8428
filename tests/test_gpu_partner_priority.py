"""Prioritized partners per env on the GPU (set_partners(pool, per_env=True, prioritized=True)): before any prioritize_partners
the mode is the uniform per-env mode byte for byte; with teams that all seat the same rows the weights change nothing but
the env-team log; the recorded statistics, the tables and the weighted draws equal the oracle (oracle/partner_priority.py)
exactly; run r of a batch equals a standalone trainer; checkpoints resume exactly; an episode makes one launch more than a
uniform one and prioritize_partners one, with no synchronisation; a deliberately poor team gets the largest weight and is
drawn as often as its weight says."""
import numpy as np
import pytest
import torch
from scipy import stats

from ia2c_b200 import _lib
from oracle import partner_priority as PP
from tests.test_gpu_env_partners import standalone_per_env
from tests.test_gpu_partners import HYPER, STATE, batch, buffers, make_pool, trainer
from tests.test_gpu_runs import BUFFERS, assert_run_equals, h

pytestmark = pytest.mark.gpu

# (N, M, E per run, seats)
CASES = [(2, 5, 64, [1]), (5, 5, 32, [1, 3]), (8, 5, 16, [0, 2, 7]), (16, 5, 16, [0, 7, 15]), (130, 5, 8, [2, 64, 129])]
KINDS = ["trainer", "batch"]


def make(kind, N, M, E, seed=7):
    return trainer(N, M, E, seed=seed) if kind == "trainer" else batch(N, M, E)


def seeds_of(obj):
    return [int(obj.desc.seed)] if obj._partner_runs()[1] is None else list(obj.seeds)


def env_log(obj):
    """The env-team log since the previous call as [n, R, E]."""
    t = obj.env_partner_history()["env_team"]
    return t[:, None] if obj._partner_runs()[1] is None else t


def priority(obj):
    torch.cuda.synchronize()
    return {k: h(obj._priority[k]) for k in ("count", "sum", "table")}


def assert_same_state(a, b, log=True):
    pa, pb = buffers(a), buffers(b)
    for k in STATE:
        assert pa[k].tobytes() == pb[k].tobytes(), k
    if log:
        assert np.array_equal(a.env_partner_history()["env_team"], b.env_partner_history()["env_team"])


@pytest.mark.parametrize("N, M, E, seats", CASES)
@pytest.mark.parametrize("kind", KINDS)
def test_prioritized_mode_before_any_prioritize_is_the_uniform_mode(kind, N, M, E, seats):
    pool, _ = make_pool(N, seats)
    uniform, prio = make(kind, N, M, E), make(kind, N, M, E)
    uniform.set_partners(pool, per_env=True)
    prio.set_partners(pool, per_env=True, prioritized=True)
    assert prio.partners_prioritized and not uniform.partners_prioritized
    for obj in (uniform, prio):
        obj.train_episodes(2)
        obj.train_episode()
    if kind == "trainer":
        uniform.rollout(), prio.rollout()
    assert_same_state(uniform, prio)
    hist_u, hist_p = uniform.history(), prio.history()
    for k in hist_u:
        assert np.array_equal(hist_u[k], hist_p[k]), k
    W = prio.partner_weights()
    assert (W == 1 << 24).all() and W.shape == ((pool.Q,) if kind == "trainer" else (prio.R, pool.Q))


@pytest.mark.parametrize("N, M, E, seats", CASES)
@pytest.mark.parametrize("kind", KINDS)
def test_teams_of_the_same_rows_make_the_weights_invisible(kind, N, M, E, seats):
    """Q teams seating the same rows: whatever the weights, the episodes are the uniform mode's; only the log differs."""
    pool, host = make_pool(N, seats, P=7, Q=6)
    from ia2c_b200.partners import PartnerPool
    same = PartnerPool(host[0], np.repeat(host[1][:1], 6, axis=0), host[2], N, device="cuda:0")
    uniform, prio = make(kind, N, M, E), make(kind, N, M, E)
    uniform.set_partners(same, per_env=True)
    prio.set_partners(same, per_env=True, prioritized=True)
    for obj in (uniform, prio):
        obj.train_episodes(2)
    prio.prioritize_partners(power=3, floor=0.0)
    R = len(seeds_of(prio))
    rng = np.random.default_rng(N)
    W = rng.integers(0, 1 << 24, size=(R, 6))
    W[:, 2] = 0                                           # a team never drawn
    prio._priority["table"].copy_(torch.from_numpy(PP.table(W)))
    for obj in (uniform, prio):
        obj.train_episodes(2)
    assert_same_state(uniform, prio, log=False)
    log = env_log(prio)[-1]
    for r, seed in enumerate(seeds_of(prio)):
        assert np.array_equal(log[r], PP.env_teams(seed, prio.episode - 1, E, PP.table(W)[r]))
    assert not (log == 2).any()


def check_statistics_tables_and_draws(obj, E, Q, episodes=3):
    """Episodes one at a time: after each, the oracle adds the episode's returns and log; the device's statistics, then a
    prioritize's table, then the next episodes' draws equal the oracle's."""
    R, seeds = len(seeds_of(obj)), seeds_of(obj)
    count, total = np.zeros((R, Q), np.int64), np.zeros((R, Q), np.int64)
    table = PP.equal_table(R, Q)
    for rnd, (p, f, reset) in enumerate(((2, 0.1, False), (1, 0.0, True), (5, 0.3, True))):
        for _ in range(episodes):
            ep = obj.episode
            obj.train_episode()
            torch.cuda.synchronize()
            ret = h(obj.ep_return).reshape(R, E)
            log = env_log(obj)[0]
            for r in range(R):
                assert np.array_equal(log[r], PP.env_teams(seeds[r], ep, E, table[r])), (rnd, r)
            count, total = PP.accumulate(count, total, ret, log)
            got = priority(obj)
            assert np.array_equal(got["count"], count) and np.array_equal(got["sum"], total)
        out = obj.partner_returns()
        mean = PP.means(count, total)
        want = (count[0], mean[0]) if obj._partner_runs()[1] is None else (count, mean)
        assert np.array_equal(out["count"], want[0]) and np.array_equal(out["mean"], want[1], equal_nan=True)
        obj.prioritize_partners(power=p, floor=f, reset=reset)
        table = PP.table(PP.weights(count, total, p, f))
        got = priority(obj)
        assert np.array_equal(got["table"], table), rnd
        if reset:
            count, total = np.zeros_like(count), np.zeros_like(total)
        assert np.array_equal(got["count"], count) and np.array_equal(got["sum"], total)
    return table


@pytest.mark.parametrize("N, M, E, seats", CASES)
@pytest.mark.parametrize("kind", KINDS)
def test_statistics_tables_and_draws_equal_the_oracle(kind, N, M, E, seats):
    pool, _ = make_pool(N, seats, P=7, Q=5)
    obj = make(kind, N, M, E, seed=100 + N)
    obj.set_partners(pool, per_env=True, prioritized=True)
    table = check_statistics_tables_and_draws(obj, E, 5)
    assert (np.diff(table, axis=1) < (1 << 24)).any()      # the weights are not all equal any more


@pytest.mark.parametrize("N, M, E, seats", CASES)
def test_batch_runs_equal_standalone_prioritized_trainers(N, M, E, seats):
    pool, _ = make_pool(N, seats, Q=4)
    b = batch(N, M, E)
    b.set_partners(pool, per_env=True, prioritized=True)
    alone = [standalone_per_env(b, r, None) for r in range(b.R)]
    for tr in alone:
        tr.set_partners(pool, per_env=True, prioritized=True)
    for obj in [b] + alone:
        obj.train_episodes(2)
        obj.prioritize_partners(power=2, floor=0.1)
        obj.train_episode()
        obj.prioritize_partners(power=4, floor=0.0, reset=False)
        obj.train_episodes(2)
    torch.cuda.synchronize()
    teams, pb = b.env_partner_history()["env_team"], priority(b)
    for r, tr in enumerate(alone):
        assert_run_equals(b, r, tr)
        assert np.array_equal(tr.env_partner_history()["env_team"], teams[:, r])
        pt = priority(tr)
        for k in pt:
            assert np.array_equal(pt[k][0], pb[k][r]), (r, k)


@pytest.mark.parametrize("N, M, E, seats", [(2, 5, 10, [1]), (16, 5, 10, [3, 8])])
def test_checkpoints_resume_prioritized_training_exactly(N, M, E, seats, tmp_path):
    pool, _ = make_pool(N, seats)
    a = batch(N, M, E)
    a.set_partners(pool, per_env=True, prioritized=True)
    a.train_episodes(2)
    a.prioritize_partners(power=2, floor=0.1, reset=False)
    a.train_episode()
    path = str(tmp_path / "prio.pt")
    a.save(path)
    b = batch(N, M, E, hyper=HYPER)
    b.load(path)
    assert b.partners_prioritized
    r = 2
    alone = standalone_per_env(a, r, None)
    alone.load_state_dict(a.run_state_dict(r))
    assert alone.partners_prioritized
    a.env_partner_history()
    for obj in (a, b, alone):
        obj.train_episodes(2)
        obj.prioritize_partners(power=3, floor=0.2)
        obj.train_episode()
    torch.cuda.synchronize()
    assert_run_equals(a, r, alone)
    for k in BUFFERS:
        assert h(getattr(a, k)).tobytes() == h(getattr(b, k)).tobytes(), k
    pa, pb, pr = priority(a), priority(b), priority(alone)
    for k in pa:
        assert np.array_equal(pa[k], pb[k]) and np.array_equal(pa[k][r], pr[k][0]), k
    assert np.array_equal(a.env_partner_history()["env_team"], b.env_partner_history()["env_team"])
    old = a.state_dict()
    del old["partner_priority"]                          # a checkpoint from before prioritized draws: uniform
    b.load_state_dict(old)
    assert b.partners_per_env and not b.partners_prioritized


def _count(obj, fn):
    torch.cuda.synchronize()
    before = _lib.launch_count()
    fn(obj)
    return _lib.launch_count() - before


@pytest.mark.parametrize("kind, N, seats", [("trainer", 2, [1]), ("trainer", 16, [3]), ("batch", 2, [1]), ("batch", 16, [3, 8])])
def test_one_launch_more_per_episode_one_per_prioritize_and_no_synchronisation(kind, N, seats, monkeypatch):
    mk = (lambda: trainer(N, 5, 64, seed=1)) if kind == "trainer" else (lambda: batch(N, 5, 10))
    uniform, prio = mk(), mk()
    pool, _ = make_pool(N, seats)
    uniform.set_partners(pool, per_env=True)
    prio.set_partners(pool, per_env=True, prioritized=True)
    prio.ENV_PARTNER_LOG_CAPACITY = uniform.ENV_PARTNER_LOG_CAPACITY = 16
    assert _count(prio, lambda o: o.train_episode()) == _count(uniform, lambda o: o.train_episode()) + 1
    if kind == "trainer":
        assert _count(prio, lambda o: o.rollout()) == _count(uniform, lambda o: o.rollout()) + 1
    base = _count(uniform, lambda o: o.train_episodes(3))
    syncs = []
    with monkeypatch.context() as m:
        for owner in (torch.cuda.Stream, torch.cuda, torch.cuda.Event):
            m.setattr(owner, "synchronize", lambda *a, **k: syncs.append(1))
        before = _lib.launch_count()
        prio.train_episodes(3)
        assert _lib.launch_count() - before == base + 3
        before = _lib.launch_count()
        prio.prioritize_partners()
        assert _lib.launch_count() - before == 1
        assert syncs == []


def poor_team_pool(N=2):
    """Q = 4 teams of one seat (seat 0): team 2 always plays action 0 (the state falls to the -100 states), the others
    always play action 2 (it climbs)."""
    from ia2c_b200.partners import PartnerPool
    rows = np.zeros((2, _lib.ACTOR_P), dtype=np.float32)
    rows[0, -3:] = [-20.0, -20.0, 20.0]
    rows[1, -3:] = [20.0, -20.0, -20.0]
    return PartnerPool(rows, np.array([[0], [0], [1], [0]], dtype=np.int32), np.array([0], dtype=np.int32), N, device="cuda:0")


@pytest.mark.parametrize("kind", KINDS)
def test_a_poor_team_gets_the_largest_weight_and_is_drawn_by_it(kind):
    E, Q, poor = 512, 4, 2
    obj = trainer(2, 5, E, seed=21) if kind == "trainer" else batch(2, 5, E, seeds=[21, 8, 13])
    obj.set_partners(poor_team_pool(), per_env=True, prioritized=True)
    obj.train_episodes(4)
    mean = obj.partner_returns()["mean"].reshape(-1, Q)
    assert (mean.argmin(axis=1) == poor).all(), mean
    obj.prioritize_partners(power=2, floor=0.1)
    W = obj.partner_weights().reshape(-1, Q)
    assert (W[:, poor] == 1 << 24).all() and (np.delete(W, poor, axis=1) < 1 << 23).all(), W
    obj.env_partner_history()
    obj.train_episodes(8)
    teams = env_log(obj)                                   # [8, R, E]
    table = PP.table(W)
    for r, seed in enumerate(seeds_of(obj)):
        counts = np.bincount(teams[:, r].reshape(-1), minlength=Q)
        assert counts.argmax() == poor
        assert stats.chisquare(counts, W[r] / W[r].sum() * counts.sum()).pvalue > 1e-4, (counts, W[r])
        assert np.array_equal(teams[-1, r], PP.env_teams(seed, obj.episode - 1, E, table[r]))
