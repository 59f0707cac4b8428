"""Frozen partners per env on the GPU (set_partners(pool, per_env=True), ia2c_train_episode_env_partners): with one team the
mode equals per-episode seating byte for byte in everything the partner seats' actor rows do not feed; the oracle replays
per-env episodes from the device's state at production shapes; run r of a per-env batch equals a per-env standalone trainer;
the pool's table is evaluate's table; a corrupted device-side team sends exactly the envs that drew it back to their own rows;
an episode makes the launches of an unpartnered one and no synchronisation; checkpoints, set_partners(None), mode switches and
PBT keep the contracts."""
import numpy as np
import pytest
import torch

from ia2c_b200 import _lib
from oracle import belief as B
from oracle import loops as L
from oracle import env_partners as EP
from oracle import philox as P
from tests.helpers import host, rel_err
from tests.test_gpu_partners import HYPER, batch, make_pool, trainer
from tests.test_gpu_runs import BUFFERS, assert_run_equals, h
from tests.test_gpu_trainer_oracle_scale import RTOL, buffers as oracle_buffers, check_sampler, oracle_state

pytestmark = pytest.mark.gpu

ACTOR_FED = ("actor_params", "actor_m", "actor_v", "actor_grad_accum", "actor_grad")   # rows the partner seats' actors feed


def standalone_per_env(b, r, pool):
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    kw = dict(actor_kernel="columns") if b.N > 8 else {}
    tr = IA2CTrainer(b.E, n_agents=b.N, n_models=b.M, seed=b.seeds[r], init=reference_init(b.N, b.M, seed=b.seeds[r]),
                     **b.run_hyper(r), **kw)
    if pool is not None:
        tr.set_partners(pool, per_env=True)
    return tr


def assert_equal_outside_partner_actors(a, b, seats, N):
    """Every buffer byte-equal, except the partner seats' actor rows, Adam moments, gradient sums and actor losses."""
    torch.cuda.synchronize()
    learners = [i for i in range(N) if i not in seats]
    for k in BUFFERS + ("filter_action",):
        x, y = h(getattr(a, k)), h(getattr(b, k))
        if k in ACTOR_FED:
            x, y = x.reshape(-1, N, x.shape[-1])[:, learners], y.reshape(-1, N, y.shape[-1])[:, learners]
        elif k == "loss_out":
            x, y = x.reshape(2, -1, N), y.reshape(2, -1, N)
            assert x[0].tobytes() == y[0].tobytes(), "critic losses"
            x, y = x[1][:, learners], y[1][:, learners]
        assert np.ascontiguousarray(x).tobytes() == np.ascontiguousarray(y).tobytes(), k


Q1_CASES = [(2, 5, 64, [1]), (2, 3, 64, [0]), (5, 5, 32, [1, 3]), (8, 5, 16, [0, 2, 7]), (16, 5, 16, [0, 7, 15]),
            (130, 5, 8, [2, 64, 129])]


@pytest.mark.parametrize("N, M, E, seats", Q1_CASES)
def test_one_team_per_env_equals_per_episode_seating(N, M, E, seats):
    pool, _ = make_pool(N, seats, Q=1)
    per_env, per_ep = trainer(N, M, E, seed=7), trainer(N, M, E, seed=7)
    per_env.set_partners(pool, per_env=True)
    per_ep.set_partners(pool)
    per_env.train_episodes(2), per_ep.train_episodes(2)
    per_env.train_episode(), per_ep.train_episode()
    assert_equal_outside_partner_actors(per_env, per_ep, seats, N)
    out = per_env.env_partner_history()
    assert out["episode"].tolist() == [0, 1, 2] and out["env_team"].shape == (3, E) and (out["env_team"] == 0).all()
    hist_a, hist_b = per_env.history(), per_ep.history()
    learners = [i for i in range(N) if i not in seats]
    for k in hist_a:
        x, y = hist_a[k], hist_b[k]
        if k == "actor_loss":
            x, y = x[:, learners], y[:, learners]
        assert np.array_equal(x, y), k


def check_env_episode(b, st, actors, seed, episode, E, N, M, T):
    """One finished per-env episode of the device (buffers b) against the oracle state st taken before it, whose env e acted
    with actors[e]."""
    d = {k: host(v) for k, v in b.items()}
    idx = np.arange(E)[:, None] * N + np.arange(N)[None, :]
    u_act = np.stack([P.uniform_f32(seed, P.STREAM_ACTION, episode, t, idx) for t in range(T + 1)])
    u_bel = np.stack([P.belief_uniforms(seed, episode, t, idx, N - 1) for t in range(T + 1)])
    act = d["act"].astype(np.int64)
    traj = L.ia2c_rollout(st, E, actions=act, u_belief=u_bel)   # replayed actions: only its probs depend on the actors
    traj["probs"] = EP.env_probs(actors, traj["obs"])
    check_sampler(traj["probs"], u_act, act)
    upd = L.ia2c_update(st, traj)
    assert np.array_equal(d["obs"], traj["obs"]) and np.array_equal(d["reward"], traj["reward"].astype(np.float32))
    true_p, pred_p = L.partner_actions(traj, N)
    assert np.array_equal(d["partner_true"], true_p) and np.array_equal(d["partner_pred"], pred_p)
    assert np.array_equal(d["ep_return"], traj["ep_return"])
    for k in ("env_state", "env_hist", "env_cls", "env_elapsed"):
        assert np.array_equal(d[k], traj[k]), k
    assert np.array_equal(d["belief_records"][..., :M], B.to_hundredths(traj["belief"][T]))
    assert np.array_equal(d["belief_records"][..., 6], traj["pred"][T])
    err = {}
    for i in range(N):
        for name, got, want in (("critic_grad", d["critic_grad"][i, :-1], upd["critic_grad"][i]),
                                ("critic_loss", d["loss_out"][0, i], upd["critic_loss"][i]),
                                ("critic_params", d["critic_params"][i], st.critic[i]),
                                ("actor_grad_accum", d["actor_grad_accum"][i], upd["actor_grad"][i]),
                                ("actor_params", d["actor_params"][i], st.actor[i]),
                                ("actor_m", d["actor_m"][i], st.adam_a[i].m), ("actor_v", d["actor_v"][i], st.adam_a[i].v)):
            err[name] = max(err.get(name, 0.0), rel_err(got, want))
        scale = max(abs(float(upd["actor_loss"][i])), float(np.abs(upd["adv"][i]).mean()))
        err["actor_loss"] = max(err.get("actor_loss", 0.0), abs(float(d["loss_out"][1, i]) - float(upd["actor_loss"][i])) / scale)
    assert max(err.values()) < RTOL, {k: f"{v:.2e}" for k, v in err.items()}


# (N, M, E, T, seats, episodes)
ORACLE_CASES = [(2, 5, 4096, 30, [1], 3), (2, 3, 512, 30, [0], 2), (5, 5, 300, 30, [1, 3], 2), (8, 5, 200, 30, [0, 2, 7], 2),
                (16, 5, 300, 30, [0, 7, 15], 2), (130, 5, 24, 4, [2, 64, 129], 2)]


@pytest.mark.parametrize("N, M, E, T, seats, episodes", ORACLE_CASES)
def test_per_env_episodes_match_the_oracle(N, M, E, T, seats, episodes):
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    seed = 300 + N
    pool, host_pool = make_pool(N, seats, P=7, Q=5)
    tr = IA2CTrainer(E, n_agents=N, n_models=M, steps_per_episode=T, max_episode_steps=T, seed=seed, init=reference_init(N, M, seed=seed))
    tr.set_partners(pool, per_env=True)
    b, hp = oracle_buffers(tr), dict(gamma=0.9, beta=0.001, lr_actor=0.0001, lr_critic=0.0002)
    seen = set()
    for _ in range(episodes):
        episode = tr.episode
        st = oracle_state(b, hp, T, T)
        actors, log = EP.env_actors(host(tr.actor_params), host_pool, seed, episode, E)
        tr.train_episode()
        torch.cuda.synchronize()
        assert np.array_equal(tr.env_partner_history()["env_team"][0], EP.env_teams(seed, episode, E, 5)) and (log >= 0).all()
        seen |= set(log.tolist())
        check_env_episode(b, st, actors, seed, episode, E, N, M, T)
    assert len(seen) > 1


CASES = [(2, 5, 10, [1]), (2, 3, 10, [1]), (8, 5, 10, [1, 3, 6]), (16, 5, 10, [0, 5, 15]), (130, 6, 37, [3, 64, 129])]


@pytest.mark.parametrize("N, M, E, seats", CASES)
def test_per_env_batch_equals_per_env_standalone_runs(N, M, E, seats):
    pool, _ = make_pool(N, seats, Q=4)
    b = batch(N, M, E)
    b.set_partners(pool, per_env=True)
    alone = [standalone_per_env(b, r, pool) for r in range(b.R)]
    b.train_episodes(2)
    b.train_episode()
    for tr in alone:
        tr.train_episodes(2)
        tr.train_episode()
    torch.cuda.synchronize()
    teams = b.env_partner_history()["env_team"]
    assert teams.shape == (3, b.R, E) and np.array_equal(teams[:, 1], teams[:, 3])   # runs 1 and 3 share seed 29
    for r, tr in enumerate(alone):
        assert_run_equals(b, r, tr)
        assert np.array_equal(tr.env_partner_history()["env_team"], teams[:, r])
        assert np.array_equal(teams[2, r], EP.env_teams(b.seeds[r], 2, E, 4))


def test_the_pool_table_is_evaluates_table():
    from ia2c_b200.evaluate import evaluate_actors
    pool, _ = make_pool(16, [3], P=9)
    table = h(pool.policy_table(_lib.load()))
    assert pool.policy_table(_lib.load()) is pool.policy_table(_lib.load())   # built once
    ref = evaluate_actors(pool.rows, 1, pool.P, 1, 1, 4, 4, False, 0, 0, pool.device)["policy"][0]
    assert table.shape == (pool.P, 9, 3) and table.tobytes() == np.ascontiguousarray(ref, dtype=np.float32).tobytes()


@pytest.mark.parametrize("N, M, E, seats", [(2, 5, 256, [1]), (5, 5, 200, [4, 0]), (16, 5, 128, [3, 8])])
def test_a_corrupted_team_sends_exactly_its_envs_back_to_their_own_rows(N, M, E, seats):
    Q, seed = 4, 41
    pool, _ = make_pool(N, seats, P=7, Q=Q)
    bad_pool, _ = make_pool(N, seats, P=7, Q=Q)
    drawn = EP.env_teams(seed, 0, E, Q)
    bad = int(drawn[0])
    bad_pool.teams[bad, len(seats) - 1] = 7                  # a row outside the pool, written on the device
    clean, corrupted, own = trainer(N, M, E, seed=seed), trainer(N, M, E, seed=seed), trainer(N, M, E, seed=seed)
    clean.set_partners(pool, per_env=True)
    corrupted.set_partners(bad_pool, per_env=True)
    for tr in (clean, corrupted, own):
        tr.rollout()
    torch.cuda.synchronize()
    log = corrupted.env_partner_history()["env_team"][0]
    hit = drawn == bad
    assert (log[hit] == -1).all() and np.array_equal(log[~hit], drawn[~hit]) and 0 < hit.sum() < E
    assert np.array_equal(clean.env_partner_history()["env_team"][0], drawn)
    for k, axis in (("obs", 1), ("reward", 1), ("act", 1), ("partner_true", 1), ("partner_pred", 1), ("env_state", 0),
                    ("env_hist", 0), ("ep_return", 0), ("belief_records", 0)):
        got = h(getattr(corrupted, k))
        for ref, sel in ((own, hit), (clean, ~hit)):
            assert np.array_equal(np.compress(sel, got, axis), np.compress(sel, h(getattr(ref, k)), axis)), k


def _count(obj, fn):
    torch.cuda.synchronize()
    before = _lib.launch_count()
    fn(obj)
    return _lib.launch_count() - before


@pytest.mark.parametrize("kind, N, seats", [("trainer", 2, [1]), ("trainer", 16, [3]), ("runs", 2, [1]), ("runs", 16, [3, 8])])
def test_a_per_env_episode_adds_no_launch_and_never_synchronises(kind, N, seats, monkeypatch):
    make = (lambda: trainer(N, 5, 64, seed=1)) if kind == "trainer" else (lambda: batch(N, 5, 10))
    plain, per_env = make(), make()
    pool, _ = make_pool(N, seats)
    assert _count(per_env, lambda o: o.set_partners(pool, per_env=True)) == (1 if N > 8 else 0)   # the table, once per pool
    assert _count(per_env, lambda o: o.set_partners(pool, per_env=True)) == 0
    per_env.ENV_PARTNER_LOG_CAPACITY = 4
    assert _count(per_env, lambda o: o.train_episode()) == _count(plain, lambda o: o.train_episode())
    if kind == "trainer":
        assert _count(per_env, lambda o: o.rollout()) == _count(plain, lambda o: o.rollout())
    per_env.env_partner_history()                      # drained: the log is empty
    base_n = _count(plain, lambda o: o.train_episodes(3))
    first = per_env.episode
    syncs = []
    with monkeypatch.context() as m:
        for owner in (torch.cuda.Stream, torch.cuda, torch.cuda.Event):
            m.setattr(owner, "synchronize", lambda *a, **k: syncs.append(1))
        before = _lib.launch_count()
        per_env.train_episodes(3)                       # 3 records: the log (capacity 4) is full only now
        assert _lib.launch_count() - before == base_n and syncs == []
        per_env.train_episode()                         # the log drains first
        assert len(syncs) == 1
    assert per_env.env_partner_history()["episode"].tolist() == list(range(first, first + 4))


@pytest.mark.parametrize("N, M, E, seats", [(2, 5, 10, [1]), (16, 5, 10, [3, 8])])
def test_save_load_resumes_per_env_training(N, M, E, seats, tmp_path):
    pool, _ = make_pool(N, seats)
    a = batch(N, M, E)
    a.set_partners(pool, per_env=True)
    a.train_episodes(2)
    path = str(tmp_path / "per_env.pt")
    a.save(path)
    b = batch(N, M, E, hyper=HYPER)
    b.load(path)
    assert b.partners_per_env and h(b.partners.rows).tobytes() == h(pool.rows).tobytes()
    r = 2
    alone = standalone_per_env(a, r, None)
    alone.load_state_dict(a.run_state_dict(r))          # the run's checkpoint carries the pool and the mode
    assert alone.partners_per_env
    a.env_partner_history()
    for obj in (a, b, alone):
        obj.train_episodes(2)
    torch.cuda.synchronize()
    assert_run_equals(a, r, alone)
    for k in BUFFERS:
        assert h(getattr(a, k)).tobytes() == h(getattr(b, k)).tobytes(), k
    assert np.array_equal(a.env_partner_history()["env_team"], b.env_partner_history()["env_team"])
    old = a.state_dict()
    del old["partners_per_env"]                          # a checkpoint from before the mode existed: per-episode
    b.load_state_dict(old)
    assert b.partners is not None and not b.partners_per_env


def test_set_partners_none_and_mode_switches():
    pool, _ = make_pool(2, [1])
    a, b = batch(2, 5, 10), batch(2, 5, 10)
    a.set_partners(pool, per_env=True)
    b.set_partners(pool, per_env=True)
    a.train_episodes(2), b.train_episodes(2)
    a.set_partners(None)                                 # self-play from the partner seats' own (trained) rows
    b.set_partners(pool)                                 # per-episode seating from here on
    a.train_episode(), b.train_episode()
    assert not a.partners_per_env and not b.partners_per_env
    assert a.partner_history()["episode"].tolist() == [] and b.partner_history()["episode"].tolist() == [2]
    assert a.env_partner_history()["episode"].tolist() == [0, 1]
    c = batch(2, 5, 10)
    c.set_partners(pool, per_env=True)
    c.train_episodes(2)
    c.set_partners(None)
    c.train_episode()
    torch.cuda.synchronize()
    for k in BUFFERS:
        assert h(getattr(a, k)).tobytes() == h(getattr(c, k)).tobytes(), k
    b.set_partners(pool, per_env=True)
    b.train_episode()
    assert b.env_partner_history()["episode"].tolist() == [0, 1, 3]


@pytest.mark.parametrize("N, M, E, seats", [(2, 5, 10, [1]), (16, 5, 10, [3, 8])])
def test_a_pbt_generation_between_per_env_episodes_keeps_runs_standalone(N, M, E, seats):
    pool, _ = make_pool(N, seats)
    b = batch(N, M, E)
    b.set_partners(pool, per_env=True)
    b.train_episodes(4)
    b.exploit_explore(4, fraction=0.34, seed=7)
    assert (b.pbt_history()["donor"] >= 0).any()
    alone = []
    for r in range(b.R):
        tr = standalone_per_env(b, r, None)
        tr.load_state_dict(b.run_state_dict(r))
        alone.append(tr)
    b.train_episodes(2)
    for tr in alone:
        tr.train_episodes(2)
    torch.cuda.synchronize()
    for r, tr in enumerate(alone):
        assert_run_equals(b, r, tr)
