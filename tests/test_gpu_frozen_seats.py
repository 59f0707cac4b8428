"""Frozen seats on the GPU (ia2c_train_episode_frozen, freeze_seats): a frozen trainer or batch equals an unfrozen twin whose
frozen seats' per-net rows are copied back after every episode, in every buffer but the documented ones (frozen losses NaN; from 9
agents, frozen partner predictions 0xFF and belief records untouched); frozen rows and step counters stand still; run r of a
frozen batch equals the standalone frozen trainer with its seed; checkpoints resume exactly; the trained seat matches
oracle/frozen_seats.py at the benchmark's shape; every refusal raises before any device work."""
import numpy as np
import pytest
import torch

from oracle import frozen_seats as FS
from oracle import loops as L
from oracle import philox as P
from tests.helpers import host, rel_err

pytestmark = pytest.mark.gpu
NET = ("actor_params", "critic_params", "actor_grad", "critic_grad", "actor_m", "actor_v", "critic_m", "critic_v", "actor_step",
       "critic_step", "actor_grad_accum")
OTHER = ("filter_action", "env_state", "env_hist", "env_cls", "env_elapsed", "ep_return", "obs", "reward", "act", "partner_true")
MODES = ("none", "seat", "env", "prio")


def make(kind, N, E=64, R=8, fused_critic=None):
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    if kind == "trainer":
        return IA2CTrainer(E, n_agents=N, seed=7 + N, init=reference_init(N, 5, seed=7 + N), actor_kernel="columns",
                           fused_critic=fused_critic)
    seeds = [100 + 3 * r for r in range(R)]
    hyper = dict(lr_actor=[1e-4 * (1 + r) for r in range(R)], lr_critic=[2e-4 * (1 + 0.5 * r) for r in range(R)],
                 beta=[0.001 * (1 + r) for r in range(R)], gamma=[0.9 - 0.01 * r for r in range(R)])
    cls = IA2CRuns if kind == "runs" else IA2CRunsMany
    return cls(E, seeds, n_agents=N, **hyper)


def pool_for(obj, seats=None):
    """A pool of 3 teams over `seats` (default N/2 .. N-1)."""
    from ia2c_b200.partners import PartnerPool
    from ia2c_b200.trainer import reference_init
    N = obj.N
    seats = np.arange(N // 2, N) if seats is None else np.asarray(seats)
    rows = np.concatenate([reference_init(N, 5, seed=900 + k)[0][seats] for k in range(3)]).astype(np.float32)
    S = len(seats)
    return PartnerPool(rows, np.arange(3 * S).reshape(3, S), seats, N, device=obj.device)


def freeze_pool_seats(obj, pool):
    """The documented call, freeze_seats(pool.seats) with the pool's device tensor, and the set it leaves."""
    obj.freeze_seats(pool.seats)
    frozen = set(int(s) for s in host(pool.seats))
    assert obj.frozen_seats == frozen
    return frozen


def set_mode(obj, mode, pool):
    if mode == "seat":
        obj.set_partners(pool)
    elif mode in ("env", "prio"):
        obj.set_partners(pool, per_env=True, prioritized=mode == "prio")


def rows_of(obj, seats):
    R = getattr(obj, "R", 1)
    return [r * obj.N + s for r in range(R) for s in sorted(seats)]


def buf(obj, k):
    return getattr(obj, k)


def assert_twins(a, b, frozen):
    """a (frozen) and b (unfrozen, frozen rows restored) hold the same bytes but where documented."""
    N, R = a.N, getattr(a, "R", 1)
    rows = rows_of(a, frozen)
    trained = [n for n in range(R * N) if n not in rows]
    for k in NET + OTHER:
        assert torch.equal(buf(a, k), buf(b, k)), k
    la, lb = host(a.loss_out).reshape(2, R * N), host(b.loss_out).reshape(2, R * N)
    assert np.isnan(la[:, rows]).all()
    assert np.array_equal(la[:, trained], lb[:, trained])
    pa, pb = host(a.partner_pred), host(b.partner_pred)
    ra, rb = host(a.belief_records), host(b.belief_records)
    seat = np.array([n in frozen for n in range(N)])
    if N <= 8:
        assert np.array_equal(pa, pb) and np.array_equal(ra, rb)
    else:
        assert np.array_equal(pa[..., ~seat], pb[..., ~seat]) and (pa[..., seat] == 0xFF).all()
        assert np.array_equal(ra[:, ~seat], rb[:, ~seat])


def run_twins(kind, N, mode, episodes=6, E=64, R=8, fused_critic=None, seats=None):
    a, b = make(kind, N, E, R, fused_critic), make(kind, N, E, R, fused_critic)
    pool = pool_for(a, seats)
    set_mode(a, mode, pool), set_mode(b, mode, pool)
    frozen = freeze_pool_seats(a, pool)
    assert b.frozen_seats == frozenset()
    rows = rows_of(a, frozen)
    start = {k: buf(a, k)[rows].clone() for k in NET}
    recs = host(a.belief_records).copy()
    stream = torch.cuda.current_stream().cuda_stream
    for ep in range(episodes):
        if mode == "seat":   # the seating is what the episode starts with (the same draw when train_episode repeats it)
            with torch.cuda.device(b.device):
                b._seat_partners(stream)
        snap = {k: buf(b, k)[rows].clone() for k in NET}
        a.train_episode(), b.train_episode()
        for k in NET:
            buf(b, k)[rows] = snap[k]
        if mode == "prio" and ep == 2:
            a.prioritize_partners(), b.prioritize_partners()
        torch.cuda.synchronize()
        assert_twins(a, b, frozen)
    for k in NET:   # frozen rows, step counters included, stand still (but the actor rows seating writes)
        if not (mode == "seat" and k == "actor_params"):
            assert torch.equal(buf(a, k)[rows], start[k]), k
    if N > 8:
        seat = np.array([n in frozen for n in range(N)])
        assert np.array_equal(host(a.belief_records)[:, seat], recs[:, seat])
    return a, b


CASES = ([("trainer", 2, m, fc, None) for m in MODES for fc in (True, False)]
         + [("trainer", n, m, None, None) for n in (4, 8, 16, 64) for m in MODES]
         + [("trainer", 130, m, None, None) for m in ("none", "env")] + [("runs", 4, m, None, None) for m in MODES]
         + [("runs", 2, "prio", None, None)] + [("many", 16, m, None, None) for m in MODES])
# frozen sets that are not a suffix of the seats, so that the trained seat list and the frozen rows' seats differ from their
# grid rows (the 130-agent set spans three words of the mask)
SCATTERED = ([("trainer", 2, m, fc, (0,)) for m in ("none", "seat", "env") for fc in (True, False)]
             + [("trainer", 4, m, None, (0, 2)) for m in MODES] + [("trainer", 8, "env", None, (1, 2, 6))]
             + [("trainer", 16, m, None, (0, 3, 4, 9, 14)) for m in ("none", "env", "prio")]
             + [("trainer", 64, m, None, (1, 7, 30, 31, 62)) for m in ("none", "env")]
             + [("trainer", 130, m, None, (0, 63, 64, 65, 129)) for m in ("none", "env")]
             + [("runs", 4, m, None, (0, 2)) for m in ("seat", "env", "prio")] + [("runs", 2, "env", None, (0,))]
             + [("many", 16, m, None, (0, 3, 4, 9, 14)) for m in ("none", "env")])


def _id(k, n, m, fc, seats):
    return f"{k}-N{n}-{m}" + ("" if fc is None else f"-fc{int(fc)}") + ("" if seats is None else "-seats" + "_".join(map(str, seats)))


@pytest.mark.parametrize("kind, N, mode, fused_critic, seats", CASES + SCATTERED, ids=[_id(*c) for c in CASES + SCATTERED])
def test_restore_equivalence(kind, N, mode, fused_critic, seats):
    E = 16 if N >= 64 else 64
    run_twins(kind, N, mode, E=E, R=4 if kind == "many" else 8, fused_critic=fused_critic, seats=seats)


@pytest.mark.parametrize("kind, N, mode, seats", [("runs", 4, "env", None), ("runs", 2, "seat", None), ("many", 16, "prio", None),
                                                  ("runs", 4, "env", (1,)), ("many", 16, "env", (2, 5, 11))])
def test_batch_run_equals_standalone(kind, N, mode, seats):
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    R = 4 if kind == "many" else 8
    batch = make(kind, N, E=32, R=R)
    pool = pool_for(batch, seats)
    set_mode(batch, mode, pool)
    frozen = freeze_pool_seats(batch, pool)
    solo = []
    for r in (0, R - 1):
        t = IA2CTrainer(32, n_agents=N, seed=batch.seeds[r], init=reference_init(N, 5, seed=batch.seeds[r]),
                        actor_kernel="columns", **batch.run_hyper(r))
        set_mode(t, mode, pool), t.freeze_seats(frozen)
        solo.append((r, t))
    for ep in range(4):
        batch.train_episode()
        for _, t in solo:
            t.train_episode()
        if mode == "prio" and ep == 1:
            batch.prioritize_partners()
            for _, t in solo:
                t.prioritize_partners()
    torch.cuda.synchronize()
    for r, t in solo:
        v = batch.run_view(r)
        for k in NET + OTHER + ("partner_pred", "belief_records"):
            assert torch.equal(v[k], getattr(t, k)), (r, k)
        assert np.array_equal(host(v["loss_out"]), host(t.loss_out), equal_nan=True)


@pytest.mark.parametrize("kind, N", [("trainer", 2), ("trainer", 16), ("runs", 4)])
def test_checkpoint_resumes_and_unfreezes(kind, N):
    a = make(kind, N, E=32, R=4)
    pool = pool_for(a)
    set_mode(a, "env", pool)
    freeze_pool_seats(a, pool)
    for _ in range(3):
        a.train_episode()
    sd = a.state_dict()
    assert sd["frozen_seats"] == sorted(a.frozen_seats)
    b = make(kind, N, E=32, R=4)
    b.load_state_dict(sd)
    assert b.frozen_seats == a.frozen_seats and b.partners_per_env
    for _ in range(3):
        a.train_episode(), b.train_episode()
    torch.cuda.synchronize()
    for k in NET + OTHER + ("partner_pred", "belief_records"):
        assert torch.equal(buf(a, k), buf(b, k)), k
    # freeze_seats(None) continues like an unfrozen trainer loaded from the same state
    sd = a.state_dict()
    c = make(kind, N, E=32, R=4)
    del sd["frozen_seats"]   # a checkpoint without the set loads as nothing frozen
    c.load_state_dict(sd)
    assert c.frozen_seats == frozenset()
    a.freeze_seats(None)
    for _ in range(2):
        a.train_episode(), c.train_episode()
    torch.cuda.synchronize()
    for k in NET + OTHER + ("partner_pred", "belief_records", "loss_out"):
        assert torch.equal(buf(a, k), buf(c, k)), k


def test_matches_oracle_at_benchmark_shape():
    """N = 2, E = 4096, seat 1 frozen, device Philox: the trained seat within the oracle tolerance of the existing oracle tests,
    the trajectory bit for bit, the frozen seat unchanged."""
    from tests.test_gpu_trainer_oracle_scale import RTOL, check_sampler, oracle_state
    N, M, E, T = 2, 5, 4096, 30
    tr = make("trainer", N, E=E)
    tr.freeze_seats({1})
    hp = dict(gamma=0.9, beta=0.001, lr_actor=0.0001, lr_critic=0.0002)
    for _ in range(2):
        b = {k: getattr(tr, k) for k in NET + OTHER + ("partner_pred", "belief_records", "loss_out")}
        st = oracle_state(b, hp, T, 30)
        episode = tr.episode
        tr.train_episode()
        torch.cuda.synchronize()
        d = {k: host(v) for k, v in b.items()}
        idx = np.arange(E)[:, None] * N + np.arange(N)[None, :]
        u_act = np.stack([P.uniform_f32(tr.seed, P.STREAM_ACTION, episode, t, idx) for t in range(T + 1)])
        u_bel = np.stack([P.belief_uniforms(tr.seed, episode, t, idx, N - 1) for t in range(T + 1)])
        traj, upd = FS.frozen_episode(st, E, {1}, actions=d["act"].astype(np.int64), u_belief=u_bel)
        check_sampler(traj["probs"], u_act, d["act"].astype(np.int64))
        assert np.array_equal(d["obs"], traj["obs"]) and np.array_equal(d["partner_pred"], traj["partner_pred"])
        assert np.array_equal(d["actor_step"], [a.t for a in st.adam_a]) and np.array_equal(d["critic_step"], [a.t for a in st.adam_c])
        assert np.isnan(d["loss_out"][:, 1]).all()
        assert np.array_equal(d["actor_params"][1], st.actor[1].astype(np.float32))
        assert np.array_equal(d["critic_params"][1], st.critic[1].astype(np.float32))
        errs = [rel_err(d["critic_params"][0], st.critic[0]), rel_err(d["actor_params"][0], st.actor[0]),
                rel_err(d["critic_grad"][0, :-1], upd["critic_grad"][0]), rel_err(d["actor_grad_accum"][0], upd["actor_grad"][0]),
                rel_err(d["loss_out"][0, 0], upd["critic_loss"][0])]
        assert max(errs) < RTOL, errs


def test_python_refusals():
    from ia2c_b200 import _lib
    from ia2c_b200.a2c import A2COrgTrainer
    from ia2c_b200.trainer import IA2CTrainer
    with pytest.raises(_lib.IA2CError, match="per-step rollout"):
        IA2CTrainer(16, n_agents=2, fused_rollout=False, actor_kernel="columns").freeze_seats({1})
    with pytest.raises(_lib.IA2CError, match="per-step rollout"):
        IA2CTrainer(16, n_agents=16, rollout_kernel="step").freeze_seats({1})
    with pytest.raises(_lib.IA2CError, match="per-step rollout"):
        IA2CTrainer(16, n_agents=16, belief_kernel="step").freeze_seats({1})
    with pytest.raises(_lib.IA2CError, match="above 256"):
        IA2CTrainer(2, n_agents=300, steps_per_episode=2).freeze_seats({1})
    with pytest.raises(_lib.IA2CError, match='actor_kernel="columns"'):
        IA2CTrainer(16, n_agents=130, steps_per_episode=2).freeze_seats({1})
    with pytest.raises(_lib.IA2CError, match="one joint agent"):
        A2COrgTrainer(num_envs=4).freeze_seats({0})
    tr = IA2CTrainer(16, n_agents=3)
    for bad in ({3}, set(), {0, 1, 2}, 1):
        with pytest.raises(ValueError):
            tr.freeze_seats(bad)
    tr.world = 2
    with pytest.raises(_lib.IA2CError, match="one GPU"):
        tr.freeze_seats({1})
    tr.world = 1
    tr.freeze_seats({1})
    sd = tr.state_dict()
    pipe = IA2CTrainer(16, n_agents=3, actor_kernel="pipe", seed=99)
    before_params = pipe.actor_params.clone()
    sd["actor_params"] = sd["actor_params"] + 1.0
    with pytest.raises(_lib.IA2CError, match='actor_kernel="columns"'):
        pipe.load_state_dict(sd)
    assert torch.equal(pipe.actor_params, before_params) and pipe.episode == 0 and pipe.frozen_seats == frozenset()
    before = _lib.launch_count()
    for call in (tr.rollout, tr.update, tr.train_episode_timed, lambda: tr.train_episodes_host([]),
                 lambda: tr.train_episode_host(None, None)):
        with pytest.raises(_lib.IA2CError, match="freeze_seats"):
            call()
    assert _lib.launch_count() == before
