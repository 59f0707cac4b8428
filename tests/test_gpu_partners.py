"""Training against frozen partners on the GPU (ia2c_seat_partners through set_partners): a seated trainer equals its twin
into whose seat rows the oracle's drawn team is written before each episode, byte for byte; run r of a seated batch equals
a standalone trainer with the same seed and pool; the call writes only the drawn seat rows and its log; bad device-side
entries leave their run untouched; pools are frozen; checkpoints, set_partners(None) and PBT keep the contracts; and a
seated episode is one launch more than an unseated one, with no synchronisation."""
import ctypes as C

import numpy as np
import pytest
import torch

from ia2c_b200 import _lib
from oracle import partners as PT
from tests.test_gpu_runs import BUFFERS, assert_run_equals, h

pytestmark = pytest.mark.gpu

STATE = BUFFERS + ("filter_action",)
SEEDS = [11, 29, 3, 29, 5, 17]
HYPER = dict(lr_actor=[1e-4, 3e-4, 5e-5, 2e-3, 7e-4, 1.5e-4], lr_critic=[2e-4, 1e-3, 7e-5, 5e-4, 3e-4, 9e-4],
             beta=[1e-3, 1e-2, 0.0, 5e-2, 2e-3, 3e-2], gamma=[0.9, 0.99, 0.5, 0.75, 0.8, 0.95])


def pool_arrays(N, seats, P=7, Q=5, seed=0):
    rng = np.random.RandomState(seed)
    rows = (rng.normal(size=(P, _lib.ACTOR_P)) * 0.5).astype(np.float32)
    return rows, rng.randint(0, P, size=(Q, len(seats))).astype(np.int32), np.asarray(seats, dtype=np.int32)


def make_pool(N, seats, **kw):
    from ia2c_b200.partners import PartnerPool
    host = pool_arrays(N, seats, **kw)
    return PartnerPool(*host, n_agents=N, device="cuda:0"), host


def trainer(N, M, E, seed, **kw):
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    return IA2CTrainer(E, n_agents=N, n_models=M, seed=seed, init=reference_init(N, M, seed=seed), **kw)


def batch(N, M, E, seeds=SEEDS, hyper=HYPER):
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    cls = IA2CRunsMany if N > 8 else IA2CRuns
    return cls(E, seeds, n_agents=N, n_models=M, **{k: v[:len(seeds)] for k, v in (hyper or {}).items()})


def buffers(obj):
    torch.cuda.synchronize()
    return {k: h(getattr(obj, k)) for k in STATE}


def differing(a, b):
    pa, pb = buffers(a), buffers(b)
    return [k for k in STATE if pa[k].tobytes() != pb[k].tobytes()]


def oracle_seat(obj, host, seed):
    """Write the oracle's drawn team into obj's seat rows for the episode obj is about to run; returns the oracle's log."""
    new, log = PT.seat(h(obj.actor_params), host, obj.episode, seed)
    obj.actor_params.copy_(torch.from_numpy(new))
    return log


@pytest.mark.parametrize("N, M, E, seats", [(2, 5, 64, [1]), (5, 5, 32, [1, 3]), (16, 5, 16, [0, 7, 15]),
                                            (130, 5, 8, [2, 64, 129])])
def test_seated_trainer_equals_its_twin_seated_by_the_oracle(N, M, E, seats):
    pool, host = make_pool(N, seats)
    tr, twin = trainer(N, M, E, seed=5), trainer(N, M, E, seed=5)
    assert (N > 64) == (not tr.desc.flags & _lib.FLAG_ACTOR_COLUMNS)   # N = 130 runs the default pipelined actor kernel
    tr.set_partners(pool)
    tr.train_episodes(2)
    tr.train_episode()
    tr.rollout(), tr.update()                # IA2CTrainer.rollout seats too (update does not advance the episode)
    logs = []
    for k in range(4):
        logs.append(oracle_seat(twin, host, 5)[0])
        if k < 3:
            twin.train_episode()
        else:
            twin.rollout(), twin.update()
    assert differing(tr, twin) == []
    out = tr.partner_history()
    assert out["episode"].tolist() == [0, 1, 2, 3]
    assert out["team"].dtype == np.int32 and out["team"].tolist() == logs == [PT.team(5, k, 5) for k in range(4)]
    assert tr.history()["episode"].tolist() == [0, 1]


def standalone_like(b, r, pool):
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    kw = dict(actor_kernel="columns") if b.N > 8 else {}
    tr = IA2CTrainer(b.E, n_agents=b.N, n_models=b.M, seed=b.seeds[r], init=reference_init(b.N, b.M, seed=b.seeds[r]),
                     **b.run_hyper(r), **kw)
    tr.set_partners(pool)
    return tr


def assert_state_dicts_equal(sa, sb):
    for k in sa:
        if isinstance(sa[k], torch.Tensor):
            assert sa[k].numpy().tobytes() == sb[k].numpy().tobytes(), k
    for k in ("rows", "teams", "seats"):
        assert sa["partners"][k].numpy().tobytes() == sb["partners"][k].numpy().tobytes(), k


CASES = [(2, 5, 10, [1]), (8, 5, 10, [1, 3, 6]), (16, 5, 10, [0, 5, 15]), (130, 6, 37, [3, 64, 129])]


@pytest.mark.parametrize("N, M, E, seats", CASES)
def test_seated_batch_equals_seated_standalone_runs(N, M, E, seats):
    pool, _ = make_pool(N, seats, Q=4)
    b = batch(N, M, E)
    b.set_partners(pool)
    alone = [standalone_like(b, r, pool) for r in range(b.R)]
    b.train_episodes(2)
    b.train_episode()
    for tr in alone:
        tr.train_episodes(2)
        tr.train_episode()
    torch.cuda.synchronize()
    teams = b.partner_history()["team"]
    assert teams.shape == (3, b.R) and teams[:, 1].tolist() == teams[:, 3].tolist()   # runs 1 and 3 share seed 29
    for r, tr in enumerate(alone):
        assert_run_equals(b, r, tr)
        assert_state_dicts_equal(b.run_state_dict(r), tr.state_dict())
        assert tr.partner_history()["team"].tolist() == teams[:, r].tolist()


def _raw_seat(b, pool_rows, teams, seats, episode):
    """ia2c_seat_partners on a batch's descriptors with caller-made device arrays (no host checks); returns the log."""
    rows_d = torch.from_numpy(pool_rows).cuda()
    teams_d, seats_d = torch.from_numpy(teams).cuda(), torch.from_numpy(seats).cuda()
    log = torch.full((b.R,), 12345, dtype=torch.int32, device="cuda")
    p = _lib.PartnerDesc()
    p.rows, p.P, p.seats, p.S = rows_d.data_ptr(), pool_rows.shape[0], seats_d.data_ptr(), seats.shape[0]
    p.teams, p.Q, p.episode, p.log_team = teams_d.data_ptr(), teams.shape[0], episode, log.data_ptr()
    _lib.check(b.lib.ia2c_seat_partners(C.byref(b.desc), C.byref(b.runs_desc), C.byref(p),
                                        torch.cuda.current_stream().cuda_stream), "ia2c_seat_partners")
    return h(log)


def everything(b):
    from ia2c_b200.runs import _ENV, _NET
    torch.cuda.synchronize()
    return {k: h(getattr(b, k)) for k in _NET + tuple(_ENV) + ("loss_out", "partials")}


def test_a_direct_call_writes_only_the_drawn_seat_rows_and_the_log():
    b = batch(5, 5, 10, seeds=SEEDS[:4])
    b.train_episodes(2)
    rows, teams, seats = pool_arrays(5, [4, 0], P=6, Q=3)
    pre = everything(b)
    log = _raw_seat(b, rows, teams, seats, episode=9)
    post = everything(b)
    new, olog = PT.seat(pre["actor_params"], (rows, teams, seats), 9, b.seeds)
    assert log.tolist() == olog.tolist() and (olog >= 0).all()
    assert post["actor_params"].tobytes() == new.tobytes()
    assert [k for k in pre if k != "actor_params" and pre[k].tobytes() != post[k].tobytes()] == []
    changed = np.flatnonzero((pre["actor_params"] != post["actor_params"]).any(1))
    assert set(changed.tolist()) <= {r * 5 + s for r in range(4) for s in (4, 0)}


def test_out_of_range_device_entries_leave_their_run_untouched():
    Q, episode = 8, 3
    seeds = []
    for s in range(1000, 2000):   # four runs that draw four different teams
        if PT.team(s, episode, Q) not in [PT.team(x, episode, Q) for x in seeds]:
            seeds.append(s)
        if len(seeds) == 4:
            break
    b = batch(4, 5, 10, seeds=seeds, hyper=None)
    b.train_episode()
    rows, teams, seats = pool_arrays(4, [1, 2], P=6, Q=Q)
    bad = PT.team(seeds[1], episode, Q)
    teams[bad, 1] = 6                                   # run 1's team seats a row outside the pool
    pre = everything(b)
    log = _raw_seat(b, rows, teams, seats, episode)
    new, olog = PT.seat(pre["actor_params"], (rows, teams, seats), episode, seeds)
    assert log.tolist() == olog.tolist() and log[1] == -1 and (np.delete(log, 1) >= 0).all()
    post = everything(b)
    assert post["actor_params"].tobytes() == new.tobytes()
    assert post["actor_params"][4:8].tobytes() == pre["actor_params"][4:8].tobytes()
    teams[bad, 1] = -1                                  # negative rows are refused the same way
    assert _raw_seat(b, rows, teams, seats, episode)[1] == -1
    log = _raw_seat(b, rows, pool_arrays(4, [1, 2], P=6, Q=Q)[1], np.array([1, 4], dtype=np.int32), episode)   # a seat >= N
    assert (log == -1).all()
    assert everything(b)["actor_params"].tobytes() == post["actor_params"].tobytes()


def test_a_pool_is_frozen_when_made():
    from ia2c_b200.partners import PartnerPool
    src = batch(4, 5, 10, seeds=[1, 2, 3], hyper=None)
    src.train_episodes(2)
    snap = src.state_dict()
    live = PartnerPool.from_sources(src)
    src.train_episodes(3)                               # the source trains on: the pool must not see it
    again = batch(4, 5, 10, seeds=[1, 2, 3], hyper=None)
    again.load_state_dict(snap)
    frozen = PartnerPool.from_sources([again], split=2)
    assert (live.S, live.Q, h(live.seats).tolist()) == (2, 3, [2, 3])
    assert h(live.rows).tobytes() == h(frozen.rows).tobytes()
    actors = snap["actor_params"].numpy().reshape(3, 4, -1)
    for team in range(3):   # team b seats agents split .. N-1 of source run b in their own seats: cross_play's cell (a, b)
        assert h(live.rows)[h(live.teams)[team]].tobytes() == actors[team, 2:].tobytes()
    a, c = batch(4, 5, 10, seeds=[7, 8], hyper=None), batch(4, 5, 10, seeds=[7, 8], hyper=None)
    a.set_partners(live), c.set_partners(frozen)
    a.train_episodes(3), c.train_episodes(3)
    assert differing(a, c) == []


def test_set_partners_none_returns_to_self_play():
    a, b = batch(2, 5, 10), batch(2, 5, 10)
    pool, _ = make_pool(2, [1])
    a.set_partners(pool)
    a.train_episodes(2)
    sd = a.state_dict()
    assert set(sd["partners"]) == {"rows", "teams", "seats"}
    a.set_partners(None)
    b.set_partners(pool)
    b.load_state_dict({k: v for k, v in sd.items() if k != "partners"})   # a checkpoint without a pool clears it
    assert b.partners is None
    a.train_episodes(2), b.train_episodes(2)
    assert differing(a, b) == []
    assert a.partner_history()["episode"].tolist() == [0, 1] and b.partner_history()["episode"].tolist() == []


@pytest.mark.parametrize("N, M, E, seats", [(2, 5, 10, [1]), (16, 5, 10, [3, 8])])
def test_save_load_resumes_seated_training(N, M, E, seats, tmp_path):
    pool, _ = make_pool(N, seats)
    a = batch(N, M, E)
    a.set_partners(pool)
    a.train_episodes(2)
    path = str(tmp_path / "seated.pt")
    a.save(path)
    b = batch(N, M, E, hyper=HYPER)
    b.load(path)
    assert b.partners is not None and h(b.partners.rows).tobytes() == h(pool.rows).tobytes()
    r = 2
    alone = standalone_like(a, r, None)
    alone.load_state_dict(a.run_state_dict(r))          # the run's checkpoint carries the pool
    assert alone.partners is not None
    a.partner_history()
    for obj in (a, b, alone):
        obj.train_episodes(2)
    assert differing(a, b) == []
    assert a.partner_history()["team"].tolist() == b.partner_history()["team"].tolist()
    torch.cuda.synchronize()
    assert_run_equals(a, r, alone)


@pytest.mark.parametrize("N, M, E, seats", [(2, 5, 10, [1]), (16, 5, 10, [3, 8])])
def test_a_pbt_generation_between_seated_episodes_keeps_runs_standalone(N, M, E, seats):
    pool, _ = make_pool(N, seats)
    b = batch(N, M, E)
    b.set_partners(pool)
    b.train_episodes(4)
    b.exploit_explore(4, fraction=0.34, seed=7)
    assert (b.pbt_history()["donor"] >= 0).any()
    alone = []
    for r in range(b.R):
        tr = standalone_like(b, r, None)
        tr.load_state_dict(b.run_state_dict(r))
        alone.append(tr)
    b.train_episodes(2)
    for tr in alone:
        tr.train_episodes(2)
    torch.cuda.synchronize()
    for r, tr in enumerate(alone):
        assert_run_equals(b, r, tr)


def _count_launches(obj, fn):
    torch.cuda.synchronize()
    before = _lib.launch_count()
    fn(obj)
    return _lib.launch_count() - before


@pytest.mark.parametrize("kind, N, seats", [("trainer", 2, [1]), ("runs", 2, [1]), ("runs", 16, [3, 8])])
def test_a_seated_episode_is_one_launch_more_and_never_synchronises(kind, N, seats, monkeypatch):
    make = (lambda: trainer(N, 5, 64, seed=1)) if kind == "trainer" else (lambda: batch(N, 5, 10))
    plain, seated = make(), make()
    pool, _ = make_pool(N, seats)
    seated.set_partners(pool)
    seated.PARTNER_LOG_CAPACITY = 4
    base = _count_launches(plain, lambda o: o.train_episode())
    assert _count_launches(seated, lambda o: o.train_episode()) == base + 1
    base_n = _count_launches(plain, lambda o: o.train_episodes(2))
    syncs = []
    with monkeypatch.context() as m:
        for owner in (torch.cuda.Stream, torch.cuda, torch.cuda.Event):
            m.setattr(owner, "synchronize", lambda *a, **k: syncs.append(1))
        before = _lib.launch_count()
        seated.train_episodes(2)                        # log slots 2 and 3 of 4: nothing to drain yet
        assert _lib.launch_count() - before == base_n + 2 and syncs == []
        seated.train_episode()                          # 3 records pending (capacity - 1): the log drains first
        assert len(syncs) == 1
    assert seated.partner_history()["episode"].tolist() == [0, 1, 2, 3]
