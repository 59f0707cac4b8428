"""Population-based training on the GPU (ia2c_pbt_step through IA2CRuns.exploit_explore): the log and every byte the step
writes equal the oracle's generation, nothing else changes, runs continue as standalone trainers with their new
hyper-parameters, and the step is deterministic, checkpointable, asynchronous and two launches long."""
import numpy as np
import pytest
import torch

from ia2c_b200 import _lib
from oracle import pbt as P
from tests.test_gpu_runs import BUFFERS, assert_run_equals, h

pytestmark = pytest.mark.gpu

# distinct per-run hyper-parameters, a repeated seed
SEEDS = [11, 29, 3, 29, 5, 17]
HYPER = dict(lr_actor=[1e-4, 3e-4, 5e-5, 2e-3, 7e-4, 1.5e-4], lr_critic=[2e-4, 1e-3, 7e-5, 5e-4, 3e-4, 9e-4],
             beta=[1e-3, 1e-2, 0.0, 5e-2, 2e-3, 3e-2], gamma=[0.9, 0.99, 0.5, 0.75, 0.8, 0.95])
STATE = BUFFERS + ("filter_action",)
LOG = (("fitness", np.float64), ("rank", np.int32), ("donor", np.int32), ("lr_actor", np.float64), ("lr_critic", np.float64),
       ("gamma", np.float32), ("beta", np.float32))
# IA2CRuns at N = 2 and 8; IA2CRunsMany at N = 16 and at N = 130 (two belief blocks per run)
CASES = [(2, 5, 10), (8, 5, 10), (16, 5, 10), (130, 6, 37)]


def make(N, M, E, seeds=SEEDS, hyper=HYPER, **kw):
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    cls = IA2CRunsMany if N > 8 else IA2CRuns
    return cls(E, seeds, n_agents=N, n_models=M, **{k: v[:len(seeds)] for k, v in (hyper or {}).items()}, **kw)


def buffers(batch):
    torch.cuda.synchronize()
    return {k: h(getattr(batch, k)) for k in STATE}


def differing(pa, pb):
    """The buffers whose bytes differ, each with whether its values are equal (a sign of zero would differ only in bytes)."""
    return [(k, np.array_equal(pa[k], pb[k])) for k in STATE if pa[k].tobytes() != pb[k].tobytes()]


def hyper_arrays(batch):
    rows = [batch.run_hyper(r) for r in range(batch.R)]
    return {k: np.array([x[k] for x in rows], dtype=np.float32 if k in ("gamma", "beta") else np.float64)
            for k in ("lr_actor", "lr_critic", "gamma", "beta")}


def oracle_generation(batch, ring_rows, pre, pre_hyper, q, seed, g, mask=7, factors=(0.8, 1.2)):
    return P.generation(ring_rows, pre_hyper, {k: pre[k] for k in P.COPIED}, q, mask, factors, seed, g)


def assert_log_equals(log, g_index, olog):
    for k, dt in LOG:
        got = log[k][g_index]
        assert got.dtype == dt and got.tobytes() == np.asarray(olog[k], dtype=dt).tobytes(), (k, got, olog[k])


def standalone_from(batch, r):
    """A standalone trainer holding run r as it is now: run_state_dict(r) and run_hyper(r), both taken now."""
    from ia2c_b200.trainer import IA2CTrainer
    kw = dict(actor_kernel="columns") if batch.N > 8 else {}
    tr = IA2CTrainer(batch.E, n_agents=batch.N, n_models=batch.M, seed=batch.seeds[r], **batch.run_hyper(r), **kw)
    tr.load_state_dict(batch.run_state_dict(r))
    return tr


@pytest.mark.parametrize("N, M, E", CASES)
def test_generation_equals_the_oracle_and_runs_continue_alone(N, M, E):
    batch = make(N, M, E)
    batch.train_episodes(5)
    rows = batch.history()["return_sum"][-4:]
    pre, pre_hyper = buffers(batch), hyper_arrays(batch)
    q = 2   # floor(0.34 * 6): two donors, two recipients, two runs kept
    batch.exploit_explore(4, fraction=0.34, seed=7)
    log = batch.pbt_history()
    assert log["generation"].tolist() == [0] and log["episode"].tolist() == [5]
    new, new_hyper, olog = oracle_generation(batch, rows, pre, pre_hyper, q, seed=7, g=0)
    assert_log_equals(log, 0, olog)
    post = buffers(batch)
    for k in STATE:   # the recipients' copied rows equal the donors' pre-call bytes; every other byte is unchanged
        assert post[k].tobytes() == (new[k] if k in P.COPIED else pre[k]).tobytes(), k
    got_hyper = hyper_arrays(batch)
    for k in new_hyper:
        assert got_hyper[k].tobytes() == new_hyper[k].tobytes(), k
    assert np.array_equal(h(batch._hyper["gamma"]), new_hyper["gamma"])

    donor = log["donor"][0]
    recipient = int(np.flatnonzero(donor >= 0)[0])
    kept = [r for r in range(batch.R) if donor[r] < 0 and r not in donor]
    assert kept, donor
    picks = [recipient, int(donor[recipient]), kept[0]]
    alone = [standalone_from(batch, r) for r in picks]
    for _ in range(3):
        batch.train_episode()
        for tr in alone:
            tr.train_episode()
    torch.cuda.synchronize()
    for r, tr in zip(picks, alone):
        assert_run_equals(batch, r, tr)
        assert np.array_equal(h(batch.filter_action[r * N:(r + 1) * N]), h(tr.filter_action))


@pytest.mark.parametrize("N, M, E", [(2, 5, 10), (16, 5, 10)])
def test_q_zero_changes_no_training_byte(N, M, E):
    a, b = make(N, M, E, hyper=None), make(N, M, E, hyper=None)
    a.train_episodes(4), b.train_episodes(4)
    a.exploit_explore(4, fraction=0.1)   # floor(0.6) = 0 recipients
    log = a.pbt_history()
    assert (log["donor"] == -1).all() and sorted(log["rank"][0].tolist()) == list(range(a.R))
    for _ in range(3):
        a.train_episode(), b.train_episode()
    pa, pb = buffers(a), buffers(b)
    for k in STATE:
        assert pa[k].tobytes() == pb[k].tobytes(), k
    assert a.run_hyper(1) == b.run_hyper(1)


def _sweep(seed, pbt_seed):
    batch = make(2, 5, 10, seeds=[seed + i % 5 for i in range(16)], hyper=None, lr_actor=list(np.geomspace(1e-5, 1e-2, 16)))
    for _ in range(2):
        batch.train_episodes(4)
        batch.exploit_explore(4, fraction=0.25, seed=pbt_seed)
    batch.train_episode()
    return batch.pbt_history(), buffers(batch), hyper_arrays(batch)


def test_identical_batches_agree_and_the_pbt_seed_matters():
    la, ba, ha = _sweep(3, 10)
    lb, bb, hb = _sweep(3, 10)
    assert all(la[k].tobytes() == lb[k].tobytes() for k in la)
    assert all(ba[k].tobytes() == bb[k].tobytes() for k in ba)
    assert all(ha[k].tobytes() == hb[k].tobytes() for k in ha)
    lc, _, _ = _sweep(3, 11)
    assert np.array_equal(la["fitness"][0], lc["fitness"][0])   # the same runs up to the first generation
    assert not np.array_equal(la["donor"], lc["donor"])


@pytest.mark.parametrize("N, M, E", [(2, 5, 10), (16, 5, 10)])
def test_save_load_continues_through_a_generation(N, M, E, tmp_path):
    a = make(N, M, E)
    a.train_episodes(4)
    a.exploit_explore(4, fraction=0.34, seed=1)
    a.train_episodes(2)
    path = str(tmp_path / "pbt.pt")
    a.save(path)
    sd = a.state_dict()
    assert sd["pbt_generation"] == 1 and set(sd["hyper"]) == {"lr_actor", "lr_critic", "gamma", "beta"}
    b = make(N, M, E, hyper=None)   # built with other hyper-parameters: the checkpoint restores the runs' own
    b.load(path)
    a.pbt_history()
    for obj in (a, b):
        obj.train_episodes(4)
        obj.exploit_explore(4, fraction=0.34, seed=1)
        obj.train_episode()
    la, lb = a.pbt_history(), b.pbt_history()
    assert la["generation"].tolist() == lb["generation"].tolist() == [1]
    assert all(la[k].tobytes() == lb[k].tobytes() for k in la)
    pa, pb = buffers(a), buffers(b)
    assert differing(pa, pb) == []
    assert all(a.run_hyper(r) == b.run_hyper(r) for r in range(a.R))


@pytest.mark.parametrize("N, M, E", [(2, 5, 10), (16, 5, 10)])
def test_training_right_after_a_generation_needs_no_synchronisation(N, M, E):
    """The next episode's first kernels stage the agents' models before their PDL wait; a generation copies those models.
    A batch that trains straight after exploit_explore must equal a twin that synchronises in between, byte for byte."""
    def run(sync):
        batch = make(N, M, E)
        for _ in range(2):
            batch.train_episodes(4)
            batch.exploit_explore(4, fraction=0.34, seed=3)
            if sync:
                torch.cuda.synchronize()
            batch.train_episodes(2)
        return buffers(batch), batch.pbt_history()

    (pa, la), (pb, lb) = run(sync=False), run(sync=True)
    assert differing(pa, pb) == []
    assert all(la[k].tobytes() == lb[k].tobytes() for k in la) and (la["donor"] >= 0).any()


@pytest.mark.parametrize("hyper", [HYPER, None])
def test_a_checkpoint_from_before_any_generation_restores_the_built_hyper_parameters(hyper):
    a, twin = make(2, 5, 10, hyper=hyper), make(2, 5, 10, hyper=hyper)
    built = hyper_arrays(a)
    twin.train_episodes(2)
    sd = twin.state_dict()
    assert "pbt_generation" not in sd
    a.train_episodes(4)
    a.exploit_explore(4, fraction=0.34, seed=1)
    assert any(hyper_arrays(a)[k].tobytes() != built[k].tobytes() for k in built)
    a.load_state_dict(sd)
    assert a._pbt_generation == 0 and all(hyper_arrays(a)[k].tobytes() == built[k].tobytes() for k in built)
    with pytest.raises(ValueError, match="only 0 episodes"):
        a.exploit_explore(4)
    for obj in (a, twin):
        obj.train_episodes(4)
    pa, pt = buffers(a), buffers(twin)
    assert differing(pa, pt) == []


def test_a_checkpoint_without_a_generation_has_no_pbt_keys():
    a = make(2, 5, 10)
    a.train_episodes(2)
    assert "pbt_generation" not in a.state_dict() and "hyper" not in a.state_dict()


@pytest.mark.parametrize("N, M, E", [(2, 5, 10), (16, 5, 10)])
def test_two_launches_and_no_synchronisation(N, M, E, monkeypatch):
    batch = make(N, M, E)
    batch.train_episodes(8)
    torch.cuda.synchronize()

    def refuse(*a, **k):
        raise AssertionError("exploit_explore synchronised")

    before = _lib.launch_count()
    with monkeypatch.context() as m:
        m.setattr(torch.cuda.Stream, "synchronize", refuse)
        m.setattr(torch.cuda, "synchronize", refuse)
        m.setattr(torch.cuda.Event, "synchronize", refuse)
        batch.exploit_explore(8)
    assert _lib.launch_count() - before == 2
    batch.train_episodes(8)
    before = _lib.launch_count()
    batch.exploit_explore(8, fraction=0.0)
    assert _lib.launch_count() - before == 2
    assert batch.pbt_history()["generation"].tolist() == [0, 1]


@pytest.mark.parametrize("N, M, E", [(2, 5, 10), (16, 5, 10)])
def test_a_nan_fitness_ranks_last_and_is_replaced(N, M, E):
    batch = make(N, M, E)
    batch.train_episodes(4)
    rows = batch.history()["return_sum"]
    best = int(np.argmax(P.fitness(rows)))
    ring = batch._history
    ret = ring._dev[ring._off[0]:ring._off[1]].view(torch.float64).view(ring.capacity, batch.R)
    ret[(ring.head - 2) % ring.capacity, best] = float("nan")   # one of the window's rows
    rows[-2, best] = np.nan
    pre, pre_hyper = buffers(batch), hyper_arrays(batch)
    batch.exploit_explore(4, fraction=0.25, seed=2)
    log = batch.pbt_history()
    assert np.isnan(log["fitness"][0, best]) and log["rank"][0, best] == batch.R - 1 and log["donor"][0, best] >= 0
    new, new_hyper, olog = oracle_generation(batch, rows, pre, pre_hyper, 1, seed=2, g=0)
    assert_log_equals(log, 0, olog)
    post = buffers(batch)
    d = int(log["donor"][0, best])
    assert post["actor_params"][best * N:(best + 1) * N].tobytes() == pre["actor_params"][d * N:(d + 1) * N].tobytes()
    assert all(post[k].tobytes() == new[k].tobytes() for k in P.COPIED)
