"""Learning curves recorded on the GPU (ia2c_record_episode through train_episodes / history): each recorded row equals the
oracle's statistics of the episode's own trajectory byte for byte on every trainer path, training is byte-identical with and
without recording, a batch's run rows equal the standalone run's, the ring drains in order, and one launch is added per
recorded episode."""
import numpy as np
import pytest
import torch

from ia2c_b200 import _lib
from oracle import history as H
from tests.test_gpu_runs import HYPER, SEEDS, h
from tests.test_gpu_runs_many import standalone
from tests.test_oracle_loops import ia2c_state_from_golden, ia2c_tapes

pytestmark = pytest.mark.gpu


def trainer(E, N, M=5, **kw):
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    return IA2CTrainer(E, n_agents=N, n_models=M, init=reference_init(N, M, seed=E + N), **kw)


def snapshot(obj, R, E, N, T):
    """The oracle's record of the episode obj just trained, from its own buffers (synchronises)."""
    return H.record(h(obj.act), h(obj.partner_true), h(obj.partner_pred), h(obj.ep_return), h(obj.loss_out), R, E, N, T)


def assert_rows_equal_oracle(hist, recs, R, N, steps, squeeze):
    """hist: history() of len(recs) episodes of ``steps`` = T * E (step, env) pairs per run; recs: the oracle's records in
    order.  Byte-for-byte equality."""
    exp = dict(return_sum=np.stack([r["return_sum"] for r in recs]),
               critic_loss=np.stack([r["loss"][0].reshape(R, N) for r in recs]),
               actor_loss=np.stack([r["loss"][1].reshape(R, N) for r in recs]),
               action_counts=np.stack([r["action_counts"].reshape(R, N, 3) for r in recs]),
               partner_hits=np.stack([r["partner_hits"].reshape(R, N) for r in recs]))
    if squeeze:
        exp = {k: v[:, 0] for k, v in exp.items()}
    exp.update(partner_accuracy=exp.pop("partner_hits") / float(steps), action_freq=exp["action_counts"] / float(steps))
    assert hist["episode"].shape == (len(recs),)
    for k, v in exp.items():
        assert hist[k].shape == v.shape and hist[k].dtype == v.dtype and hist[k].tobytes() == v.tobytes(), k


@pytest.mark.parametrize("name", ["ia2c_E10.npz", "ia2c_E64.npz"])
def test_golden_replay(golden, name):
    g = golden(name)
    T, E = int(g["meta_T"]), int(g["meta_n_envs"])
    st = ia2c_state_from_golden(g)
    lr_c, lr_a, beta, gamma = g["meta_hyper"]
    from ia2c_b200.trainer import IA2CTrainer
    tr = IA2CTrainer(E, n_agents=2, n_models=5, init=(st.actor, st.critic, st.filter_action), lr_critic=lr_c, lr_actor=lr_a,
                     beta=beta, gamma=gamma, steps_per_episode=T)
    episodes, losses = int(g["meta_episodes"]), []
    for ep in range(episodes):
        sl, actions, u = ia2c_tapes(g, ep)
        tr.inject(actions=actions, u_belief=u)
        tr.train_episodes(1)
        losses.append(h(tr.loss_out))
    hist = tr.history()
    assert hist["episode"].tolist() == list(range(episodes))
    for ep in range(episodes):
        sl = slice(ep * (T + 1), (ep + 1) * (T + 1))
        a1, a2 = g["act1/sampled"][sl], g["act2/sampled"][sl]
        rec = H.record(np.stack([a1, a2], -1), np.stack([a2, a1], -1), np.stack([g["bf0/ap"][sl], g["bf1/ap"][sl]], -1),
                       g["reward_lst"][ep], losses[ep], 1, E, 2, T)
        assert hist["action_counts"][ep].tobytes() == rec["action_counts"].tobytes()
        assert np.array_equal(hist["partner_accuracy"][ep], rec["partner_hits"] / float(T * E))
        assert hist["return_sum"][ep].tobytes() == rec["return_sum"][0].tobytes()
        assert hist["critic_loss"][ep].tobytes() == losses[ep][0].tobytes()
        assert hist["actor_loss"][ep].tobytes() == losses[ep][1].tobytes()
        assert np.array_equal(hist["mean_return"][ep], rec["return_sum"][0] / E)


# every path that fills the trajectory: fused N <= 8 (M = 5, and N = 2 with M = 3; E = 600 wraps the 256 return lanes),
# whole-episode rollout + belief kernels (16, 64, 130; columns and pipe actor kernels), per-step kernels (N = 300 by default,
# and N = 16 with rollout_kernel / belief_kernel = "step")
@pytest.mark.parametrize("N, M, E, T, kw", [
    (2, 5, 600, 30, {}), (5, 5, 37, 30, {}), (2, 3, 37, 30, {}), (16, 5, 37, 30, {}),
    (64, 5, 7, 12, dict(actor_kernel="columns")), (64, 5, 7, 12, dict(actor_kernel="pipe")),
    (130, 5, 5, 8, dict(actor_kernel="columns")), (130, 5, 5, 8, dict(actor_kernel="pipe")), (300, 5, 3, 6, {}),
    (16, 5, 37, 30, dict(rollout_kernel="step")), (16, 5, 37, 30, dict(belief_kernel="step"))])
def test_every_trainer_path_against_the_oracle(N, M, E, T, kw):
    tr = trainer(E, N, M, steps_per_episode=T, max_episode_steps=T, seed=N, **kw)
    recs = []
    for _ in range(3):
        tr.train_episodes(1)
        recs.append(snapshot(tr, 1, E, N, T))
    hist = tr.history()
    assert hist["episode"].tolist() == [0, 1, 2]
    assert_rows_equal_oracle(hist, recs, 1, N, T * E, squeeze=True)
    assert hist["action_counts"].sum(-1).min() == T * E


def _ckpt_bytes(obj):
    torch.cuda.synchronize()
    from ia2c_b200.trainer import IA2CTrainer
    names = IA2CTrainer._CKPT_TENSORS + ("loss_out", "ep_return")
    return {k: h(getattr(obj, k)).tobytes() for k in names}


@pytest.mark.parametrize("kind", ["trainer", "runs", "runs_many"])
def test_training_is_untouched_by_recording(kind):
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany

    def make():
        if kind == "trainer":
            return trainer(64, 2, seed=5)
        if kind == "runs":
            return IA2CRuns(37, SEEDS, n_agents=3, **HYPER)
        return IA2CRunsMany(10, SEEDS[:2], n_agents=16, **{k: v[:2] for k, v in HYPER.items()})

    plain, rec = make(), make()
    rec.HISTORY_CAPACITY = 3   # drains inside the loop too
    for _ in range(5):
        plain.train_episode()
    rec.train_episodes(5)
    assert _ckpt_bytes(plain) == _ckpt_bytes(rec)
    assert plain.episode == rec.episode == 5
    assert rec.history()["episode"].tolist() == [0, 1, 2, 3, 4]
    assert rec.critic_losses == [] and rec.reward_lst == []   # recorded episodes stay out of the read_stats windows


@pytest.mark.parametrize("many, R", [(False, 4), (False, 1), (True, 2)])
def test_batch_rows_equal_standalone_history(many, R):
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    N, M, E = (16, 5, 10) if many else (2, 5, 37)
    seeds, hyper = SEEDS[:R], {k: v[:R] for k, v in HYPER.items()}
    batch = (IA2CRunsMany if many else IA2CRuns)(E, seeds, n_agents=N, n_models=M, **hyper)
    alone = [standalone(E, s, N, M, r, hyper) for r, s in enumerate(seeds)]
    batch.train_episodes(4)
    for tr in alone:
        tr.train_episodes(4)
    hb = batch.history()
    for r, tr in enumerate(alone):
        ha = tr.history()
        assert np.array_equal(hb["episode"], ha["episode"])
        for k in ("return_sum", "mean_return", "critic_loss", "actor_loss", "action_counts", "action_freq", "partner_accuracy"):
            assert hb[k][:, r].tobytes() == ha[k].tobytes(), (r, k)


def test_ring_wraps_and_drains_in_order():
    E, N, T = 37, 2, 30
    tr = trainer(E, N, seed=3)
    tr.HISTORY_CAPACITY = 2
    recs = []
    for k in range(7):
        if k == 3:   # unrecorded episodes in between are absent from the history
            tr.train_episode()
            tr.train_episode()
        tr.train_episodes(1)
        recs.append(snapshot(tr, 1, E, N, T))
    hist = tr.history()
    assert hist["episode"].tolist() == [0, 1, 2, 5, 6, 7, 8]
    assert_rows_equal_oracle(hist, recs, 1, N, T * E, squeeze=True)
    tr.train_episodes(3)
    again = tr.history()
    assert again["episode"].tolist() == [9, 10, 11]
    assert tr.history()["episode"].shape == (0,)
    assert tr._history.capacity == 2


def test_ring_wraps_inside_one_call():
    """train_episodes(n) with n well above the capacity drains itself; the rows equal those of a deep ring."""
    deep, shallow = trainer(64, 2, seed=9), trainer(64, 2, seed=9)
    shallow.HISTORY_CAPACITY = 3
    deep.train_episodes(11)
    shallow.train_episodes(11)
    a, b = deep.history(), shallow.history()
    assert all(a[k].tobytes() == b[k].tobytes() for k in a)


@pytest.mark.parametrize("kind, expected", [("fused", 5), ("runs_many", 7)])
def test_one_extra_launch_per_recorded_episode(kind, expected):
    from ia2c_b200.runs import IA2CRunsMany
    obj = trainer(64, 2) if kind == "fused" else IA2CRunsMany(10, SEEDS, n_agents=16)
    obj.train_episodes(1)
    torch.cuda.synchronize()
    before = _lib.launch_count()
    obj.train_episode()
    plain = _lib.launch_count() - before
    before = _lib.launch_count()
    obj.train_episodes(1)
    assert _lib.launch_count() - before == expected == plain + 1


def test_determinism():
    from ia2c_b200.runs import IA2CRuns
    a, b = (IA2CRuns(37, SEEDS, n_agents=5, **HYPER) for _ in range(2))
    a.train_episodes(6), b.train_episodes(6)
    ha, hb = a.history(), b.history()
    assert all(ha[k].tobytes() == hb[k].tobytes() for k in ha)
