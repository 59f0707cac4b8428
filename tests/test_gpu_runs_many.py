"""A batch of independent Org-N runs (IA2CRunsMany, ia2c_train_episode_runs_many, 9 <= N <= 256) against the same runs trained
alone: every run's slice of every buffer must equal a standalone IA2CTrainer(actor_kernel="columns") byte for byte."""
import numpy as np
import pytest
import torch

from ia2c_b200 import _lib
from tests.test_gpu_runs import BUFFERS, HYPER, SEEDS, assert_run_equals, h

pytestmark = pytest.mark.gpu


def standalone(E, seed, N, M, r=None, hyper=None, **kw):
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    hp = {k: (v[r] if r is not None else v) for k, v in (hyper or {}).items()}
    return IA2CTrainer(E, n_agents=N, n_models=M, seed=seed, init=reference_init(N, M, seed=seed), actor_kernel="columns", **hp, **kw)


# (9, 2, 600): two belief blocks per run; (130, 6, 37): two belief blocks per run, the last one partial; max_episode_steps = 12
# < T = 30 makes same-step autoresets happen inside the episode
@pytest.mark.parametrize("N, M, E, max_steps", [(9, 5, 37, 30), (9, 2, 600, 12), (16, 3, 10, 30), (33, 5, 37, 12), (64, 4, 7, 30),
                                                (130, 6, 37, 30), (256, 5, 10, 12)])
def test_batch_equals_standalone_columns_runs(N, M, E, max_steps):
    from ia2c_b200.runs import IA2CRunsMany
    batch = IA2CRunsMany(E, SEEDS, n_agents=N, n_models=M, max_episode_steps=max_steps, **HYPER)
    alone = [standalone(E, s, N, M, r, HYPER, max_episode_steps=max_steps) for r, s in enumerate(SEEDS)]
    for _ in range(4):
        batch.train_episode()
        for tr in alone:
            tr.train_episode()
    torch.cuda.synchronize()
    for r, tr in enumerate(alone):
        assert_run_equals(batch, r, tr)
    assert int(h(batch.actor_step).min()) == 4 and int(h(batch.critic_step).max()) == 4
    if max_steps < 30:
        assert int(h(batch.env_elapsed).max()) < max_steps


def test_single_run_stats_equal_standalone():
    from ia2c_b200.runs import IA2CRunsMany
    batch = IA2CRunsMany(64, [7], n_agents=12, n_models=5)
    tr = standalone(64, 7, 12, 5)
    for _ in range(4):
        s_batch = batch.train_episode(sync_stats=True)
        s_alone = tr.train_episode(sync_stats=True)
    assert_run_equals(batch, 0, tr)
    for k in ("critic_loss", "actor_loss", "ep_return", "critic_loss_window", "actor_loss_window", "mean_return"):
        assert np.array_equal(np.asarray(s_batch[k])[0], np.asarray(s_alone[k])), k


def test_run_state_dict_continues_alone():
    from ia2c_b200.runs import IA2CRunsMany
    from ia2c_b200.trainer import IA2CTrainer
    N, M, E = 130, 5, 37
    batch = IA2CRunsMany(E, SEEDS, n_agents=N, n_models=M, **HYPER)
    for _ in range(2):
        batch.train_episode(sync_stats=True)
    r = 1
    tr = IA2CTrainer(E, n_agents=N, n_models=M, seed=SEEDS[r], actor_kernel="columns", **{k: v[r] for k, v in HYPER.items()})
    tr.load_state_dict(batch.run_state_dict(r))
    for _ in range(3):
        s_batch = batch.train_episode(sync_stats=True)
        s_alone = tr.train_episode(sync_stats=True)
    assert_run_equals(batch, r, tr)
    assert np.array_equal(s_batch["mean_return"][r], s_alone["mean_return"])
    assert np.array_equal(s_batch["actor_loss_window"][r], s_alone["actor_loss_window"])


def test_batch_checkpoint_resumes_bit_identically(tmp_path):
    from ia2c_b200.runs import IA2CRunsMany
    a = IA2CRunsMany(10, SEEDS, n_agents=20, n_models=4, **HYPER)
    for _ in range(2):
        a.train_episode(sync_stats=True)
    a.save(tmp_path / "batch.pt")
    b = IA2CRunsMany(10, [0, 0, 0, 0], n_agents=20, n_models=4, **HYPER)   # seeds, parameters and state come from the checkpoint
    b.load(tmp_path / "batch.pt")
    for _ in range(3):
        sa, sb = a.train_episode(sync_stats=True), b.train_episode(sync_stats=True)
    torch.cuda.synchronize()
    for name in BUFFERS:
        assert np.array_equal(h(getattr(a, name)), h(getattr(b, name))), name
    for k in ("critic_loss_window", "actor_loss_window", "mean_return"):
        assert np.array_equal(sa[k], sb[k]), k


def test_deterministic():
    from ia2c_b200.runs import IA2CRunsMany
    a, b = (IA2CRunsMany(23, [5, 6, 7], n_agents=40, n_models=5, gamma=[0.9, 0.8, 0.7]) for _ in range(2))
    for _ in range(3):
        a.train_episode()
        b.train_episode()
    torch.cuda.synchronize()
    for name in BUFFERS:
        assert np.array_equal(h(getattr(a, name)).view(np.uint8), h(getattr(b, name)).view(np.uint8)), name


@pytest.mark.parametrize("R", [1, 8])
def test_six_launches_per_episode(R):
    from ia2c_b200.runs import IA2CRunsMany
    batch = IA2CRunsMany(10, list(range(R)), n_agents=16)
    batch.train_episode()
    before = _lib.launch_count()
    batch.train_episode()
    batch.train_episode()
    assert _lib.launch_count() - before == 12


def test_evaluate_equals_standalone_trainers():
    from ia2c_b200.runs import IA2CRunsMany
    from ia2c_b200.trainer import IA2CTrainer
    N, M, E = 16, 5, 10
    batch = IA2CRunsMany(E, SEEDS, n_agents=N, n_models=M, **HYPER)
    for _ in range(3):
        batch.train_episode()
    res = batch.evaluate(episodes=3, num_envs=17, seed=99)
    for r in range(len(SEEDS)):
        tr = IA2CTrainer(E, n_agents=N, n_models=M, seed=SEEDS[r], actor_kernel="columns")
        tr.load_state_dict(batch.run_state_dict(r))
        alone = tr.evaluate(episodes=3, num_envs=17, seed=99)
        for k in ("returns", "mean_return", "action_counts", "policy"):
            assert np.array_equal(np.asarray(res[k])[r], np.asarray(alone[k])), (r, k)
