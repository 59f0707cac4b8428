"""A batch of independent runs (IA2CRuns, ia2c_train_episode_runs) against the same runs trained alone: every run's slice of
every buffer must equal the standalone IA2CTrainer byte for byte."""
import numpy as np
import pytest
import torch

from ia2c_b200 import _lib

pytestmark = pytest.mark.gpu

# distinct per-run hyper-parameters: identical ones would hide a wrong run offset in the kernels' per-run reads
SEEDS = [11, 29, 3, 29]   # a repeated seed is allowed (sweeps that vary only the hyper-parameters)
HYPER = dict(lr_actor=[1e-4, 3e-4, 5e-5, 2e-3], lr_critic=[2e-4, 1e-3, 7e-5, 5e-4],
             beta=[1e-3, 1e-2, 0.0, 5e-2], gamma=[0.9, 0.99, 0.5, 0.75])
# every buffer the contract covers, under the names IA2CTrainer uses
BUFFERS = ("obs", "reward", "act", "partner_true", "partner_pred", "belief_records", "ep_return", "loss_out",
           "actor_grad", "critic_grad", "actor_params", "critic_params", "actor_m", "actor_v", "critic_m", "critic_v",
           "actor_step", "critic_step", "actor_grad_accum", "env_state", "env_hist", "env_cls", "env_elapsed")


def standalone(E, seed, N, M, r=None, hyper=None):
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    hp = {k: (v[r] if r is not None else v) for k, v in (hyper or {}).items()}
    return IA2CTrainer(E, n_agents=N, n_models=M, seed=seed, init=reference_init(N, M, seed=seed), **hp)


def h(t):
    return np.ascontiguousarray(t.detach().cpu().numpy())


def assert_run_equals(batch, r, tr):
    v = batch.run_view(r)
    for name in BUFFERS:
        a, b = h(v[name]), h(getattr(tr, name))
        assert a.shape == b.shape and a.dtype == b.dtype, (name, a.shape, b.shape)
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), f"run {r}: {name} differs"


@pytest.mark.parametrize("N, M", [(2, 5), (2, 3), (3, 5), (8, 5)])
@pytest.mark.parametrize("E", [10, 37])
def test_batch_equals_standalone_runs(E, N, M):
    from ia2c_b200.runs import IA2CRuns
    batch = IA2CRuns(E, SEEDS, n_agents=N, n_models=M, **HYPER)
    alone = [standalone(E, s, N, M, r, HYPER) for r, s in enumerate(SEEDS)]
    for _ in range(5):
        batch.train_episode()
        for tr in alone:
            tr.train_episode()
    torch.cuda.synchronize()
    for r, tr in enumerate(alone):
        assert_run_equals(batch, r, tr)
    assert int(h(batch.actor_step).min()) == 5 and int(h(batch.critic_step).max()) == 5


def test_single_run_equals_standalone():
    from ia2c_b200.runs import IA2CRuns
    batch = IA2CRuns(64, [7])
    tr = standalone(64, 7, 2, 5)
    for _ in range(4):
        s_batch = batch.train_episode(sync_stats=True)
        s_alone = tr.train_episode(sync_stats=True)
    assert_run_equals(batch, 0, tr)
    for k in ("critic_loss", "actor_loss", "ep_return", "critic_loss_window", "actor_loss_window", "mean_return"):
        assert np.array_equal(np.asarray(s_batch[k])[0], np.asarray(s_alone[k])), k


def test_scalar_hyper_parameters_broadcast():
    from ia2c_b200.runs import IA2CRuns
    seeds = [1, 2, 3]
    scalar = IA2CRuns(16, seeds, lr_actor=3e-4, gamma=0.8, beta=0.02, lr_critic=1e-3)
    listed = IA2CRuns(16, seeds, lr_actor=[3e-4] * 3, gamma=[0.8] * 3, beta=[0.02] * 3, lr_critic=[1e-3] * 3)
    for _ in range(3):
        scalar.train_episode()
        listed.train_episode()
    torch.cuda.synchronize()
    for name in BUFFERS:
        assert np.array_equal(h(getattr(scalar, name)), h(getattr(listed, name))), name
    tr = standalone(16, 2, 2, 5, hyper=dict(lr_actor=3e-4, gamma=0.8, beta=0.02, lr_critic=1e-3))
    for _ in range(3):
        tr.train_episode()
    assert_run_equals(scalar, 1, tr)


def test_run_state_dict_continues_alone(tmp_path):
    from ia2c_b200.runs import IA2CRuns
    from ia2c_b200.trainer import IA2CTrainer
    batch = IA2CRuns(37, SEEDS, **HYPER)
    for _ in range(3):
        batch.train_episode(sync_stats=True)
    r = 2
    tr = IA2CTrainer(37, seed=SEEDS[r], **{k: v[r] for k, v in HYPER.items()})
    tr.load_state_dict(batch.run_state_dict(r))
    for _ in range(3):
        s_batch = batch.train_episode(sync_stats=True)
        s_alone = tr.train_episode(sync_stats=True)
    assert_run_equals(batch, r, tr)
    assert np.array_equal(s_batch["mean_return"][r], s_alone["mean_return"])
    assert np.array_equal(s_batch["critic_loss_window"][r], s_alone["critic_loss_window"])


def test_batch_checkpoint_resumes_bit_identically(tmp_path):
    from ia2c_b200.runs import IA2CRuns
    a = IA2CRuns(10, SEEDS, n_agents=3, **HYPER)
    for _ in range(2):
        a.train_episode(sync_stats=True)
    a.save(tmp_path / "batch.pt")
    b = IA2CRuns(10, [0, 0, 0, 0], n_agents=3, **HYPER)   # seeds, parameters and state all come from the checkpoint
    b.load(tmp_path / "batch.pt")
    for _ in range(3):
        sa, sb = a.train_episode(sync_stats=True), b.train_episode(sync_stats=True)
    torch.cuda.synchronize()
    for name in BUFFERS:
        assert np.array_equal(h(getattr(a, name)), h(getattr(b, name))), name
    for k in ("critic_loss_window", "actor_loss_window", "mean_return"):
        assert np.array_equal(sa[k], sb[k]), k


def test_refusals():
    from ia2c_b200.runs import IA2CRuns
    with pytest.raises(ValueError):
        IA2CRuns(10, [1, 2], n_agents=9)
    with pytest.raises(ValueError):
        IA2CRuns(10, [1, 2], n_agents=3, n_models=3)
    with pytest.raises(ValueError):
        IA2CRuns(10, [1, 2], gamma=[0.9, 0.9, 0.9])
    with pytest.raises(ValueError):
        IA2CRuns(10, [1, 2], init=[None])
    with pytest.raises(ValueError):
        IA2CRuns(10, range(_lib.MAX_RUN_NETS // 8 + 1), n_agents=8)
    with pytest.raises(IndexError):
        IA2CRuns(10, [1, 2]).run_view(2)
