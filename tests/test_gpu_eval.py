"""Frozen-policy evaluation on the GPU (ia2c_evaluate, IA2CTrainer.evaluate, IA2CRuns.evaluate): the policy table is the
training samplers' distribution, injected-tape episodes replay the training rollout's env byte for byte, the Philox
stream-4 counters follow the documented layout, greedy follows the argmax, a run of a batch equals the same actors alone,
and training state is untouched."""
import numpy as np
import pytest
import torch

from ia2c_b200 import _lib
from oracle import evaluate as EV
from tests.test_gpu_runs import BUFFERS, HYPER, SEEDS

pytestmark = pytest.mark.gpu


def h(t):
    return np.ascontiguousarray(t.detach().cpu().numpy())


def same_bytes(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def random_actors(rows, seed):
    return torch.from_numpy(np.random.RandomState(seed).normal(0.0, 0.6, size=(rows, _lib.ACTOR_P)).astype(np.float32)).cuda()


def evaluate(params, R, N, E, K, T, mes, greedy=False, seed=0, episode0=0, u=None):
    from ia2c_b200.evaluate import evaluate_actors
    return evaluate_actors(params, R, N, E, K, T, mes, greedy, seed, episode0, params.device, u_action=u)


@pytest.mark.parametrize("N", [2, 8, 64, 300])
def test_policy_table_is_the_samplers_distribution(N):
    params = random_actors(N, N)
    out = evaluate(params, 1, N, 3, 1, 5, 30)
    lib = _lib.load()
    x = torch.from_numpy(EV.OBS9).cuda()
    u = torch.zeros(9, device="cuda")
    act = torch.empty(9, dtype=torch.int64, device="cuda")
    probs = torch.empty(9, 3, device="cuda")
    for i in range(N):
        _lib.check(lib.ia2c_actor_sample(params[i].data_ptr(), x.data_ptr(), u.data_ptr(), act.data_ptr(), probs.data_ptr(),
                                         9, 6, 3, 0, 0, _lib.stream_ptr()), "ia2c_actor_sample")
        assert same_bytes(out["policy"][0, i], h(probs)), i
    ref = EV.policy_table(h(params).astype(np.float64))
    assert np.abs(out["policy"][0] - ref).max() < 1e-6


@pytest.mark.parametrize("N, M", [(2, 5), (2, 3), (3, 5), (8, 5), (16, 5), (64, 5), (130, 5)])
@pytest.mark.parametrize("E", [10, 37])
@pytest.mark.parametrize("mes", [30, 7])
def test_injected_episode_equals_the_training_rollout(N, M, E, mes):
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    T = 30
    tr = IA2CTrainer(E, n_agents=N, n_models=M, steps_per_episode=T, max_episode_steps=mes, init=reference_init(N, M, seed=N + E))
    U = np.random.RandomState(N * E + mes).rand(T + 1, E, N).astype(np.float32)
    tr.inject(u_action=U)
    tr.rollout()
    out = evaluate(tr.actor_params, 1, N, E, 1, T, mes, u=U[None, :T])
    assert same_bytes(out["returns"][0, 0], h(tr.ep_return))
    act = h(tr.act)[:T].astype(np.int64)
    assert np.array_equal(out["action_counts"][0], np.stack([(act == a).sum(axis=(0, 1)) for a in range(3)], -1).astype(np.uint64))


@pytest.mark.parametrize("N", [2, 5, 9, 64])
@pytest.mark.parametrize("R", [1, 3])
def test_philox_counters_follow_the_documented_layout(N, R):
    K, E, T, mes, seed = 3, 37, 30, 7, 0xDEADBEEF12
    params = random_actors(R * N, 7 * N + R)
    results = []
    for ep0 in (0, 4096):
        a = evaluate(params, R, N, E, K, T, mes, seed=seed, episode0=ep0)
        U = np.stack([[np.tile(EV.eval_uniforms(seed, ep0 + k, t, E, N), (R, 1)) for t in range(T)] for k in range(K)])
        b = evaluate(params, R, N, E, K, T, mes, u=U)
        for key in ("returns", "action_counts", "policy"):
            assert same_bytes(a[key], b[key]), (ep0, key)
        for r in range(R):   # and the env the kernel steps is the oracle's, bit for bit
            ref = EV.evaluate(np.zeros((N, 105)), E, K, T, mes, u=U[:, :, r * E:(r + 1) * E], table=a["policy"][r])
            assert same_bytes(a["returns"][r], ref["returns"]), r
            assert np.array_equal(a["action_counts"][r], ref["counts"].astype(np.uint64)), r
        results.append(a["returns"])
    assert not np.array_equal(results[0], results[1])
    assert not np.array_equal(evaluate(params, R, N, E, K, T, mes, seed=seed + 1)["returns"], results[0])


@pytest.mark.parametrize("N", [2, 5, 64])
def test_greedy_follows_the_argmax(N):
    from ia2c_b200.trainer import IA2CTrainer
    R, T, mes = 2, 40, 30
    params = random_actors(R * N, 3 * N)
    # run 1's agents 0 and 1: constant logits with exact ties (all three; actions 1 and 2)
    params[N:N + 2, 84:] = 0.0
    params[N + 1, 103:] = 1.0
    out = evaluate(params, R, N, 1, 1, T, mes, greedy=True)
    assert np.array_equal(out["greedy_actions"], out["policy"].argmax(-1))
    assert out["policy"][1, 0, 4, 0] == out["policy"][1, 0, 4, 1] == out["policy"][1, 0, 4, 2]
    assert (out["greedy_actions"][1, 0] == 0).all() and (out["greedy_actions"][1, 1] == 1).all()
    for r in range(R):
        ref = EV.evaluate(np.zeros((N, 105)), 1, 1, T, mes, greedy=True, table=out["policy"][r])
        assert same_bytes(out["returns"][r], ref["returns"]), r
        assert np.array_equal(out["action_counts"][r], ref["counts"].astype(np.uint64)), r
    with pytest.raises(ValueError, match="greedy"):
        evaluate(params, R, N, 2, 1, T, mes, greedy=True)
    tr = IA2CTrainer(4, n_agents=N)
    with pytest.raises(ValueError, match="greedy"):
        tr.evaluate(greedy=True, num_envs=4)
    g = tr.evaluate(greedy=True)
    assert g["returns"].shape == (1, 1) and g["greedy_actions"].shape == (N, 9)


@pytest.mark.parametrize("N", [2, 8])
def test_run_of_a_batch_equals_the_same_actors_alone(N):
    from ia2c_b200.runs import IA2CRuns
    from ia2c_b200.trainer import IA2CTrainer
    E = 10
    batch = IA2CRuns(E, SEEDS, n_agents=N, **HYPER)
    for _ in range(3):
        batch.train_episode()
    modes = (dict(episodes=2, seed=9, first_episode=4), dict(num_envs=33, episodes=1, seed=2), dict(greedy=True))
    results = [batch.evaluate(**kw) for kw in modes]
    for r, s in enumerate(SEEDS):
        tr = IA2CTrainer(E, n_agents=N, seed=s, **{k: v[r] for k, v in HYPER.items()})
        tr.load_state_dict(batch.run_state_dict(r))
        for kw, b in zip(modes, results):
            alone = tr.evaluate(**kw)
            assert set(alone) == set(b)
            for key, v in alone.items():
                assert same_bytes(b[key][r], v), (r, kw, key)


def _trainer_state(tr):
    return {name: h(getattr(tr, name)) for name in BUFFERS}


@pytest.mark.parametrize("N", [3, 16])
def test_evaluation_leaves_a_trainer_untouched(N):
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    a, b = (IA2CTrainer(37, n_agents=N, seed=4, init=reference_init(N, 5, seed=4)) for _ in range(2))
    for _ in range(3):
        a.train_episode()
        b.train_episode()
    a.evaluate(episodes=2, seed=1)
    a.evaluate(greedy=True)
    for _ in range(3):
        a.train_episode()
        b.train_episode()
    torch.cuda.synchronize()
    sa, sb = _trainer_state(a), _trainer_state(b)
    for name in sa:
        assert same_bytes(sa[name], sb[name]), name
    assert a.episode == b.episode == 6


def test_evaluation_leaves_a_batch_untouched():
    from ia2c_b200.runs import IA2CRuns
    a, b = (IA2CRuns(10, SEEDS, **HYPER) for _ in range(2))
    for _ in range(3):
        a.train_episode()
        b.train_episode()
    a.evaluate(episodes=3, num_envs=64)
    a.evaluate(greedy=True)
    for _ in range(3):
        a.train_episode()
        b.train_episode()
    torch.cuda.synchronize()
    sa, sb = _trainer_state(a), _trainer_state(b)
    for name in sa:
        assert same_bytes(sa[name], sb[name]), name


@pytest.mark.parametrize("N, greedy", [(2, False), (8, False), (64, False), (1023, False), (5, True)])
def test_deterministic_in_two_launches(N, greedy):
    R = 2 if N < 1023 else 1
    E, K = (1, 1) if greedy else (19, 2)
    params = random_actors(R * N, N)
    before = _lib.launch_count()
    a = evaluate(params, R, N, E, K, 30, 7, greedy=greedy, seed=3)
    assert _lib.launch_count() - before == 2
    b = evaluate(params, R, N, E, K, 30, 7, greedy=greedy, seed=3)
    for key in a:
        assert same_bytes(a[key], b[key]), key
    assert int(a["action_counts"].sum()) == R * N * E * K * 30
