"""Oracle pin of the frozen-policy evaluation (oracle/evaluate.py): under one injected uniform tape it plays exactly the
actions, rewards and step-order returns of the training rollout's oracle (oracle.loops.ia2c_rollout, pinned to the golden
tapes), autoresets inside an episode included; its Philox stream-4 uniforms follow the documented counter layout."""
import numpy as np
import pytest

from oracle import evaluate as EV
from oracle import loops as L
from oracle import philox as PX


def actors(N, seed):
    return np.random.RandomState(seed).normal(0.0, 0.6, size=(N, 105)).astype(np.float32)


@pytest.mark.parametrize("N", [2, 3, 9])
@pytest.mark.parametrize("T, mes", [(12, 30), (12, 5), (20, 7)])
def test_evaluation_replays_the_training_rollout(N, T, mes):
    E, M = 11, 5
    rng = np.random.RandomState(100 * N + T + mes)
    act = actors(N, N + mes)
    st = L.IA2CState(actor=act, critic=np.zeros((N, 147), np.float32), filter_action=rng.dirichlet(np.ones(3), size=(N, M)),
                     T=T, max_episode_steps=mes)
    u = rng.rand(T + 1, E, N).astype(np.float32)
    traj = L.ia2c_rollout(st, E, u_act=u, u_belief=rng.rand(T + 1, E, N, N - 1))
    ev = EV.evaluate(act, E, 1, T, mes, u=u[None, :T])
    assert np.array_equal(ev["act"][0], traj["act"][:T])
    assert np.array_equal(ev["reward"][0], traj["reward"])              # fp64 bit-exact
    ret = np.zeros(E)
    for t in range(T):
        ret = ret + traj["reward"][t]
    assert np.array_equal(ev["returns"][0], ret)
    assert np.array_equal(ev["counts"], np.stack([(traj["act"][:T] == a).sum(axis=(0, 1)) for a in range(3)], -1))
    if mes < T:   # the episode crosses the time limit: every env is back at the reset observation after step mes - 1
        assert np.array_equal(traj["obs"][mes], np.tile([0, 1, 0, 0, 1, 0], (E, 1)).astype(np.float32))


def test_policy_table_is_the_forward_on_the_nine_observations():
    act = actors(4, 1)
    P = EV.policy_table(act)
    for c in range(9):
        x = np.zeros(6, np.float32)
        x[c // 3], x[3 + c % 3] = 1.0, 1.0
        for i in range(4):
            assert np.allclose(P[i, c], L.NN.forward(act[i], x, 6, 3, softmax=True)[0], rtol=0, atol=1e-7)
    assert np.allclose(P.sum(-1), 1.0, atol=1e-6)


@pytest.mark.parametrize("N", [2, 5, 9])
def test_eval_uniforms_follow_the_counter_layout(N):
    seed, ep, t, E = 0x1234_5678_9ABC, 7, 3, 6
    u = EV.eval_uniforms(seed, ep, t, E, N)
    assert u.shape == (E, N) and u.dtype == np.float32
    kq = (N + 3) // 4
    for e in range(E):
        for i in range(N):
            words = PX.draw(seed, EV.STREAM_EVAL, ep, t, np.array([e * kq + i // 4], dtype=np.uint64))
            w = np.uint32(words[i % 4][0])
            assert u[e, i] == np.float32(int(w) >> 8) * np.float32(2.0 ** -24)
            if i % 4 == 0:   # word .x: the conversion of the training sampler
                assert u[e, i] == PX.uniform_f32(seed, EV.STREAM_EVAL, ep, t, np.array([e * kq + i // 4], dtype=np.uint64))[0]
    assert not np.array_equal(u, EV.eval_uniforms(seed, ep + 1, t, E, N))


def test_greedy_follows_the_argmax_and_sampling_is_reproducible():
    act = actors(3, 5)
    g = EV.evaluate(act, 1, 1, 25, 30, greedy=True)
    P = EV.policy_table(act)
    assert np.array_equal(g["act"][0, 0, 0], P[:, 4].argmax(-1))        # step 0: reset observation, class 3 * 1 + 1
    a = EV.evaluate(act, 4, 2, 25, 7, seed=3, episode0=10)
    b = EV.evaluate(act, 4, 2, 25, 7, u=np.stack([[EV.eval_uniforms(3, 10 + k, t, 4, 3) for t in range(25)] for k in range(2)]))
    assert np.array_equal(a["returns"], b["returns"]) and np.array_equal(a["act"], b["act"])
