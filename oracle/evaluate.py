"""CPU restatement of the frozen-policy evaluation (ia2c_evaluate).  TEST INFRASTRUCTURE (see oracle/__init__.py).

  * ``eval_uniforms`` — the evaluation sampler's Philox stream 4 (ia2c_b200/csrc/evaluate.cu): key = seed, counter =
    (e * ceil(N/4) + agent // 4, t | 4 << 16, episode) for env e within its run; agent i takes word i mod 4 as a 24-bit
    uniform, (w >> 8) * 2^-24, the conversion of oracle.philox.uniform_f32.
  * ``evaluate`` — K episodes of T steps in E envs of ONE run's actors, each from the reset state: the actors' softmax
    tabulated on the 9 observations, the inverse-CDF sampler (or the argmax) on the table row, Org-N stepped as
    oracle/loops.py steps it, and the fp64 return summed in step order.

Pinned against: oracle.loops.ia2c_rollout under one injected uniform tape (tests/test_oracle_eval.py), whose env is pinned to
the golden tapes.
"""
from __future__ import annotations

import numpy as np

from . import nets as NN
from . import philox
from .org import OrgBatchRef, make_obs

STREAM_EVAL = 4
N_ACT, N_FEAT = 3, 6

# the 9 observations, class c = 3 * prev_cls + cur_cls
OBS9 = make_obs(np.repeat(np.arange(3), 3), np.tile(np.arange(3), 3))


def eval_uniforms(seed, episode, t, E, N):
    """f32[E, N]: the uniforms of step t of evaluation episode `episode` for envs 0..E-1 of a run."""
    kq = (N + 3) // 4
    idx = np.arange(E, dtype=np.uint64)[:, None] * np.uint64(kq) + np.arange(kq, dtype=np.uint64)
    words = np.stack(philox.draw(seed, STREAM_EVAL, episode, t, idx), axis=-1).reshape(E, 4 * kq)[:, :N]
    return (words >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)


def policy_table(actors):
    """[N, 9, 3]: each actor's action distribution at the 9 observations."""
    return np.stack([NN.forward(a, OBS9, N_FEAT, N_ACT, softmax=True) for a in actors])


def evaluate(actors, E, K, T, max_episode_steps, u=None, greedy=False, seed=0, episode0=0, table=None):
    """actors [N, 105]; u f32[K, T, E, N] or None -> eval_uniforms(seed, episode0 + k, t, E, N).  ``table`` [N, 9, 3]
    replaces the tabulated forward (to drive the env with another implementation's table).  Returns returns f64[K, E],
    act int[K, T, E, N], reward f64[K, T, E], counts int[N, 3] and policy [N, 9, 3]."""
    actors = np.asarray(actors)
    N = actors.shape[0]
    P = policy_table(actors) if table is None else np.asarray(table)
    greedy_act = P.argmax(-1)                                   # [N, 9], ties -> lowest
    ACT = np.zeros((K, T, E, N), dtype=np.int64)
    REW = np.zeros((K, T, E), dtype=np.float64)
    RET = np.zeros((K, E), dtype=np.float64)
    agents = np.arange(N)
    for k in range(K):
        env = OrgBatchRef(E, max_episode_steps=max_episode_steps or None)
        env.reset()
        for t in range(T):
            c = 3 * env.prev_cls + env.cls                           # [E] observation class
            if greedy:
                a = greedy_act[agents[None, :], c[:, None]]
            else:
                uu = u[k, t] if u is not None else eval_uniforms(seed, episode0 + k, t, E, N)
                a = NN.sample_inverse_cdf(P[agents[None, :], c[:, None]], uu)
            if N == 2:
                _, r, _ = env.step_joint(a[:, 0] * N_ACT + a[:, 1])
            else:
                _, r, _ = env.step_agents(a)
            ACT[k, t], REW[k, t] = a, r
            RET[k] = RET[k] + r                                      # fp64, in step order
    counts = np.stack([(ACT == j).sum(axis=(0, 1, 2)) for j in range(N_ACT)], axis=-1)
    return dict(returns=RET, act=ACT, reward=REW, counts=counts, policy=P)
