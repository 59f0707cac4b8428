"""CPU restatement of frozen partners per env (ia2c_train_episode_env_partners).  TEST INFRASTRUCTURE (see oracle/__init__.py).

  * ``env_teams``  — the stream-7 Philox block of env e of a run keyed by ``seed`` before ``episode`` (``oracle.philox.draw``,
    index e, t 0): team ((x * Q) >> 32).
  * ``env_actors`` — the actor rows each env acts with: its team's pool rows in the partner seats (a repeated seat takes the
    lowest slot j); an env whose team or seats hold an entry out of range plays its own rows and logs -1.
  * ``env_probs``  — every agent's action probabilities along a trajectory's observations when env e acts with its own rows
    (envs grouped by distinct row, one forward per group, so the 4096-env case runs in seconds).  With the actions replayed,
    ``oracle.loops.ia2c_rollout`` does not depend on the actors except through its ``probs``: a per-env episode is that rollout
    with ``probs`` replaced by these.

Pinned against: the definitions in include/ia2c_b200.h and the device (tests/test_gpu_env_partners.py).
"""
from __future__ import annotations

import numpy as np

from oracle import nets as NN
from oracle import philox

STREAM_ENV_PARTNERS = 7
N_FEAT, N_ACT = 6, 3


def env_teams(seed, episode, E, Q):
    """The team (in [0, Q)) each of the E envs of a run keyed by ``seed`` draws before ``episode``: int64[E]."""
    x = philox.draw(seed, STREAM_ENV_PARTNERS, episode, 0, np.arange(E, dtype=np.uint64))[0]
    return ((x.astype(np.uint64) * np.uint64(Q)) >> np.uint64(32)).astype(np.int64)


def env_actors(actor, pool, seed, episode, E):
    """The actor rows every env of one run (``actor`` f32[N, 105], keyed by ``seed``) acts with in ``episode`` under ``pool`` =
    (rows, teams, seats): returns (actors f32[E, N, 105], log int32[E]: the drawn team or -1)."""
    rows, teams, seats = (np.asarray(x) for x in pool)
    actor = np.asarray(actor, dtype=np.float32)
    N = actor.shape[0]
    out = np.repeat(actor[None], E, axis=0)
    log = env_teams(seed, episode, E, teams.shape[0]).astype(np.int32)
    if (seats < 0).any() or (seats >= N).any():
        log[:] = -1
        return out, log
    bad = ((teams < 0) | (teams >= rows.shape[0])).any(1)
    log[bad[log]] = -1
    for j in range(len(seats) - 1, -1, -1):   # descending, so that the lowest slot of a repeated seat is written last
        ok = log >= 0
        out[ok, seats[j]] = rows[teams[log[ok], j]]
    return out, log


def env_probs(actors, obs, dtype=np.float64):
    """Action probabilities [T+1, E, N, 3] of agent i in env e at ``obs`` [T+1, E, 6] under ``actors`` [E, N, 105]."""
    T1, E = obs.shape[:2]
    N = actors.shape[1]
    out = np.zeros((T1, E, N, N_ACT), dtype=dtype)
    for i in range(N):
        rows, inv = np.unique(actors[:, i], axis=0, return_inverse=True)
        inv = inv.reshape(-1)
        for g in range(rows.shape[0]):
            sel = inv == g
            x = obs[:, sel].reshape(-1, N_FEAT)
            out[:, sel, i] = NN.forward(rows[g].astype(dtype), x, N_FEAT, N_ACT, softmax=True).reshape(T1, -1, N_ACT)
    return out
