"""CPU restatement of frozen-partner seating (ia2c_seat_partners).  TEST INFRASTRUCTURE (see oracle/__init__.py).

  * ``team`` — the stream-6 Philox block of (seed, episode) (``oracle.philox.draw``, index 0, t 0): team ((x * Q) >> 32).
  * ``seat`` — each run's drawn team copied into its partner seats' actor rows; a run whose team or seats hold an entry out of
    range keeps its rows and logs -1.

Pinned against: the definitions in include/ia2c_b200.h and the device (tests/test_gpu_partners.py).
"""
from __future__ import annotations

import numpy as np

from oracle import philox

STREAM_PARTNERS = 6


def words(seed, episode):
    """The stream-6 Philox words (x, y, z, w) a run keyed by ``seed`` draws before ``episode``."""
    return tuple(int(w[0]) for w in philox.draw(seed, STREAM_PARTNERS, episode, 0, np.zeros(1, dtype=np.uint64)))


def team(seed, episode, Q):
    """The team (in [0, Q)) a run keyed by ``seed`` plays in ``episode``."""
    return (words(seed, episode)[0] * int(Q)) >> 32


def seat(actor_params, pool, episode, seed):
    """``actor_params`` f32[R*N, 105] after seating ``pool`` = (rows f32[P, 105], teams int[Q, S], seats int[S]) before
    ``episode``; ``seed`` is one run's training seed (R = 1) or a sequence of R seeds.  Returns (new actor_params, log int32[R]:
    the drawn team or -1)."""
    rows, teams, seats = (np.asarray(x) for x in pool)
    seeds = [int(seed)] if np.ndim(seed) == 0 else [int(s) for s in seed]
    R = len(seeds)
    out = np.array(actor_params, dtype=np.float32, copy=True)
    N = out.shape[0] // R
    log = np.full(R, -1, dtype=np.int32)
    for r, s in enumerate(seeds):
        t = team(s, episode, teams.shape[0])
        picks = teams[t]
        if (picks < 0).any() or (picks >= rows.shape[0]).any() or (seats < 0).any() or (seats >= N).any():
            continue
        out[r * N + seats] = rows[picks]
        log[r] = t
    return out, log
