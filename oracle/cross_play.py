"""CPU restatement of cross-play (ia2c_evaluate_lineups).  TEST INFRASTRUCTURE (see oracle/__init__.py).

  * ``evaluate_lineups`` — lineup p is oracle.evaluate.evaluate on the pool rows lineups[p], its table gathered from the
    pool's table, its uniforms the tape's columns of lineup p (or stream 4 with the env index within the lineup).
  * ``lineup_stats`` — the fixed-order return_sum and return_m2 of each lineup's returns (include/ia2c_b200.h).

Pinned against: oracle.evaluate.evaluate per run and on the gathered actors, and numpy's mean / std
(tests/test_oracle_cross_play.py).
"""
from __future__ import annotations

import numpy as np

from .evaluate import evaluate, policy_table
from .history import fixed_order_sum


def evaluate_lineups(pool, lineups, E, K, T, max_episode_steps, u=None, greedy=False, seed=0, episode0=0, table=None):
    """pool [nets, 105], lineups int[P, N]; u f32[K, T, P*E, N] or None (Philox, the same numbers for every lineup).  ``table``
    [nets, 9, 3] replaces the pool's tabulated forward.  Returns one ``evaluate`` result per lineup."""
    pool, lineups = np.asarray(pool), np.asarray(lineups)
    tab = policy_table(pool) if table is None else np.asarray(table)
    out = []
    for p, rows in enumerate(lineups):
        up = u[:, :, p * E:(p + 1) * E] if u is not None else None
        out.append(evaluate(pool[rows], E, K, T, max_episode_steps, u=up, greedy=greedy, seed=seed, episode0=episode0,
                            table=tab[rows]))
    return out


def lineup_stats(returns):
    """returns f64[P, K, E] -> (return_sum, return_m2) f64[P]: over the n = K * E items of each lineup in row-major order, the
    fixed-order sum (oracle.history.fixed_order_sum: 256 lanes, then the halving tree), mean = sum / n (one IEEE divide), and
    the same fixed-order sum of (x - mean) * (x - mean), one subtract and one multiply per item."""
    x = np.asarray(returns, dtype=np.float64)
    x = x.reshape(x.shape[0], -1)
    s = fixed_order_sum(x)
    mean = s / np.float64(x.shape[1])
    dev = x - mean[:, None]
    return s, fixed_order_sum(dev * dev)
