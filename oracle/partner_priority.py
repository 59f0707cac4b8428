"""CPU restatement of prioritized partners per env (ia2c_record_partner_returns, ia2c_prioritize_partners and the weighted
draw of ia2c_train_episode_env_partners_prioritized).  TEST INFRASTRUCTURE (see oracle/__init__.py).

  * ``fixed``       — a return's fixed-point value llrint(v * 2^20) (round half to even), or None where it is skipped.
  * ``accumulate``  — count / sum i64[R, Q] after the record of one episode's returns [R, E] and env-team log [R, E].
  * ``weights``     — W [R, Q] from count / sum, with power p and floor f, one Python float (IEEE fp64) operation at a time.
  * ``table``       — the prefix table C [R, Q + 1] of W; ``equal_table`` is the one before the first prioritize.
  * ``draw``        — the team of a stream-7 word x under a table row, the 128-bit product in Python integers.
  * ``env_teams``   — the teams of the E envs of a run keyed by ``seed`` before ``episode``, under its table row.

Pinned against: the definitions in include/ia2c_b200.h and the device (tests/test_gpu_partner_priority.py).
"""
from __future__ import annotations

import math

import numpy as np

from oracle import philox
from oracle.env_partners import STREAM_ENV_PARTNERS

FIX = 2.0 ** 20
LIMIT = 2.0 ** 62
UNIT = 1 << 24


def fixed(v):
    """llrint(v * 2^20) as a Python int, or None where the record skips the return (not finite, |v| * 2^20 >= 2^62)."""
    s = float(v) * FIX
    if not abs(s) < LIMIT:
        return None
    return int(np.rint(s))   # round half to even; s is exact (a power-of-two scaling), |s| < 2^62 converts exactly


def accumulate(count, total, ep_return, env_team):
    """Add one episode (``ep_return`` f64[R, E], ``env_team`` int[R, E]) to ``count`` / ``total`` i64[R, Q] (new arrays)."""
    count, total = np.array(count, dtype=np.int64), np.array(total, dtype=np.int64)
    Q = count.shape[1]
    for r, e in np.ndindex(*np.shape(env_team)):
        t, v = int(env_team[r][e]), fixed(ep_return[r][e])
        if t < 0 or t >= Q or v is None:
            continue
        count[r, t] += 1
        total[r, t] = np.int64(((int(total[r, t]) + v + (1 << 63)) % (1 << 64)) - (1 << 63))   # the device's wrapping add
    return count, total


def means(count, total):
    """m [R, Q] f64 as the weights see it: (sum * 2^-20) / count, NaN where count is 0."""
    out = np.full(np.shape(count), np.nan)
    for idx in np.ndindex(*np.shape(count)):
        n = int(count[idx])
        if n > 0:
            out[idx] = (float(int(total[idx])) * 2.0 ** -20) / float(n)
    return out


def weights(count, total, power, floor):
    """W [R, Q] i64 (include/ia2c_b200.h: weights)."""
    m = means(count, total)
    R, Q = m.shape
    W = np.full((R, Q), UNIT, dtype=np.int64)
    f = float(floor)
    for r in range(R):
        played = [float(x) for x in m[r] if not math.isnan(x)]
        if not played:
            continue
        hi, lo = max(played), min(played)
        if hi == lo:
            continue
        for q in range(Q):
            if math.isnan(m[r, q]):
                continue                                  # unplayed: w = 1
            x = (hi - float(m[r, q])) / (hi - lo)
            xp = 1.0
            for _ in range(int(power)):
                xp = xp * x
            w = f + (1.0 - f) * xp
            W[r, q] = min(UNIT, int(math.floor(w * UNIT)))
    return W


def table(W):
    """C [R, Q + 1] i64: C_0 = 0, C_{q+1} = C_q + W_q."""
    W = np.asarray(W, dtype=np.int64)
    return np.concatenate([np.zeros((W.shape[0], 1), dtype=np.int64), np.cumsum(W, axis=1)], axis=1)


def equal_table(R, Q):
    return table(np.full((R, Q), UNIT, dtype=np.int64))


def draw(x, row):
    """The team of word ``x`` under table row ``row`` (C_0 .. C_Q): y = (x * C_Q) >> 32, q with C_q <= y < C_{q+1}; -1 where
    C_Q = 0."""
    row = np.asarray(row, dtype=np.int64)
    total = int(row[-1])
    if total == 0:
        return -1
    y = (int(x) * total) >> 32   # the 128-bit product; y < C_Q <= 2^44 fits the table's integers
    return int(np.searchsorted(row, y, side="right")) - 1


def env_teams(seed, episode, E, row):
    """The teams int64[E] the E envs of a run keyed by ``seed`` draw before ``episode`` under its table row."""
    x = philox.draw(seed, STREAM_ENV_PARTNERS, episode, 0, np.arange(E, dtype=np.uint64))[0]
    return np.array([draw(v, row) for v in x], dtype=np.int64)
