"""CPU restatement of the per-episode statistics of ia2c_record_episode.  TEST INFRASTRUCTURE (see oracle/__init__.py).

  * ``fixed_order_sum`` — the return sum's fixed order (include/ia2c_b200.h): lane j of 256 adds x[j], x[j + 256],
    x[j + 512], ... in increasing order from +0.0, then a halving tree combines the lanes, s[j] += s[j + w] for j < w and
    w = 128, 64, ..., 1; the sum is s[0].  Every addition is one IEEE fp64 add (numpy's float64 +, round to nearest).
  * ``record`` — the statistics of one episode of R runs from its trajectory arrays, as ia2c_record_episode writes them.

Pinned against: ``math.fsum`` (the sum's value) and the golden reference tapes (tests/test_oracle_history.py).
"""
from __future__ import annotations

import numpy as np

LANES = 256
N_ACT = 3


def fixed_order_sum(x):
    """x f64[..., E] -> f64[...]: the sum over the last axis in the fixed order above."""
    x = np.asarray(x, dtype=np.float64)
    E = x.shape[-1]
    rows = -(-E // LANES)
    # padding adds +0.0 to a lane sum, which leaves it unchanged: a lane sum started at +0.0 is never -0.0
    pad = np.zeros(x.shape[:-1] + (rows * LANES,), dtype=np.float64)
    pad[..., :E] = x
    pad = pad.reshape(x.shape[:-1] + (rows, LANES))
    s = np.zeros(x.shape[:-1] + (LANES,), dtype=np.float64)
    for k in range(rows):
        s = s + pad[..., k, :]
    w = LANES // 2
    while w > 0:
        s = s[..., :w] + s[..., w:2 * w]
        w //= 2
    return s[..., 0]


def record(act, partner_true, partner_pred, ep_return, loss_out, R, E, N, T):
    """act, partner_true, partner_pred [>= T, R*E, N] (only steps 0..T-1 are read); ep_return f64[R*E]; loss_out f32[2, R*N].
    Returns return_sum f64[R], loss f32[2, R*N], action_counts u32[R*N, 3] and partner_hits u32[R*N]."""
    a = np.asarray(act)[:T].reshape(T, R, E, N)
    hit = (np.asarray(partner_pred)[:T] == np.asarray(partner_true)[:T]).reshape(T, R, E, N)
    counts = np.stack([(a == k).sum(axis=(0, 2)) for k in range(N_ACT)], axis=-1)         # [R, N, 3]
    return dict(return_sum=fixed_order_sum(np.asarray(ep_return, dtype=np.float64).reshape(R, E)),
                loss=np.array(loss_out, dtype=np.float32).reshape(2, R * N),
                action_counts=counts.reshape(R * N, N_ACT).astype(np.uint32),
                partner_hits=hit.sum(axis=(0, 2)).reshape(R * N).astype(np.uint32))
