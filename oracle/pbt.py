"""CPU restatement of one population-based-training generation (ia2c_pbt_step).  TEST INFRASTRUCTURE (see oracle/__init__.py).

  * ``fitness`` — the fp64 sum of each run's ring rows, oldest first, from +0.0 (numpy's float64 +, round to nearest).
  * ``rank_order`` — runs sorted by fitness, higher first, NaN below every non-NaN value, ties to the lower run index.
  * ``donor_ranks`` — stream-5 Philox words of each recipient (``oracle.philox.draw``): donor rank ((x >> 8) * q) >> 24.
  * ``perturb`` — lr: one fp64 multiply; beta: the f32 value widened to f64, one fp64 multiply, rounded to f32.
  * ``generation`` — the whole step: the new per-net state, the new hyper-parameters and the log row.

Pinned against: the definitions in include/ia2c_b200.h and the device log (tests/test_gpu_pbt.py).
"""
from __future__ import annotations

import numpy as np

from oracle import philox

STREAM_PBT = 5
LR_ACTOR, LR_CRITIC, BETA = 1, 2, 4
# the per-net buffers a recipient copies from its donor
COPIED = ("actor_params", "critic_params", "actor_m", "actor_v", "critic_m", "critic_v", "actor_step", "critic_step",
          "actor_grad_accum", "filter_action")


def fitness(ring_rows):
    """ring_rows f64[window, R], oldest first -> f64[R]."""
    rows = np.asarray(ring_rows, dtype=np.float64)
    f = np.zeros(rows.shape[1], dtype=np.float64)
    for row in rows:
        f = f + row
    return f


def rank_order(fit):
    """-> (order i32[R] with order[rank] = run, rank i32[R])."""
    fit = np.asarray(fit, dtype=np.float64)
    nan = np.isnan(fit)
    key = [(bool(nan[r]), 0.0 if nan[r] else -float(fit[r]), r) for r in range(fit.shape[0])]
    order = np.array(sorted(range(fit.shape[0]), key=lambda r: key[r]), dtype=np.int32)
    rank = np.empty_like(order)
    rank[order] = np.arange(order.shape[0], dtype=np.int32)
    return order, rank


def words(seed, g, runs):
    """The stream-5 Philox words (x, y, z, w) of the given recipient runs at generation g, each u32[len(runs)]."""
    return philox.draw(seed, STREAM_PBT, g, 0, np.asarray(runs, dtype=np.uint64))


def donor_ranks(x, q):
    """Word x (u32) -> donor rank in [0, q): ((x >> 8) * q) >> 24 in integer arithmetic."""
    return ((np.asarray(x, dtype=np.uint64) >> np.uint64(8)) * np.uint64(q) >> np.uint64(24)).astype(np.int64)


def perturb_lr(lr, word, factors):
    return np.float64(lr) * np.float64(factors[1] if int(word) >> 31 else factors[0])


def perturb_beta(beta, word, factors):
    return np.float32(np.float64(np.float32(beta)) * np.float64(factors[1] if int(word) >> 31 else factors[0]))


def generation(ring_rows, hyper, state, q, mask, factors, seed, g):
    """One generation.  ring_rows f64[window, R] oldest first; hyper: lr_actor, lr_critic f64[R], gamma, beta f32[R];
    state: the COPIED buffers with R*N rows on axis 0 (others are returned as given); q recipients; mask of LR_ACTOR,
    LR_CRITIC, BETA; factors (for a clear, a set top bit); seed and g key the draws.
    Returns (new state, new hyper, log) with log = fitness, rank, donor (-1: kept) and the four hyper-parameters after."""
    fit = fitness(ring_rows)
    R = fit.shape[0]
    assert 0 <= 2 * q <= R
    order, rank = rank_order(fit)
    new_hyper = {k: np.array(hyper[k], dtype=np.float64 if k.startswith("lr") else np.float32).copy()
                 for k in ("lr_actor", "lr_critic", "gamma", "beta")}
    new_state = {k: np.array(v, copy=True) for k, v in state.items()}
    donor = np.full(R, -1, dtype=np.int32)
    recipients = order[R - q:]
    if q:
        x, y, z, w = words(seed, g, recipients)
        picks = order[donor_ranks(x, q)]
        for j, (v, d) in enumerate(zip(recipients.tolist(), picks.tolist())):
            donor[v] = d
            lra, lrc = np.float64(hyper["lr_actor"][d]), np.float64(hyper["lr_critic"][d])
            beta, gamma = np.float32(hyper["beta"][d]), np.float32(hyper["gamma"][d])
            if mask & LR_ACTOR:
                lra = perturb_lr(lra, y[j], factors)
            if mask & LR_CRITIC:
                lrc = perturb_lr(lrc, z[j], factors)
            if mask & BETA:
                beta = perturb_beta(beta, w[j], factors)
            new_hyper["lr_actor"][v], new_hyper["lr_critic"][v] = lra, lrc
            new_hyper["gamma"][v], new_hyper["beta"][v] = gamma, beta
            for k in COPIED:
                if k in state:
                    n = state[k].shape[0] // R
                    new_state[k][v * n:(v + 1) * n] = np.asarray(state[k])[d * n:(d + 1) * n]
    log = dict(fitness=fit, rank=rank, donor=donor, **{k: new_hyper[k].copy() for k in new_hyper})
    return new_state, new_hyper, log
