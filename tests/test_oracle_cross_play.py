"""The oracle's cross-play restatement (oracle.cross_play.evaluate_lineups, lineup_stats): identity lineups are each run's
evaluation, permuted and duplicated lineups are the evaluation of the gathered actors, and the fixed-order statistics are the
mean and (ddof 0) variance."""
import numpy as np
import pytest

from oracle import cross_play as XP
from oracle import evaluate as EV


def _pool(nets, seed):
    return np.random.RandomState(seed).normal(0.0, 0.6, size=(nets, 105))


def _same(a, b):
    return a.shape == b.shape and np.array_equal(a, b)


@pytest.mark.parametrize("N", [2, 5])
def test_identity_lineups_are_each_runs_evaluation(N):
    R, E, K, T, mes = 3, 6, 2, 12, 7
    pool = _pool(R * N, N)
    out = XP.evaluate_lineups(pool, np.arange(R * N).reshape(R, N), E, K, T, mes, seed=4, episode0=2)
    for r in range(R):
        ref = EV.evaluate(pool[r * N:(r + 1) * N], E, K, T, mes, seed=4, episode0=2)
        for key in ("returns", "act", "counts", "policy"):
            assert _same(out[r][key], ref[key]), (r, key)


@pytest.mark.parametrize("greedy", [False, True])
def test_permuted_and_duplicated_lineups_are_the_gathered_actors(greedy):
    N, nets, E, K, T, mes = 4, 10, 5, 2, 15, 9
    if greedy:
        E = K = 1
    pool = _pool(nets, 7)
    lineups = np.array([[3, 2, 1, 0], [5, 5, 5, 5], [9, 0, 9, 1]])
    P = len(lineups)
    u = None if greedy else np.random.RandomState(1).rand(K, T, P * E, N).astype(np.float32)
    out = XP.evaluate_lineups(pool, lineups, E, K, T, mes, u=u, greedy=greedy)
    for p, rows in enumerate(lineups):
        ref = EV.evaluate(pool[rows], E, K, T, mes, u=None if u is None else u[:, :, p * E:(p + 1) * E], greedy=greedy)
        for key in ("returns", "counts"):
            assert _same(out[p][key], ref[key]), (p, key)
    assert _same(out[1]["policy"], np.repeat(EV.policy_table(pool[5:6]), N, axis=0))


@pytest.mark.parametrize("shape", [(1, 1, 1), (4, 16, 10), (2, 3, 300), (3, 1, 257)])
def test_lineup_stats_are_the_mean_and_variance(shape):
    x = np.random.RandomState(sum(shape)).normal(5.0, 40.0, size=shape)
    s, m2 = XP.lineup_stats(x)
    flat = x.reshape(shape[0], -1)
    n = flat.shape[1]
    assert np.allclose(s / n, flat.mean(1), rtol=1e-12, atol=0)
    assert np.allclose(np.sqrt(m2 / n), flat.std(1), rtol=1e-12, atol=1e-12)


def test_lineup_stats_follow_the_documented_order():
    """Lane j of 256 adds items j, j + 256, ... from +0.0, then the halving tree: restated with Python float adds."""
    x = np.random.RandomState(5).normal(0.0, 1e3, size=(2, 3, 300))
    s, m2 = XP.lineup_stats(x)
    for p in range(2):
        items = [float(v) for v in x[p].reshape(-1)]
        n = len(items)

        def tree(vals):
            lanes = [0.0] * 256
            for j in range(n):
                lanes[j % 256] += vals[j]
            w = 128
            while w:
                lanes = [lanes[j] + lanes[j + w] for j in range(w)]
                w //= 2
            return lanes[0]

        total = tree(items)
        mean = total / n
        assert s[p] == total
        assert m2[p] == tree([(v - mean) * (v - mean) for v in items])
