"""The oracle of prioritized partners per env (oracle/partner_priority.py) against the definitions in include/ia2c_b200.h:
the equal-weight draw is the uniform stream-7 draw, zero weights are never drawn, weighted draws follow W, the weight edge
cases, and the fixed-point rounding and skip rules of the recorded returns."""
import numpy as np
import pytest
from scipy import stats

from oracle import env_partners as EP
from oracle import partner_priority as PP
from oracle import philox

UNIT = 1 << 24


@pytest.mark.parametrize("Q", [1, 2, 3, 1000, 1 << 20])
def test_equal_weights_draw_the_uniform_team(Q):
    rng = np.random.default_rng(Q)
    xs = np.concatenate([rng.integers(0, 1 << 32, size=2000, dtype=np.uint64), [0, 1, (1 << 32) - 1, 1 << 31]]).astype(np.uint64)
    row = PP.equal_table(1, Q)[0]
    assert row[-1] == Q * UNIT
    for x in xs:
        assert PP.draw(int(x), row) == (int(x) * Q) >> 32
    assert np.array_equal(PP.env_teams(77, 3, 500, row), EP.env_teams(77, 3, 500, Q))


def test_zero_weight_teams_are_never_drawn():
    W = np.array([[0, UNIT, 0, 0, 5, 0, UNIT // 2, 0]], dtype=np.int64)
    row = PP.table(W)[0]
    x = philox.draw(5, 7, 0, 0, np.arange(20000, dtype=np.uint64))[0]
    teams = np.array([PP.draw(int(v), row) for v in x])
    assert set(teams.tolist()) <= {1, 4, 6}
    edges = [int(row[q]) for q in range(len(row))]   # a word landing exactly on each boundary
    for q in (1, 4, 6):
        x = -(-(edges[q] << 32) // int(row[-1]))      # the smallest x with y >= C_q
        assert PP.draw(x, row) == q
    assert PP.draw(123, PP.table(np.zeros((1, 4), dtype=np.int64))[0]) == -1


def test_weighted_draws_follow_the_weights():
    W = np.array([[UNIT, UNIT // 2, UNIT // 4, 3 * UNIT // 4, UNIT // 10, UNIT]], dtype=np.int64)
    row = PP.table(W)[0]
    x = np.concatenate([philox.draw(s, 7, 2, 0, np.arange(15000, dtype=np.uint64))[0] for s in (1, 2, 3, 4)])
    counts = np.bincount([PP.draw(int(v), row) for v in x], minlength=W.shape[1])
    expected = W[0] / W[0].sum() * x.shape[0]
    assert stats.chisquare(counts, expected).pvalue > 1e-4


def test_fixed_point_rounds_half_to_even_and_skips():
    ulp = 2.0 ** -21   # half a fixed-point unit
    assert PP.fixed(1.0) == 1 << 20 and PP.fixed(-2.5) == -5 * (1 << 19)
    assert PP.fixed(ulp) == 0 and PP.fixed(3 * ulp) == 2 and PP.fixed(-ulp) == 0 and PP.fixed(-3 * ulp) == -2
    assert PP.fixed(5 * ulp) == 2 and PP.fixed(7 * ulp) == 4
    assert PP.fixed(float("nan")) is None and PP.fixed(float("inf")) is None and PP.fixed(-float("inf")) is None
    assert PP.fixed(2.0 ** 42) is None and PP.fixed(-2.0 ** 42) is None       # |v| * 2^20 = 2^62
    assert PP.fixed(np.nextafter(2.0 ** 42, 0)) == int(np.nextafter(2.0 ** 42, 0) * 2.0 ** 20)


def test_accumulate_adds_per_run_and_team_and_skips():
    ret = np.array([[1.0, 2.0, -0.5, np.nan, 3.0], [0.25, np.inf, 1.0, 1.0, 2.0 ** 50]])
    team = np.array([[0, 2, 0, 1, -1], [1, 1, 1, 0, 0]])
    count, total = PP.accumulate(np.zeros((2, 3)), np.zeros((2, 3)), ret, team)
    assert count.tolist() == [[2, 0, 1], [1, 2, 0]]
    assert total.tolist() == [[1 << 19, 0, 2 << 20], [1 << 20, (5 << 18), 0]]
    c2, t2 = PP.accumulate(count, total, ret, team)
    assert np.array_equal(c2, 2 * count) and np.array_equal(t2, 2 * total)
    m = PP.means(count, total)
    assert m[0, 0] == 0.25 and np.isnan(m[0, 1]) and m[1, 1] == 0.625


def _stats(means, counts):
    """count / sum arrays whose means are exactly ``means`` (NaN: unplayed)."""
    c = np.array([[0 if np.isnan(m) else n for m, n in zip(means, counts)]], dtype=np.int64)
    s = np.array([[0 if np.isnan(m) else int(round(m * n * 2 ** 20)) for m, n in zip(means, counts)]], dtype=np.int64)
    return c, s


def test_weight_edge_cases():
    nan = float("nan")
    c, s = _stats([nan] * 4, [0] * 4)                                   # no team played
    assert (PP.weights(c, s, 2, 0.1) == UNIT).all()
    c, s = _stats([3.0, 3.0, nan], [4, 2, 0])                           # hi == lo
    assert (PP.weights(c, s, 2, 0.1) == UNIT).all()
    c, s = _stats([1.0, 3.0, 2.0, nan], [4, 2, 8, 0])
    W = PP.weights(c, s, 1, 0.0)
    assert W[0].tolist() == [UNIT, 0, UNIT // 2, UNIT]                  # worst 1, best 0 (f = 0), unplayed 1
    W = PP.weights(c, s, 0, 0.0)                                        # p = 0: x^0 = 1 for every played team
    assert (W == UNIT).all()
    W = PP.weights(c, s, 2, 0.5)
    assert W[0].tolist() == [UNIT, UNIT // 2, int(np.floor((0.5 + 0.5 * 0.25) * UNIT)), UNIT]
    W = PP.weights(c, s, 16, 0.1)
    assert W[0, 1] == int(np.floor(0.1 * UNIT)) and W[0, 0] == UNIT
    C = PP.table(W)
    assert C[0, 0] == 0 and np.array_equal(np.diff(C[0]), W[0])


def test_weights_are_the_fp64_formula_step_by_step():
    rng = np.random.default_rng(3)
    c = rng.integers(0, 5, size=(3, 40)).astype(np.int64)
    s = rng.integers(-(1 << 30), 1 << 30, size=(3, 40)).astype(np.int64)
    for p, f in ((2, 0.1), (3, 0.37), (7, 0.0), (1, 1.0)):
        W = PP.weights(c, s, p, f)
        for r in range(3):
            m = np.array([(float(s[r, q]) * 2.0 ** -20) / float(c[r, q]) if c[r, q] else np.nan for q in range(40)])
            hi, lo = np.nanmax(m), np.nanmin(m)
            for q in range(40):
                if c[r, q] == 0:
                    assert W[r, q] == UNIT
                elif p <= 2:   # x ** p is x * x (or x): the same rounding as the left-to-right product
                    x = (hi - m[q]) / (hi - lo)
                    assert W[r, q] == min(UNIT, int(np.floor((f + (1 - f) * x ** p) * UNIT)))
        assert ((W >= 0) & (W <= UNIT)).all() and (W.max(axis=1) == UNIT).all()
