"""The partner oracle (oracle/partners.py) against its definition: the draw is ((x * Q) >> 32) of the stream-6 word x, one team
is always team 0, the draws are uniform over the teams, and the seating writes exactly the drawn rows of valid runs."""
import numpy as np
import pytest
from scipy import stats

from oracle import partners as PT
from oracle import philox


def test_draw_is_the_formula_applied_to_stream_6_words():
    for seed in (0, 7, 2 ** 40 + 3, 2 ** 64 - 1):
        for episode in (0, 1, 999, 2 ** 32 - 1):
            x = philox.draw(seed, 6, episode, 0, np.zeros(1, dtype=np.uint64))[0][0]
            ref = philox.philox4x32(np.uint32(0), 0, 6 << 16, episode, seed & 0xFFFFFFFF, seed >> 32)[0]
            assert int(x) == int(ref)
            for Q in (1, 2, 3, 1000, 1 << 20):
                assert PT.team(seed, episode, Q) == (int(x) * Q) >> 32
                assert 0 <= PT.team(seed, episode, Q) < Q


def test_one_team_is_always_team_zero():
    assert {PT.team(s, k, 1) for s in range(20) for k in range(50)} == {0}


@pytest.mark.parametrize("Q", [2, 7, 16, 100])
def test_draws_are_uniform_over_the_teams(Q):
    counts = np.bincount([PT.team(seed, k, Q) for seed in range(40) for k in range(100)], minlength=Q)
    assert counts.sum() == 4000 and counts.shape == (Q,)
    assert stats.chisquare(counts).pvalue > 1e-3


def test_runs_with_the_same_seed_draw_the_same_team():
    assert PT.words(5, 3) == PT.words(5, 3) and PT.words(5, 3) != PT.words(6, 3) and PT.words(5, 3) != PT.words(5, 4)


def test_seat_writes_only_the_drawn_rows_and_guards_bad_entries():
    R, N = 4, 5
    rows = np.arange(6 * 105, dtype=np.float32).reshape(6, 105) + 0.5
    teams, seats = np.array([[0, 1], [2, 3], [4, 5]]), np.array([1, 3])
    actor = -np.ones((R * N, 105), dtype=np.float32)
    seeds = [3, 9, 3, 11]
    out, log = PT.seat(actor, (rows, teams, seats), 7, seeds)
    for r, s in enumerate(seeds):
        t = PT.team(s, 7, 3)
        assert log[r] == t
        assert np.array_equal(out[r * N + seats], rows[teams[t]])
        keep = [i for i in range(N) if i not in seats]
        assert np.array_equal(out[r * N + np.array(keep)], actor[r * N + np.array(keep)])
    assert log[0] == log[2]   # a repeated seed draws the same team
    bad_teams = teams.copy()
    bad_teams[log[1], 0] = 6
    out2, log2 = PT.seat(actor, (rows, bad_teams, seats), 7, seeds)
    assert log2[1] == -1 and np.array_equal(out2[N:2 * N], actor[N:2 * N])
    assert all(log2[r] == log[r] for r in (0, 2, 3) if log[r] != log[1])
    _, log3 = PT.seat(actor, (rows, teams, np.array([1, 5])), 7, seeds)
    assert (log3 == -1).all()


def test_seat_of_one_run_takes_a_scalar_seed():
    actor = np.zeros((2, 105), dtype=np.float32)
    rows = np.ones((3, 105), dtype=np.float32) * np.arange(3, dtype=np.float32)[:, None]
    out, log = PT.seat(actor, (rows, np.array([[0], [1], [2]]), np.array([1])), 0, 42)
    assert log.shape == (1,) and log[0] == PT.team(42, 0, 3)
    assert (out[1] == log[0]).all() and (out[0] == 0).all()
