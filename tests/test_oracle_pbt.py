"""The PBT oracle (oracle/pbt.py) against its definition: ranks form a permutation with the NaN and tie rules, q recipients
take donors from the disjoint top q, donor draws are uniform over the top q, and the perturbation arithmetic is exact."""
import math
from fractions import Fraction

import numpy as np
import pytest
from scipy import stats

from oracle import pbt as P
from oracle import philox


def test_fitness_adds_oldest_first_from_plus_zero():
    rows = np.array([[1e16, -0.0], [1.0, -0.0], [-1e16, -0.0]])
    f = P.fitness(rows)
    assert f[0] == ((0.0 + 1e16) + 1.0) + -1e16 == 0.0   # the 1.0 is lost in this order, not in fsum
    assert math.copysign(1.0, f[1]) == 1.0                # +0.0 + -0.0 = +0.0


@pytest.mark.parametrize("R", [1, 2, 7, 64, 300])
def test_ranks_form_a_permutation(R):
    fit = np.random.RandomState(R).normal(size=R)
    order, rank = P.rank_order(fit)
    assert sorted(order.tolist()) == list(range(R)) and sorted(rank.tolist()) == list(range(R))
    assert np.array_equal(order[rank], np.arange(R))
    assert np.all(np.diff(fit[order]) <= 0)


def test_ties_go_to_the_lower_index_and_nan_ranks_last():
    fit = np.array([1.0, np.nan, 3.0, 1.0, -np.inf, np.nan, 3.0, -0.0, 0.0])
    order, rank = P.rank_order(fit)
    assert order.tolist() == [2, 6, 0, 3, 7, 8, 4, 1, 5]
    assert rank[1] == 7 and rank[5] == 8


@pytest.mark.parametrize("R, fraction", [(8, 0.25), (7, 0.5), (10, 0.3), (3, 0.25), (128, 0.5), (5, 0.0)])
def test_recipients_take_donors_from_the_disjoint_top_q(R, fraction):
    rng = np.random.RandomState(R)
    q = math.floor(fraction * R)
    hyper = dict(lr_actor=rng.uniform(1e-5, 1e-3, R), lr_critic=rng.uniform(1e-5, 1e-3, R),
                 gamma=rng.uniform(0.5, 0.99, R).astype(np.float32), beta=rng.uniform(0, 0.1, R).astype(np.float32))
    state = dict(actor_params=rng.normal(size=(R * 3, 105)).astype(np.float32), actor_step=np.arange(R * 3, dtype=np.int32))
    rows = rng.normal(size=(4, R))
    new, hyp, log = P.generation(rows, hyper, state, q, 7, (0.8, 1.2), seed=9, g=3)
    order = np.argsort(-log["fitness"], kind="stable")
    top, bottom = set(order[:q].tolist()), set(order[R - q:].tolist())
    assert not top & bottom
    recipients = np.flatnonzero(log["donor"] >= 0)
    assert set(recipients.tolist()) == bottom
    for v in recipients:
        d = log["donor"][v]
        assert d in top
        assert np.array_equal(new["actor_params"][v * 3:(v + 1) * 3], state["actor_params"][d * 3:(d + 1) * 3])
        assert hyp["gamma"][v] == hyper["gamma"][d]
    kept = np.flatnonzero(log["donor"] < 0)
    for r in kept:
        assert np.array_equal(new["actor_step"][r * 3:(r + 1) * 3], state["actor_step"][r * 3:(r + 1) * 3])
        assert all(hyp[k][r] == np.asarray(hyper[k])[r] for k in hyp)


def test_donor_draws_are_uniform_over_the_top_q():
    q, recipients, gens = 5, np.arange(100, 110), 400
    counts = np.zeros(q, dtype=np.int64)
    for g in range(gens):
        x, _, _, _ = P.words(12345, g, recipients)
        counts += np.bincount(P.donor_ranks(x, q), minlength=q)
    assert counts.sum() == gens * recipients.size
    assert stats.chisquare(counts).pvalue > 1e-3


def test_donor_rank_stays_below_q_at_the_extremes():
    x = np.array([0, 0xFF, 0x100, 0xFFFFFFFF], dtype=np.uint32)
    for q in (1, 2, 3, 16383, 32767):
        r = P.donor_ranks(x, q)
        assert r.min() >= 0 and r.max() < q
        assert r[-1] == ((0xFFFFFF * q) >> 24)


def test_words_are_stream_5_of_the_shared_generator():
    x, y, z, w = P.words(2 ** 40 + 3, 7, [0, 5])
    ref = philox.philox4x32(np.array([0, 5], dtype=np.uint32), 0, 5 << 16, 7, 3, 2 ** 8)
    for a, b in zip((x, y, z, w), ref):
        assert np.array_equal(a, b)


def test_perturbation_arithmetic_is_exact():
    rng = np.random.RandomState(1)
    for lr, beta, f in zip(rng.uniform(1e-6, 1e-2, 200), rng.uniform(0, 0.2, 200).astype(np.float32),
                           rng.uniform(0.1, 3.0, 200)):
        for top in (0, 1 << 31):
            factors = (f, 1.0 / f)
            fv = factors[1] if top else factors[0]
            got = P.perturb_lr(lr, top, factors)
            assert got.dtype == np.float64
            assert Fraction(float(got)) == _round_f64(Fraction(float(lr)) * Fraction(fv))
            b = P.perturb_beta(beta, top | 5, factors)
            assert b.dtype == np.float32
            wide = float(np.float64(beta) * np.float64(fv))          # one fp64 product ...
            assert Fraction(wide) == _round_f64(Fraction(float(beta)) * Fraction(fv))
            assert b == np.float32(wide)                              # ... rounded once to f32
            err = abs(Fraction(float(b)) - Fraction(wide))
            for nb in (np.nextafter(b, np.float32(np.inf)), np.nextafter(b, np.float32(-np.inf))):
                assert err <= abs(Fraction(float(nb)) - Fraction(wide))   # no f32 neighbour is nearer


def _round_f64(x):
    """The fp64 nearest to the rational x (ties to even), for positive normal x."""
    f = float(x)   # Fraction -> float rounds correctly (to nearest, ties to even)
    return Fraction(f)


def test_gamma_is_never_perturbed_and_q_zero_changes_nothing():
    R = 6
    hyper = dict(lr_actor=np.full(R, 1e-4), lr_critic=np.full(R, 2e-4), gamma=np.full(R, 0.9, np.float32),
                 beta=np.full(R, 1e-3, np.float32))
    state = dict(actor_params=np.arange(R * 2 * 4, dtype=np.float32).reshape(R * 2, 4))
    new, hyp, log = P.generation(np.ones((2, R)), hyper, state, 0, 7, (0.5, 2.0), 0, 0)
    assert np.array_equal(new["actor_params"], state["actor_params"]) and (log["donor"] == -1).all()
    new, hyp, log = P.generation(np.arange(2 * R, dtype=np.float64).reshape(2, R), hyper, state, 3, 7, (0.5, 2.0), 0, 0)
    assert (hyp["gamma"] == np.float32(0.9)).all()
    assert set(np.unique(hyp["lr_actor"][log["donor"] >= 0])) <= {5e-5, 2e-4}
