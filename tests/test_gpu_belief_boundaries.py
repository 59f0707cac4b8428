"""Every belief-filter kernel against the oracle at its decision boundaries, bit for bit.

Each output of the belief filter is a decision: the stored posterior is rint(100 * b), which becomes the next prior (Q10),
and the predicted action is an inverse-CDF comparison of u with the cumulative prediction (Q11).  Random models almost
never put a value on a rounding tie; structured ones do all the time.  The papers' ORG models reach an exact fp64 37.5
after the other agent plays 0, 0, 0, 1, 1, and decimal models (entries k / 20) reach exact halves within a few updates.
When every agent plays the same actions, every record of an env reaches the same tie in the same step.

Inputs are priors a run can hold (a breadth-first search from round(1/M, 2) under the agent's models), seen actions and
uniforms placed on the boundaries.  `Bands` classifies every record from the exact real values (fractions.Fraction of the
fp64 inputs) of 100 * bp / S and of each cumulative c_a, next to the oracle's fp64 values, and each case asserts a minimum
count in every band it claims and prints the counts, so no case can go vacuous.  The bands:

  rounding  half_even / half_odd   the fp64 100 * b is exactly k + 1/2 (rint must round half to even)
            op_order               real distance to k + 1/2 below 1e-12, fp64 value not on the half (operation order decides)
            refine                 distance in [1e-12, 1e-6 (n + 1)], n the nearest integer: inside the episode kernel's
                                   second-level bound
            first                  distance in (1e-6 (n + 1), 1e-4): inside the fp32 screen's first-level window only
            outside                distance in [1e-4, 3e-4): just outside the window, fp32 decides
  cdf       eq / ulp               u == c_a, or one fp64 step either side of it
            d1e-12 ... d1.1e-5     |u - c_a| about 1e-12, 1e-7, 1e-6, 9e-6 (inside the 1e-5 window) and 1.1e-5 (outside)
            fall                   u >= the fp64 total of the prediction, which is below 1: falls through to action 0
            near1 / zero           u in (1 - 2e-5, 1), u == 0
            philox_split           device Philox: the fp64 u = (w + 1/2) 2^-32 and the fp32 screen's floor(w / 2^9) 2^-23 lie on
                                   opposite sides of some c_a

The kernels: belief_dense_kernel<5,3>, <3,3>, <5,5> and the generic one (class API), belief_pairs_kernel (K < 32),
belief_pairs_table_kernel (K >= 32, fp32 screen, a 1024-entry exact queue per block and the inline path behind it, both
templates), belief_pairs_episode_kernel (second-level screen, per-warp exact pass, both templates) and the belief stage of
rollout_fused_kernel, which only a trainer reaches: trainers on every rollout path, with saturated actors that make all
agents play one action, against the oracle (tests/test_gpu_trainer_oracle_scale.py: check_episode)."""
import functools
from collections import Counter
from fractions import Fraction

import numpy as np
import pytest

from ia2c_b200.belief import HVT_KNOWN_FILTER_ACTION, ORG_KNOWN_FILTER_ACTION
from oracle import belief as B
from oracle import philox as P
from oracle.loops import mode3, others_of
from tests.helpers import host

# Decimal models with exact fp64 halves reachable from the uniform prior.  Found by a CPU search: for M = 2..6,
# RandomState(M) draws rows (a, b, 20 - a - b) with a in 1..18 and b in 1..19 - a, the model is rows / 20, and the first
# candidate whose breadth-first search (depth 8, all three seen actions) meets a fp64 100 * b == k + 1/2 is kept.  M = 5
# is the model quoted with the issue of these tests instead: it reaches 37.5 at the FIRST update (uniform prior, seen 0).
DECIMAL_MODELS = {
    2: np.array([[18, 1, 1], [12, 6, 2]]) / 20.0,
    3: np.array([[11, 1, 8], [4, 6, 10], [9, 4, 7]]) / 20.0,
    4: np.array([[15, 4, 1], [6, 9, 5], [2, 10, 8], [9, 8, 3]]) / 20.0,
    5: np.array([[5, 11, 4], [4, 2, 14], [4, 7, 9], [2, 17, 1], [13, 2, 5]]) / 20.0,
    6: np.array([[11, 3, 6], [10, 1, 9], [4, 15, 1], [11, 2, 7], [14, 2, 4], [16, 2, 2]]) / 20.0,
}
ROUND_BANDS = ("half_even", "half_odd", "op_order", "refine", "first", "outside")
CDF_OFFSETS = {"d1e-12": 1e-12, "d1e-7": 1e-7, "d1e-6": 1e-6, "d9e-6": 9e-6, "d1.1e-5": 1.1e-5}
CDF_BANDS = ("eq", "ulp", *CDF_OFFSETS, "fall", "near1", "zero")
_HALF = Fraction(1, 2)


# ------------------------------------------------------------------------------------------------ inputs
def lik_rows(seen, A):
    return B.likelihood_from_action(np.asarray(seen), A)


def fp64_sequence(fa, k, seen):
    """The oracle's fp64 sequence with one model per row: fa [R,M,A], k [R,M] hundredths, seen [R] -> (x = 100 * b [R,M],
    cumulative prediction c [R,A]).  Same operations in the same order as oracle/belief.py."""
    fa = np.asarray(fa, dtype=np.float64)
    prev = B.from_hundredths(k)
    lik = lik_rows(seen, fa.shape[-1])
    bp = None
    for a in range(fa.shape[-1]):
        term = lik[:, a:a + 1] * (fa[:, :, a] * prev)
        bp = term if bp is None else bp + term
    S = bp[:, 0].copy()
    for m in range(1, bp.shape[1]):
        S = S + bp[:, m]
    b = bp / S[:, None]
    pred = np.zeros((b.shape[0], fa.shape[-1]))
    for m in range(b.shape[1]):
        pred = pred + b[:, m:m + 1] * fa[:, m, :]
    return b * 100.0, np.cumsum(pred, axis=1)   # numpy's cumsum adds left to right, like the oracle's running c


@functools.lru_cache(maxsize=None)
def _exact(fa_bytes, shape, k, seen):
    """Exact real 100 * bp / S per model and cumulative c_a of the fp64 inputs (models, k / 100, 0.8 / 0.1)."""
    fa = np.frombuffer(fa_bytes, dtype=np.float64).reshape(shape)
    M, A = shape
    lik = [Fraction(B.LIK_HIT if a == seen else B.LIK_MISS) for a in range(A)]
    F = [[Fraction(float(fa[m, a])) for a in range(A)] for m in range(M)]
    bp = [sum(lik[a] * F[m][a] * Fraction(k[m] / 100.0) for a in range(A)) for m in range(M)]
    S = sum(bp)
    x = tuple(100 * v / S for v in bp)
    c, acc = [], Fraction(0)
    for a in range(A):
        acc += sum(bp[m] / S * F[m][a] for m in range(M))
        c.append(acc)
    return x, tuple(c)


def exact(fa, k, seen):
    fa = np.ascontiguousarray(fa, dtype=np.float64)
    return _exact(fa.tobytes(), fa.shape, tuple(int(v) for v in k), int(seen))


@functools.lru_cache(maxsize=None)
def _exact_round_band(fa_bytes, shape, k, seen):
    fa = np.frombuffer(fa_bytes, dtype=np.float64).reshape(shape)
    best = "clear"
    for xm in exact(fa, k, seen)[0]:
        fl = xm.numerator // xm.denominator
        d = abs(xm - fl - _HALF)
        near = fl + (xm - fl > _HALF)     # the integer nearest x: rint(x32) in the episode kernel's bound 1e-6 (rint + 1)
        band = ("op_order" if d < Fraction(1, 10 ** 12) else "refine" if d <= Fraction(near + 1, 10 ** 6) else
                "first" if d < Fraction(1, 10 ** 4) else "outside" if d < Fraction(3, 10 ** 4) else "clear")
        best = min(best, band, key=("op_order", "refine", "first", "outside", "clear").index)
    return best


def _per_unique(rows, fn):
    """fn(first index) evaluated once per distinct row of `rows` -> object array over all rows."""
    out = np.empty(len(rows), dtype=object)
    if len(rows):
        _, first, inv = np.unique(rows, axis=0, return_index=True, return_inverse=True)
        vals = np.array([fn(f) for f in first], dtype=object)
        out[:] = vals[np.asarray(inv).reshape(-1)]
    return out


def round_bands(fa, k, seen):
    """Rounding band of every record (fa [R,M,A], k [R,M], seen [R]): the most critical of its M posterior values.  A fp64
    value exactly on k + 1/2 is classified by the parity of k; otherwise the real distance decides (Fraction), for every
    record whose fp64 values come within 1e-3 of a half-integer (the fp64 values are within 1e-13 of the real ones, so
    the others are clear)."""
    x64, _ = fp64_sequence(fa, k, seen)
    frac = x64 - np.floor(x64)
    R = len(k)
    out = np.full(R, "clear", dtype=object)
    half = frac == 0.5
    anyhalf = half.any(1)
    even = np.floor(x64)[np.arange(R), np.argmax(half, 1)] % 2 == 0
    out[anyhalf & even] = "half_even"
    out[anyhalf & ~even] = "half_odd"
    cand = np.flatnonzero(~anyhalf & (np.abs(frac - 0.5).min(1) <= 1e-3))
    rows = np.concatenate([fa[cand].reshape(len(cand), fa[0].size), k[cand].astype(np.float64), seen[cand, None].astype(np.float64)], axis=1)
    out[cand] = _per_unique(rows, lambda f: _exact_round_band(np.ascontiguousarray(fa[cand[f]]).tobytes(), fa.shape[1:],
                                                             tuple(int(v) for v in k[cand[f]]), int(seen[cand[f]])))
    return out


def cdf_bands(c64, u):
    """Inverse-CDF band of every record at its injected u (c64 [R,A] the oracle's cumulative prediction).  u - c_a is exact
    in fp64 near a boundary and c_a is within 1e-16 of the real cumulative, far below the 10 % width of the offset bands
    (test_band_classifier_agrees_with_direct_fractions checks both against Fraction)."""
    inner = c64[:, :-1]
    d = np.abs(inner - u[:, None]).min(1)
    out = np.full(len(u), "far", dtype=object)
    for name, off in CDF_OFFSETS.items():
        out[(d >= 0.9 * off) & (d <= 1.1 * off)] = name
    out[(d > 0) & (d < 2e-12)] = "d1e-12"
    out[(u > 1.0 - 2e-5) & (u < 1.0)] = "near1"
    out[(c64[:, -1] < 1.0) & (u >= c64[:, -1])] = "fall"
    out[np.any(u[:, None] == np.nextafter(inner, 2.0), 1) | np.any(u[:, None] == np.nextafter(inner, -1.0), 1)] = "ulp"
    out[np.any(u[:, None] == inner, 1)] = "eq"
    out[u == 0.0] = "zero"
    return out


def philox_split(c64, u):
    w = np.round(u * 2.0 ** 32 - 0.5)
    uf = np.floor(w / 512.0) * 2.0 ** -23
    inner = c64[:, :-1]
    return np.any((u[:, None] < inner) != (uf[:, None] < inner), axis=1)


class Bands:
    """Band counts of a set of records (fa [R,M,A], k [R,M], seen [R], u [R] or None, philox: u came from device Philox)."""

    def __init__(self, fa, k, seen, u=None, philox=False):
        fa, k, seen = np.asarray(fa, dtype=np.float64), np.asarray(k), np.asarray(seen)
        self.rounding = round_bands(fa, k, seen)
        self.counts = Counter(self.rounding.tolist())
        self.cdf = None
        if u is not None:
            u = np.asarray(u, dtype=np.float64).reshape(-1)
            c64 = fp64_sequence(fa, k, seen)[1]
            if philox:
                self.counts["philox_split"] += int(philox_split(c64, u).sum())
            else:
                self.cdf = cdf_bands(c64, u)
                self.counts.update(self.cdf.tolist())

    def merge(self, other):
        self.counts.update(other.counts)
        return self

    def require(self, label, **minimum):
        print(f"\n[{label}] " + " ".join(f"{b}={self.counts[b]}" for b in (*ROUND_BANDS, *CDF_BANDS, "philox_split") if self.counts[b]))
        for band, n in minimum.items():   # "half": an exact fp64 half of either parity
            if band == "half":
                self.counts["half"] = self.counts["half_even"] + self.counts["half_odd"]
            assert self.counts[band] >= n, f"{label}: {self.counts[band]} records in band {band}, want >= {n}"
        return self


@functools.lru_cache(maxsize=None)
def _catalog(fa_bytes, shape, depth, cap):
    fa = np.frombuffer(fa_bytes, dtype=np.float64).reshape(shape)
    M, A = shape
    start = tuple(int(v) for v in B.to_hundredths(B.uniform_prior(1, M)[0]))
    paths = {start: ()}
    front = [start]
    for _ in range(depth):
        nxt = []
        ks = np.array(front)
        for a in range(A):
            _, bp, _ = B.belief_update(fa, lik_rows(np.full(len(front), a), A), B.from_hundredths(ks), np.full(len(front), 0.5))
            for s, row in zip(front, B.to_hundredths(bp)):
                key = tuple(int(v) for v in row)
                if key not in paths:
                    paths[key] = paths[s] + (a,)
                    nxt.append(key)
        front = nxt
        if not front or len(paths) >= cap:
            break
    states = np.array(list(paths), dtype=np.uint8)
    bands, cvals = {}, {}
    for s in range(A):
        rows = np.ascontiguousarray(np.broadcast_to(fa, (len(states), M, A)))
        bands[s] = round_bands(rows, states, np.full(len(states), s))
        cvals[s] = fp64_sequence(rows, states, np.full(len(states), s))[1]
    return states, paths, bands, cvals


def catalog(fa, depth=12, cap=6000):
    """States a run can hold under model fa (breadth-first from the uniform prior), a shortest action path to each, and
    per seen action the rounding band and the fp64 cumulative prediction of every state."""
    fa = np.ascontiguousarray(fa, dtype=np.float64)
    return _catalog(fa.tobytes(), fa.shape, depth, cap)


def random_models(n, M, seed):
    rng = np.random.RandomState(seed)
    fa = rng.rand(n, M, 3)
    return fa / fa.sum(-1, keepdims=True)


def agent_models(N, M, seed):
    """Every third agent holds a random model (bands that ties do not cover), the others the tie models."""
    tie = [DECIMAL_MODELS[M]] + ([ORG_KNOWN_FILTER_ACTION] if M == 3 else [])
    rnd = random_models(2, M, seed)
    return np.stack([tie[i % len(tie)] if i % 3 != 2 else rnd[i % 2] for i in range(N)])


def pick_priors(rng, fa, seen, boundary=0.6):
    """One catalog state per record (fa [R,M,A], seen [R]); a `boundary` share is drawn band-first among the states whose
    posterior rounds near a half-integer."""
    R, M = seen.shape[0], fa.shape[1]
    k = np.zeros((R, M), dtype=np.uint8)
    keys = np.unique(np.concatenate([fa.reshape(R, -1), seen[:, None].astype(np.float64)], axis=1), axis=0, return_inverse=True)[1]
    keys = np.asarray(keys).reshape(-1)
    for g in np.unique(keys):
        idx = np.flatnonzero(keys == g)
        states, _, bands, _ = catalog(fa[idx[0]])
        band = bands[int(seen[idx[0]])]
        pools = [np.flatnonzero(band == b) for b in ROUND_BANDS]
        pools = [p for p in pools if len(p)]
        choice = rng.randint(len(states), size=len(idx))
        if pools:
            tie = rng.rand(len(idx)) < boundary
            which = rng.randint(len(pools), size=len(idx))
            for n, p in enumerate(pools):
                sel = tie & (which == n)
                choice[sel] = p[rng.randint(len(p), size=int(sel.sum()))]
        k[idx] = states[choice]
    return k


def boundary_uniforms(rng, fa, k, seen, share=0.7):
    """Injected uniforms: a `share` of the records on a CDF boundary of their own fp64 prediction, the rest uniform."""
    _, c64 = fp64_sequence(fa, k, seen)
    R = len(k)
    u = rng.rand(R)
    kind = rng.randint(0, 14, size=R)
    a = rng.randint(0, 2, size=R)
    c = c64[np.arange(R), a]
    side = np.where(rng.rand(R) < 0.5, -1.0, 1.0)
    offs = list(CDF_OFFSETS.values())
    for n in range(14):
        sel = (kind == n) & (rng.rand(R) < share)
        if n == 0:
            u[sel] = c[sel]
        elif n == 1:
            u[sel] = np.nextafter(c[sel], 2.0)
        elif n == 2:
            u[sel] = np.nextafter(c[sel], -1.0)
        elif n < 8:
            u[sel] = c[sel] + side[sel] * offs[n - 3]
        elif n == 8:
            low = sel & (c64[:, -1] < 1.0)
            u[low] = c64[low, -1] + (1.0 - c64[low, -1]) * rng.rand(int(low.sum()))
        elif n == 9:
            u[sel] = 1.0 - 2e-5 * rng.rand(int(sel.sum())) * 0.999
        elif n == 10:
            u[sel] = 0.0
    return np.clip(u, 0.0, np.nextafter(1.0, 0.0))


# ------------------------------------------------------------------------------------------------ oracle of the packed layout
def pairs_oracle(fa, act, prior, u):
    """fa [N,M,3]; act [E,N]; prior [E,N,K,M] hundredths; u [E,N,K] -> ap [E,N,K], posterior hundredths [E,N,K,M]."""
    E, N = act.shape
    K, M = N - 1, fa.shape[1]
    ap = np.zeros((E, N, K), dtype=np.int64)
    post = np.zeros((E, N, K, M), dtype=np.uint8)
    for i in range(N):
        others = np.asarray(others_of(i, N))
        a, b, _ = B.belief_update(fa[i], lik_rows(act[:, others].reshape(-1), 3), B.from_hundredths(prior[:, i].reshape(-1, M)),
                                  u[:, i].reshape(-1))
        ap[:, i], post[:, i] = a.reshape(E, K), B.to_hundredths(b).reshape(E, K, M)
    return ap, post


def seen_of(act):
    """act [E,N] -> the action each record (e, i, jj) sees: act[e, j] with j the jj-th other of i, [E,N,K]."""
    E, N = act.shape
    return np.stack([act[:, others_of(i, N)] for i in range(N)], axis=1)


def record_views(fa, act, prior, u=None):
    """Flatten records for Bands: per-record model, prior, seen action and uniform."""
    E, N, K, M = prior.shape
    fa_r = np.broadcast_to(fa[None, :, None], (E, N, K) + fa.shape[1:]).reshape(-1, M, 3)
    return fa_r, prior.reshape(-1, M), seen_of(act).reshape(-1), None if u is None else np.asarray(u).reshape(-1)


def assert_records(rec, M, ap, post):
    assert np.array_equal(rec[..., :M], post), "posterior bytes differ from the oracle"
    assert np.array_equal(rec[..., 6], ap), "predicted action (byte 6) differs from the oracle"
    assert not rec[..., M:6].any() and not rec[..., 7].any(), "bytes M..5 and 7 must be zero"


def belief_rows(E, N, env_offset):
    return (np.arange(E)[:, None] + env_offset) * N + np.arange(N)[None, :]


# ------------------------------------------------------------------------------------------------ CPU pins
def _x(fa, prior, seen):
    return fp64_sequence(np.asarray(fa)[None], B.to_hundredths(np.asarray(prior))[None], np.array([seen]))[0][0]


def test_org_sequences_reach_ties_on_the_oracle():
    fa = ORG_KNOWN_FILTER_ACTION
    prior = B.uniform_prior(1, 3)
    trail = []
    for a in (0, 0, 0, 1, 1):
        x = _x(fa, prior[0], a)
        _, prior, _ = B.belief_update(fa, lik_rows([a], 3), prior, [0.5])
        trail.append(tuple(B.to_hundredths(prior[0])))
    assert trail == [(42, 33, 24), (51, 32, 17), (59, 29, 11), (49, 34, 17), (38, 38, 24)]
    assert x[1] == 37.5                                                  # exact fp64 tie, rounded half to even
    # the same real value, two operation orders: 42.50000000000001 -> 43 after seeing 1, exactly 42.5 -> 42 after seeing 2
    p = np.array([[0.55, 0.23, 0.23]])
    x1, x2 = _x(fa, p[0], 1), _x(fa, p[0], 2)
    assert x1[0] == np.nextafter(42.5, 43.0) and x2[0] == 42.5
    assert exact(fa, (55, 23, 23), 1)[0][0] == exact(fa, (55, 23, 23), 2)[0][0]
    assert B.to_hundredths(B.belief_update(fa, lik_rows([1], 3), p, [0.5])[1])[0, 0] == 43
    assert B.to_hundredths(B.belief_update(fa, lik_rows([2], 3), p, [0.5])[1])[0, 0] == 42
    two = round_bands(np.stack([fa, fa]), np.array([[55, 23, 23]] * 2, dtype=np.uint8), np.array([1, 2]))
    assert list(two) == ["op_order", "half_even"]


def test_decimal_models_reach_exact_halves():
    x = _x(DECIMAL_MODELS[5], B.uniform_prior(1, 5)[0], 0)
    assert x[4] == 37.5 and B.to_hundredths(B.belief_update(DECIMAL_MODELS[5], lik_rows([0], 3), B.uniform_prior(1, 5), [0.5])[1])[0, 4] == 38
    for M, fa in DECIMAL_MODELS.items():
        states, paths, bands, _ = catalog(fa)
        halves = [(s, a) for a in range(3) for s in np.flatnonzero(np.isin(bands[a], ("half_even", "half_odd")))]
        assert halves, f"M={M}: no exact fp64 half reachable"
        assert min(len(paths[tuple(int(v) for v in states[s])]) for s, _ in halves) <= 7


def test_golden_near_tie_rows(golden):
    """The five near-tie values of the golden class vectors; the real class rounded each of them as the oracle does."""
    g = golden("belief_vectors.npz")
    hits = []
    for tag, t in (("org_known", 44), ("org_known", 64), ("org_known", 67), ("org_known", 68), ("hvt_known", 25)):
        fa = g[f"{tag}/filterAction"]
        lik, prev, u = g[f"{tag}/obs"][t], g[f"{tag}/prev"][t], g[f"{tag}/u"][t]
        ap, bp, _ = B.belief_update(fa, lik, prev, u)
        assert np.array_equal(bp, g[f"{tag}/bprime"][t]) and np.array_equal(ap, g[f"{tag}/ap"][t])
        b64 = fp64_sequence(np.broadcast_to(fa, (len(prev),) + fa.shape), B.to_hundredths(prev), np.asarray(lik).argmax(1))[0]
        assert np.array_equal(lik, lik_rows(np.asarray(lik).argmax(1), fa.shape[1])) and np.array_equal(np.rint(b64) / 100.0, bp)
        near = np.argwhere(np.abs(b64 - np.floor(b64) - 0.5) < 1e-9)
        assert len(near) >= 1, (tag, t)
        for r, m in near:
            hits.append((tag, t, int(r), int(m), float(b64[r, m]), int(np.rint(bp[r, m] * 100))))
    print("\n" + "\n".join(map(str, hits)))
    assert len(hits) >= 5


def test_band_classifier_agrees_with_direct_fractions():
    rng = np.random.RandomState(3)
    fa = np.stack([DECIMAL_MODELS[5]] * 400 + [random_models(1, 5, 9)[0]] * 400)
    seen = rng.randint(0, 3, size=800)
    k = pick_priors(rng, fa, seen, boundary=0.8)
    u = boundary_uniforms(rng, fa, k, seen)
    bands = Bands(fa, k, seen, u).require("sample", half_even=1, half_odd=1, op_order=1, refine=1, first=1, outside=1, eq=1, ulp=1,
                                          zero=1, near1=1, fall=1, **{"d1e-12": 1, "d1e-7": 1, "d1e-6": 1, "d9e-6": 1, "d1.1e-5": 1})
    x64, c64 = fp64_sequence(fa, k, seen)
    for r in range(800):
        lik = [Fraction(0.8) if a == seen[r] else Fraction(0.1) for a in range(3)]
        bp = [sum(lik[a] * Fraction(fa[r, m, a]) * Fraction(k[r, m] / 100.0) for a in range(3)) for m in range(5)]
        xs = [100 * v / sum(bp) for v in bp]
        # per value: distance to the nearest half-integer and the episode kernel's bound 1e-6 (nearest integer + 1)
        dist = [(abs(v - (v.numerator // v.denominator) - _HALF), Fraction(round(v) + 1, 10 ** 6)) for v in xs]
        band = bands.rounding[r]
        if band in ("half_even", "half_odd"):
            x = x64[r][x64[r] - np.floor(x64[r]) == 0.5]
            assert len(x) and (int(np.floor(x[0])) % 2 == 0) == (band == "half_even")
        elif band == "op_order":
            assert not np.any(x64[r] - np.floor(x64[r]) == 0.5) and min(d for d, _ in dist) < Fraction(1, 10 ** 12)
        elif band == "refine":
            assert any(Fraction(1, 10 ** 12) <= d <= bound for d, bound in dist) and min(d for d, _ in dist) >= Fraction(1, 10 ** 12)
        elif band == "first":
            assert any(bound < d < Fraction(1, 10 ** 4) for d, bound in dist) and all(d > bound for d, bound in dist)
        elif band == "outside":
            assert min(d for d, _ in dist) >= Fraction(1, 10 ** 4) and min(d for d, _ in dist) < Fraction(3, 10 ** 4)
        else:
            assert min(d for d, _ in dist) >= Fraction(3, 10 ** 4)
        cb = bands.cdf[r]
        cs = [sum(b / sum(bp) * Fraction(fa[r, m, a]) for m, b in enumerate(bp) for a in range(j + 1)) for j in range(3)]
        ur = Fraction(u[r])
        du = min(abs(ur - c) for c in cs[:2])
        if cb == "zero":
            assert ur == 0
        elif cb in ("eq", "ulp"):
            assert du < Fraction(1, 10 ** 15) and (cb == "eq") == bool(np.any(u[r] == c64[r, :2]))
        elif cb == "fall":
            assert c64[r, 2] < 1 and ur >= Fraction(c64[r, 2]) and abs(Fraction(c64[r, 2]) - cs[2]) < Fraction(1, 10 ** 15)
        elif cb == "near1":
            assert 1 - Fraction(2, 10 ** 5) < ur < 1 and du > Fraction(1, 10 ** 15)
        elif cb in CDF_OFFSETS:
            assert Fraction(0.9 * CDF_OFFSETS[cb]) * Fraction(99, 100) <= du <= Fraction(1.1 * CDF_OFFSETS[cb]) * Fraction(101, 100) or \
                (cb == "d1e-12" and du < Fraction(2, 10 ** 12))
        else:
            assert cb == "far" and (du > Fraction(2, 10 ** 5) or (du > Fraction(1, 10 ** 15) and 1 - Fraction(2, 10 ** 5) < ur))


# ------------------------------------------------------------------------------------------------ GPU: dense (class API)
def _dense(fa, lik, prev, u):
    import torch
    from ia2c_b200 import _lib
    from tests.helpers import dptr
    lib = _lib.load()
    R, A = lik.shape
    M = prev.shape[1]
    ap = torch.empty(R, dtype=torch.int64, device="cuda")
    bp = torch.empty(R, M, dtype=torch.float64, device="cuda")
    pred = torch.empty(R, A, dtype=torch.float64, device="cuda")
    _lib.check(lib.ia2c_belief_update_dense(dptr(fa), dptr(lik), dptr(prev), dptr(u.reshape(-1)), _lib.ptr(ap), _lib.ptr(bp),
                                            _lib.ptr(pred), R, M, A, _lib.stream_ptr()))
    return host(ap), host(bp), host(pred)


def _dense_rows(fa, rng, R):
    M, A = fa.shape
    seen = rng.randint(0, A, size=R)
    fa_r = np.ascontiguousarray(np.broadcast_to(fa, (R, M, A)))
    k = pick_priors(rng, fa_r, seen)
    return fa_r, k, seen, boundary_uniforms(rng, fa_r, k, seen)


@pytest.mark.gpu
@pytest.mark.parametrize("name,fa", [("5x3", DECIMAL_MODELS[5]), ("3x3-org", ORG_KNOWN_FILTER_ACTION), ("3x3", DECIMAL_MODELS[3]),
                                     ("5x5-hvt", HVT_KNOWN_FILTER_ACTION), ("2x3", DECIMAL_MODELS[2]), ("4x3", DECIMAL_MODELS[4]),
                                     ("6x3", DECIMAL_MODELS[6])])
def test_dense_kernels_at_boundaries(name, fa):
    """belief_dense_kernel<5,3>, <3,3>, <5,5> and the generic kernel (M = 2, 4, 6) on catalog rows: posteriors, predicted
    actions and predictions equal the oracle bit for bit."""
    rng = np.random.RandomState(len(name))
    R = 3000
    fa_r, k, seen, u = _dense_rows(fa, rng, R)
    A = fa.shape[1]
    want = dict(half=1, op_order=1, eq=1, ulp=1, zero=1, near1=1, **{"d1e-6": 1, "d9e-6": 1, "d1.1e-5": 1})
    if name == "2x3":
        want.pop("op_order")
    if name in ("5x3", "3x3", "4x3", "6x3"):
        want["half_even"] = 1   # k even: round half to even and half up disagree
    Bands(fa_r, k, seen, u).require(f"dense {name}", **want)
    lik = lik_rows(seen, A)
    prev = B.from_hundredths(k)
    ap, bp, pred = _dense(fa, lik, prev, u)
    oap, obp, opred = B.belief_update(fa, lik, prev, u)
    assert np.array_equal(bp, obp) and np.array_equal(ap, oap) and np.array_equal(pred, opred)


@pytest.mark.gpu
def test_class_api_known_org_on_tie_rows(monkeypatch):
    from ia2c_b200.belief import BeliefFilter
    bf = BeliefFilter(3, 3, 4, known="org")
    # rows: the ORG sequence's exact 37.5, the two operation orders of (55, 23, 23), a plain row
    prev = np.array([[0.49, 0.34, 0.17], [0.55, 0.23, 0.23], [0.55, 0.23, 0.23], [0.33, 0.33, 0.33]])
    obs = lik_rows([1, 1, 2, 0], 3)
    tape = np.array([[0.3], [0.5], [0.7], [0.9]])
    monkeypatch.setattr(np.random, "rand", lambda *shape: tape.copy())
    ap, bprime, pred = bf.update(obs, prev)
    oap, obp, opred = B.belief_update(ORG_KNOWN_FILTER_ACTION, obs, prev, tape)
    assert np.array_equal(bprime, obp) and np.array_equal(ap, oap) and np.array_equal(pred, opred)
    assert list(np.rint(bprime[:3] * 100).astype(int)[:, [1, 0, 0]].diagonal()) == [38, 43, 42]


# ------------------------------------------------------------------------------------------------ GPU: pairs and table kernels
def _run_pairs(fa, act, prior, u, reset, dumps, seed, episode, t, env_offset, partner=True):
    """One ia2c_belief_update_pairs call on records holding `prior` (bytes M..7 junk) -> (records, pred, belief, partner)."""
    import torch
    from ia2c_b200 import _lib
    from tests.helpers import dev
    lib = _lib.load()
    E, N, K, M = prior.shape
    rec0 = np.full((E, N, K, 8), 0xA5, dtype=np.uint8)
    rec0[..., :M] = prior
    rec = dev(rec0)
    keep = [dev(fa), dev(act)] + ([dev(u)] if u is not None else [])
    pred = torch.empty(E, N, K, dtype=torch.uint8, device="cuda") if dumps else None
    bel = torch.empty(E, N, K, M, dtype=torch.uint8, device="cuda") if dumps else None
    part = torch.empty(E, N, dtype=torch.uint8, device="cuda") if partner else None
    p = lambda x: _lib.ptr(x) if x is not None else None
    _lib.check(lib.ia2c_belief_update_pairs(_lib.ptr(rec), _lib.ptr(keep[0]), _lib.ptr(keep[1]), _lib.ptr(keep[2]) if u is not None else None,
                                            p(pred), p(bel), p(part), E, N, M, int(reset), seed, episode, t, env_offset, _lib.stream_ptr()))
    torch.cuda.synchronize()
    return host(rec), None if pred is None else host(pred), None if bel is None else host(bel), None if part is None else host(part)


def _pairs_case(N, M, E, form, reset=False, seed=0):
    """form: 'injected' (u tapes, dumps, partner modes) or 'philox' (device Philox; FAST when not reset and no dumps)."""
    rng = np.random.RandomState(1000 * N + 10 * M + seed)
    K = N - 1
    fa = agent_models(N, M, seed=N * M)
    act = rng.randint(0, 3, size=(E, N)).astype(np.uint8)
    seen = seen_of(act)
    fa_r = np.broadcast_to(fa[None, :, None], (E, N, K, M, 3)).reshape(-1, M, 3)
    if reset:
        prior = np.broadcast_to(B.to_hundredths(B.uniform_prior(1, M)[0]), (E, N, K, M)).copy()
    else:
        prior = pick_priors(rng, fa_r, seen.reshape(-1)).reshape(E, N, K, M)
    pseed, episode, t, env_offset = 0x5EED0000 + N, 3, 7, 11
    if form == "injected":
        u = boundary_uniforms(rng, fa_r, prior.reshape(-1, M), seen.reshape(-1)).reshape(E, N, K)
    else:
        u = P.belief_uniforms(pseed, episode, t, belief_rows(E, N, env_offset), K)
        if not reset:   # priors from a sorted table of boundary values: the fp64 u and the fp32 screen's u straddle a c_a
            prior = _philox_priors(rng, fa, seen, u, prior)
    bands = Bands(*record_views(fa, act, prior, u), philox=form == "philox")
    rec, pred, bel, part = _run_pairs(fa, act, prior, u if form == "injected" else None, reset, form == "injected",
                                      pseed, episode, t, env_offset)
    ap, post = pairs_oracle(fa, act, prior, u)
    assert_records(rec, M, ap, post)
    if pred is not None:
        assert np.array_equal(pred, ap) and np.array_equal(bel, post)
    assert np.array_equal(part, mode3(ap))
    return bands


def _philox_priors(rng, fa, seen, u, prior):
    """Replace records' priors by catalog states whose fp64 c_0 or c_1 lies between the record's fp32 screen uniform and
    its fp64 uniform, where such a state exists."""
    E, N, K, M = prior.shape
    w = np.round(u * 2.0 ** 32 - 0.5)
    uf = np.floor(w / 512.0) * 2.0 ** -23
    out = prior.copy()
    for i in range(N):
        states, _, _, cvals = catalog(fa[i])
        for s in range(3):
            table = np.concatenate([cvals[s][:, 0], cvals[s][:, 1]])
            owner = np.concatenate([np.arange(len(states))] * 2)
            order = np.argsort(table, kind="stable")
            table, owner = table[order], owner[order]
            sel = seen[:, i] == s
            lo, hi = uf[:, i][sel], u[:, i][sel]
            pos = np.searchsorted(table, lo, side="right")   # first c > uf; it splits when c <= u
            ok = (pos < len(table)) & (table[np.minimum(pos, len(table) - 1)] <= hi)
            picked = out[:, i][sel]
            picked[ok] = states[owner[pos[ok]]]
            sub = out[:, i]
            sub[sel] = picked
            out[:, i] = sub
    return out


PAIRS_SHAPES = [(2, 2, 400), (3, 3, 300), (5, 4, 120), (8, 5, 60), (17, 6, 12), (32, 3, 6), (32, 5, 6)]


@pytest.mark.gpu
@pytest.mark.parametrize("N,M,E", PAIRS_SHAPES)
def test_pairs_kernel_at_boundaries(N, M, E):
    """belief_pairs_kernel (K < 32, fp64 throughout) with injected boundary uniforms and with device Philox."""
    _pairs_case(N, M, E, "injected").require(f"pairs N={N} M={M} injected", half=1, half_even=int(M != 2), op_order=int(M != 2), first=int(M != 2), eq=1, ulp=1, zero=1, fall=1,
                                            **{"d1e-7": 1, "d9e-6": 1})
    _pairs_case(N, M, E, "philox", seed=1).require(f"pairs N={N} M={M} philox", half=1, first=int(M != 2))


TABLE_SHAPES = [(33, 2, 40), (36, 3, 40), (130, 4, 3), (37, 5, 24), (65, 6, 8), (130, 5, 3), (1023, 3, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("N,M,E", TABLE_SHAPES)
def test_table_kernel_at_boundaries(N, M, E):
    """belief_pairs_table_kernel, both templates: non-FAST with injected uniforms, dumps and reset_prior 0 / 1; FAST with
    device Philox and partner modes only.  N % 4 == 0 stages the others' actions by words, other N by bytes."""
    _pairs_case(N, M, E, "injected").require(f"table N={N} M={M} injected", half=1, half_even=int(M != 2), op_order=int(M != 2), fall=1, refine=int(M != 2), first=int(M != 2), outside=int(M != 2), eq=1, ulp=1,
                                            zero=1, near1=1, **{"d1e-12": 1, "d1e-7": 1, "d1e-6": 1, "d9e-6": 1, "d1.1e-5": 1})
    _pairs_case(N, M, E, "injected", reset=True, seed=2).require(f"table N={N} M={M} injected reset", eq=1, ulp=1, **{"d9e-6": 1})
    _pairs_case(N, M, E, "philox", seed=1).require(f"table N={N} M={M} philox FAST", half=1, first=int(M != 2),
                                                  philox_split=int(M != 2))


@pytest.mark.gpu
@pytest.mark.parametrize("N,E", [(34, 20), (36, 20), (131, 3)])
def test_table_kernel_flagged_last_record_of_a_hanging_quad(N, E):
    """K % 4 != 0: the last quad of each row hangs over the end and re-reads the row's last record into its padding slots.
    With that last record on an exact tie, the padding copies are flagged too; they must not be queued, stored or counted."""
    rng = np.random.RandomState(N)
    K, M = N - 1, 3
    assert K % 4 != 0
    fa = np.broadcast_to(DECIMAL_MODELS[M], (N, M, 3)).copy()
    states, _, bands, _ = catalog(DECIMAL_MODELS[M])
    s = next(a for a in range(3) if (bands[a] == "half_even").any())
    act = np.full((E, N), s, dtype=np.uint8)
    tie = np.flatnonzero(bands[s] == "half_even")
    clear = np.flatnonzero(bands[s] == "clear")
    prior = states[clear[rng.randint(len(clear), size=(E, N, K))]]
    prior[:, :, K - 1] = states[tie[rng.randint(len(tie), size=(E, N))]]
    u = rng.rand(E, N, K)
    Bands(*record_views(fa, act, prior, u)).require(f"hanging quad N={N}", half_even=E * N)
    for form_u, dumps in ((u, True), (None, False)):
        rec, pred, bel, part = _run_pairs(fa, act, prior, form_u, False, dumps, 5, 1, 2, 0)
        uu = u if form_u is not None else P.belief_uniforms(5, 1, 2, belief_rows(E, N, 0), K)
        ap, post = pairs_oracle(fa, act, prior, uu)
        assert_records(rec, M, ap, post)
        assert np.array_equal(part, mode3(ap))
        if dumps:
            assert np.array_equal(pred, ap) and np.array_equal(bel, post)


# ------------------------------------------------------------------------------------------------ GPU: the exact queue overflows
def _overflow_inputs(N, M, targets, rng):
    """Blocks of belief_pairs_table_kernel (envs_per_block = min(64, 16384 // K) envs of one agent) with chosen numbers of
    records that the fp32 screen must flag: a flagged record holds a prior whose posterior lies within 3e-5 of a
    half-integer (the screen's fp32 error is below 6e-5, its window 1e-4), every other record lies 3e-4 or more from every
    half-integer and far from every CDF boundary, both with its injected u (the middle of its action's interval) and with
    the device Philox u of the FAST call (3e-5 or more from c_0 and c_1; a record whose Philox u lies above 1 - 3e-5 is
    one of the flagged ones), so the two templates flag the same records.  -> (..., u injected, u Philox, ...).  In blocks
    whose every record is flagged, each env's predicted actions are 13 / 12 / 10 (action 2 / 1 / 0 at K = 35): the partner
    mode is action 2 only when every record is counted."""
    K = N - 1
    EC = min(64, 16384 // K)
    E = EC * len(targets)
    fa = np.broadcast_to(DECIMAL_MODELS[M], (N, M, 3)).copy()
    states, _, _, cvals = catalog(DECIMAL_MODELS[M])
    s_act = 1
    act = np.full((E, N), s_act, dtype=np.uint8)
    x64, _ = fp64_sequence(np.broadcast_to(DECIMAL_MODELS[M], (len(states), M, 3)), states, np.full(len(states), s_act))
    dist = np.array([min(float(abs(x - (x.numerator // x.denominator) - _HALF)) for x in exact(DECIMAL_MODELS[M], st, s_act)[0])
                     if np.min(np.abs(x64[r] - np.floor(x64[r]) - 0.5)) < 1e-3 else 1.0 for r, st in enumerate(states)])
    c = cvals[s_act]
    width = np.min(np.diff(np.concatenate([np.zeros((len(states), 1)), c], axis=1)), axis=1)
    flag_pool = np.flatnonzero(dist < 3e-5)
    clear_pool = np.flatnonzero((dist >= 3e-4) & (width > 1e-3))
    assert len(flag_pool) >= 2 and len(clear_pool) >= 10, (len(flag_pool), len(clear_pool))
    u_philox = P.belief_uniforms(9, 2, 4, belief_rows(E, N, 0), K)
    near1 = u_philox > 1.0 - 3e-5
    flagged = np.zeros((E, N, K), dtype=bool)
    for b, n in enumerate(targets):
        for i in range(N):
            must = np.flatnonzero(near1[b * EC:(b + 1) * EC, i].reshape(-1))
            rest = np.setdiff1d(np.arange(EC * K), must)
            cells = np.concatenate([must, rng.choice(rest, n - len(must), replace=False)])
            flagged[b * EC + cells // K, i, cells % K] = True
    choice = clear_pool[rng.randint(len(clear_pool), size=(E, N, K))]
    for _ in range(100):   # redraw the clear records whose c_0 or c_1 lies near their Philox u
        bad = ~flagged & (np.abs(c[choice][..., :2] - u_philox[..., None]).min(-1) < 3e-5)
        if not bad.any():
            break
        choice[bad] = clear_pool[rng.randint(len(clear_pool), size=int(bad.sum()))]
    assert not bad.any()
    choice[flagged] = flag_pool[rng.randint(len(flag_pool), size=int(flagged.sum()))]
    prior = states[choice]
    want = rng.randint(0, 3, size=(E, N, K))
    full = [b for b, n in enumerate(targets) if n == EC * K]
    if K == 35:
        for b in full:
            pattern = np.array([2] * 13 + [1] * 12 + [0] * 10)
            for e in range(b * EC, (b + 1) * EC):
                for i in range(N):
                    want[e, i] = rng.permutation(pattern)
    cc = c[choice]
    lo = np.where(want == 0, 0.0, np.take_along_axis(cc, np.maximum(want - 1, 0)[..., None], -1)[..., 0])
    hi = np.take_along_axis(cc, want[..., None], -1)[..., 0]
    u = 0.5 * (lo + hi)
    return fa, act, prior, u, u_philox, flagged, EC


@pytest.mark.gpu
@pytest.mark.parametrize("N,M", [(36, 3), (36, 5)])
def test_table_kernel_exact_queue_overflow(N, M):
    """Blocks with exactly 1024 flagged records (the queue fills), 1025 (one record computed inline) and every record
    flagged (more than 2048: over half inline), both templates, against the oracle; the partner modes of the full blocks
    count every inline record."""
    rng = np.random.RandomState(N + M)
    K = N - 1
    targets = (1024, 1025, min(64, 16384 // K) * K)
    fa, act, prior, u, uu, flagged, EC = _overflow_inputs(N, M, targets, rng)
    per_block = flagged.reshape(len(targets), EC, N, K).sum(axis=(1, 3))   # [env block, agent]
    print(f"\n[overflow N={N} M={M}] envs_per_block={EC} records_per_block={EC * K} flagged per block: "
          + ", ".join(sorted({str(v) for v in per_block.reshape(-1)})))
    assert (per_block == np.array(targets)[:, None]).all() and targets[2] > 2048
    bands = Bands(*record_views(fa, act, prior, u))
    rb = np.array(bands.rounding).reshape(flagged.shape)
    assert np.isin(rb[flagged], ("half_even", "half_odd", "op_order", "refine", "first")).all() and (rb[~flagged] == "clear").all()
    assert bands.counts["far"] == flagged.size
    rec, pred, bel, part = _run_pairs(fa, act, prior, u, False, True, 9, 2, 4, 0)
    ap, post = pairs_oracle(fa, act, prior, u)
    assert_records(rec, M, ap, post)
    assert np.array_equal(pred, ap) and np.array_equal(bel, post) and np.array_equal(part, mode3(ap))
    if K == 35:
        assert (part[2 * EC:] == 2).all()
    # FAST: device Philox, the same flagged records
    _, c64 = fp64_sequence(*record_views(fa, act, prior)[:3])
    c64 = c64.reshape(flagged.shape + (3,))
    assert (np.abs(c64[..., :2] - uu[..., None]).min(-1)[~flagged] >= 3e-5).all() and not (uu[~flagged] > 1 - 3e-5).any()
    rec, _, _, part = _run_pairs(fa, act, prior, None, False, False, 9, 2, 4, 0)
    ap, post = pairs_oracle(fa, act, prior, uu)
    assert_records(rec, M, ap, post)
    assert np.array_equal(part, mode3(ap))


# ------------------------------------------------------------------------------------------------ GPU: the episode kernel
def _run_episode(fa, act, u, seed, episode, env_offset):
    """One ia2c_belief_update_pairs_episode call from the uniform prior; u None -> the FAST template (device Philox, no dumps)."""
    import torch
    from ia2c_b200 import _lib
    from tests.helpers import dev
    lib = _lib.load()
    T1, E, N = act.shape
    K, M = N - 1, fa.shape[1]
    z = lambda *shape: torch.zeros(*shape, dtype=torch.uint8, device="cuda")
    fa_d, act_d = dev(fa), dev(act)
    rec, part = z(E, N, K, 8) + 0xA5, z(T1, E, N)
    if u is not None:
        u_d, pred, bel = dev(u), z(T1, E, N, K), z(T1, E, N, K, M)
        _lib.check(lib.ia2c_belief_update_pairs_episode(_lib.ptr(rec), _lib.ptr(fa_d), _lib.ptr(act_d), _lib.ptr(u_d), _lib.ptr(pred),
                                                        _lib.ptr(bel), _lib.ptr(part), E, N, M, T1, seed, episode, env_offset,
                                                        _lib.stream_ptr()))
    else:
        pred = bel = None
        _lib.check(lib.ia2c_belief_update_pairs_episode(_lib.ptr(rec), _lib.ptr(fa_d), _lib.ptr(act_d), None, None, None, _lib.ptr(part),
                                                        E, N, M, T1, seed, episode, env_offset, _lib.stream_ptr()))
    torch.cuda.synchronize()
    return host(rec), None if pred is None else host(pred), None if bel is None else host(bel), host(part)


def _episode_tape(fa, T1, rng, bands_wanted):
    """An action tape that, played by every agent, leads records of model fa into the first of `bands_wanted` it can reach
    within T1 steps: a catalog path to a state plus the seen action that puts its posterior there, padded with random
    actions.  -> (tape, band)"""
    states, paths, bands, _ = catalog(fa, depth=T1 - 1)
    for b in bands_wanted:
        pool = [paths[tuple(int(v) for v in states[s])] + (a,) for a in range(3) for s in np.flatnonzero(bands[a] == b)]
        pool = [p for p in pool if len(p) <= T1]
        if pool:
            p = pool[rng.randint(len(pool))]
            return np.concatenate([p, rng.randint(0, 3, size=T1 - len(p))]).astype(np.uint8), b
    raise AssertionError(f"no tape reaches {bands_wanted}")


EPISODE_SHAPES = [(9, 4), (12, 3), (36, 4), (64, 5), (65, 6), (130, 3), (256, 5), (512, 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("N,M", EPISODE_SHAPES)
def test_episode_kernel_against_the_oracle_at_every_step(N, M):
    """belief_pairs_episode_kernel compared with the oracle directly: every step's predictions, posteriors and partner modes
    and the final records, both templates.  A warp of the kernel owns 128 // ceil(K / 4) whole envs; the envs of the first
    warp all play one tape that reaches an exact half, so that every lane enters the exact pass in the same step, those of
    the second warp one that reaches the second-level band, and the third warp's agents play random actions.  Every fifth
    agent holds a random model."""
    rng = np.random.RandomState(N * 10 + M)
    K, T1 = N - 1, 10
    epw = max(1, 128 // ((K + 3) // 4))
    E = 3 * epw
    fa = np.broadcast_to(DECIMAL_MODELS[M], (N, M, 3)).copy()
    fa[2::5] = random_models(1, M, N)[0]
    act = rng.randint(0, 3, size=(T1, E, N)).astype(np.uint8)
    tape, _ = _episode_tape(DECIMAL_MODELS[M], T1, rng, ("half_even", "half_odd"))
    act[:, :epw] = tape[:, None, None]
    tape, band2 = _episode_tape(DECIMAL_MODELS[M], T1, rng, ("refine", "op_order", "first"))
    act[:, epw:2 * epw] = tape[:, None, None]
    seed, episode, env_offset = 0xB0B + N, 6, 0
    for form in ("injected", "philox"):
        prior = np.broadcast_to(B.to_hundredths(B.uniform_prior(1, M)[0]), (E, N, K, M)).copy()
        u = np.empty((T1, E, N, K))
        steps, bands = [], None
        for t in range(T1):
            if form == "injected":
                fa_r, k_r, s_r, _ = record_views(fa, act[t], prior)
                u[t] = boundary_uniforms(rng, fa_r, k_r, s_r, share=0.5).reshape(E, N, K)
            else:
                u[t] = P.belief_uniforms(seed, episode, t, belief_rows(E, N, env_offset), K)
            b = Bands(*record_views(fa, act[t], prior, u[t]), philox=form == "philox")
            bands = b if bands is None else bands.merge(b)
            ap, post = pairs_oracle(fa, act[t], prior, u[t])
            steps.append((ap, post))
            prior = post
        bands.require(f"episode N={N} M={M} {form}", half=1, **{band2: epw * (N - 1)}, **({"eq": 1, "d9e-6": 1} if form == "injected" else {}))
        rec, pred, bel, part = _run_episode(fa, act, u if form == "injected" else None, seed, episode, env_offset)
        for t, (ap, post) in enumerate(steps):
            if pred is not None:
                assert np.array_equal(pred[t], ap), f"step {t}: predicted actions"
                assert np.array_equal(bel[t], post), f"step {t}: posteriors"
            assert np.array_equal(part[t], mode3(ap)), f"step {t}: partner modes"
        assert_records(rec, M, *steps[-1])


# ------------------------------------------------------------------------------------------------ GPU: trainers
# Models on which an agent that sees the others play action 0 at every step reaches an exact fp64 half within three updates.
# Found like DECIMAL_MODELS with RandomState(100 + M), constant seen action 0 and depth 4 (M = 2 has none in 20000 draws).
CONSTANT_TIE_MODELS = {
    3: np.array([[4, 4, 12], [9, 6, 5], [7, 6, 7]]) / 20.0,
    4: np.array([[12, 6, 2], [17, 1, 2], [1, 1, 18], [10, 6, 4]]) / 20.0,
    5: np.array([[3, 10, 7], [1, 16, 3], [15, 3, 2], [7, 8, 5], [9, 2, 9]]) / 20.0,
    6: np.array([[2, 10, 8], [5, 9, 6], [4, 4, 12], [7, 9, 4], [8, 11, 1], [14, 3, 3]]) / 20.0,
}


def episode_bands(fa, act, u, philox=False):
    """Band counts over every record and step of an episode (act [T1,E,N], u [T1,E,N,K]) from the uniform prior."""
    T1, E, N = act.shape
    M = fa.shape[1]
    prior = np.broadcast_to(B.to_hundredths(B.uniform_prior(1, M)[0]), (E, N, N - 1, M)).copy()
    bands = None
    for t in range(T1):
        b = Bands(*record_views(fa, act[t], prior, u[t]), philox=philox)
        bands = b if bands is None else bands.merge(b)
        prior = pairs_oracle(fa, act[t], prior, u[t])[1]
    return bands


def tie_init(N, M, seed):
    """reference_init nets whose actors all play action 0: W3 of scale 0.05 and logit gaps of 25 or more, so the fp32 q of
    action 0 rounds to 1 and the 24-bit inverse-CDF sampler draws it for every u; every agent holds the constant-tie model.
    The trainers run with beta = 0 (SATURATED_HP): every policy-gradient term of such a row is zero through the clamp in fp32
    and fp64 alike, while the entropy term is a product with 1 - q, which fp32 rounds to 0 and fp64 keeps at ~1e-11, so the
    1e-5 comparison of actor gradients would measure that rounding and not the kernels."""
    from ia2c_b200.trainer import reference_init
    from tests.test_gpu_saturated_policies import H, w3_offset
    actor, critic, _ = reference_init(N, M, seed=seed)
    actor = np.array(actor, dtype=np.float32).copy()
    rng = np.random.RandomState(seed)
    w3 = w3_offset(6)
    for n in range(N):
        actor[n, w3:w3 + H * 3] = rng.uniform(-0.05, 0.05, H * 3)
        actor[n, w3 + H * 3:w3 + H * 3 + 3] = [0.0, -25.0 - 4.0 * rng.rand(), -25.0 - 4.0 * rng.rand()]
    return actor, critic, np.broadcast_to(CONSTANT_TIE_MODELS[M], (N, M, 3)).copy()


SATURATED_HP = dict(gamma=0.9, beta=0.0, lr_actor=0.0001, lr_critic=0.0002)
# id: (N, M, E, T, kernel path, trainer options); the actor kernel is the default one (pipelined above 64 agents)
TRAINER_CASES = {
    "fused-2-M3": (2, 3, 512, 30, "fused", {}),
    "fused-2-M5": (2, 5, 512, 30, "fused", {}),
    "fused-5": (5, 5, 64, 12, "fused", {}),
    "fused-8": (8, 5, 33, 12, "fused", {}),
    "step-4-M4": (4, 4, 64, 12, "step", {}),
    "many-12": (12, 4, 64, 8, "many", {}),
    "many-36": (36, 6, 16, 6, "many", {}),
    "many-130": (130, 3, 3, 4, "many", {}),
    # 64 envs per block of the per-step table kernel, all on the same tie: 2240 flagged records per block
    "table-36": (36, 5, 192, 4, "table", dict(belief_kernel="step")),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(TRAINER_CASES))
def test_trainer_at_ties(case):
    """A trainer in Philox mode whose agents all play action 0: every belief record of every env reaches an exact fp64 half in
    the same step.  The episode against the oracle (check_episode: trajectory, partner modes and final records bit for bit,
    the rest within 1e-5)."""
    import torch
    from ia2c_b200.trainer import IA2CTrainer
    from tests.test_gpu_trainer_oracle_scale import assert_path, buffers, check_episodes
    N, M, E, T, path, kw = TRAINER_CASES[case]
    seed = 500 + N + M
    tr = IA2CTrainer(E, n_agents=N, n_models=M, steps_per_episode=T, max_episode_steps=T, seed=seed, init=tie_init(N, M, seed),
                     **SATURATED_HP, **kw)
    assert_path(tr, N, M, path, "pipe" if N > 64 else "columns")
    check_episodes(tr, [(buffers(tr), seed, SATURATED_HP)], 1, E, N, M, T, T)
    torch.cuda.synchronize()
    act = host(tr.act)
    assert not act.any(), "a saturated actor played an action other than 0"
    idx = belief_rows(E, N, 0)
    u = np.stack([P.belief_uniforms(seed, 0, t, idx, N - 1) for t in range(T + 1)])
    fa = host(tr.filter_action)
    episode_bands(fa, act, u, philox=True).require(f"trainer {case}", half=E * N * (N - 1))


@pytest.mark.gpu
@pytest.mark.parametrize("path, N, M, E, T, kw", [("fused", 2, 5, 64, 12, {}), ("fused", 8, 5, 9, 6, {}), ("step", 4, 4, 32, 8, {}),
                                                  ("many", 12, 4, 16, 6, {}), ("table", 36, 5, 4, 4, dict(belief_kernel="step"))])
def test_trainer_injected_at_boundaries(path, N, M, E, T, kw):
    """One injected episode per rollout path (dumps): even envs play action 0 throughout (exact halves), odd envs random
    actions, and the belief uniforms sit on the CDF boundaries of each step's oracle prediction.  Against the oracle with
    tests/test_gpu_trainer.py's comparison (every step's predictions and posteriors bit for bit)."""
    from ia2c_b200.trainer import IA2CTrainer
    from oracle import loops as L
    from tests.test_gpu_trainer import _compare_with_oracle
    from tests.test_gpu_trainer_oracle_scale import assert_path
    rng = np.random.RandomState(N * 7 + M)
    actor, critic, fa = tie_init(N, M, seed=N)
    K = N - 1
    actions = rng.randint(0, 3, size=(T + 1, E, N))
    actions[:, ::2] = 0
    prior = np.broadcast_to(B.to_hundredths(B.uniform_prior(1, M)[0]), (E, N, K, M)).copy()
    u = np.empty((T + 1, E, N, K))
    for t in range(T + 1):   # the posteriors do not depend on u: place each step's u on that step's boundaries
        fa_r, k_r, s_r, _ = record_views(fa, actions[t], prior)
        u[t] = boundary_uniforms(rng, fa_r, k_r, s_r).reshape(E, N, K)
        prior = pairs_oracle(fa, actions[t], prior, u[t])[1]
    episode_bands(fa, actions, u).require(f"trainer injected {path} N={N} M={M}", half=1, eq=1, ulp=1, zero=1, near1=1,
                                          **{"d1e-7": 1, "d9e-6": 1, "d1.1e-5": 1})
    st = L.IA2CState(actor=actor.astype(np.float64), critic=critic.astype(np.float64), filter_action=fa, T=T, max_episode_steps=T,
                     beta=0.0)
    tr = IA2CTrainer(E, n_agents=N, n_models=M, steps_per_episode=T, max_episode_steps=T, init=(actor, critic, fa), dumps=True,
                     **SATURATED_HP, **kw)
    assert_path(tr, N, M, path, "columns")
    tr.inject(actions=actions, u_belief=u)
    tr.train_episode(sync_stats=True)
    traj, upd = L.ia2c_episode(st, E, actions=actions, u_belief=u)
    _compare_with_oracle(tr, st, traj, upd, N)


@pytest.mark.gpu
def test_runs_many_at_ties():
    """IA2CRunsMany (belief_pairs_episode_kernel's RUNS instantiation), runs whose agents all play action 0: each run against
    the oracle and byte for byte against a standalone trainer with its seed and init."""
    import torch
    from ia2c_b200.runs import IA2CRunsMany
    from ia2c_b200.trainer import IA2CTrainer
    from tests.test_gpu_runs import assert_run_equals
    from tests.test_gpu_trainer_oracle_scale import buffers, check_episode, oracle_state
    N, M, E, T = 12, 4, 32, 8
    seeds = [21, 2 ** 40 + 5]
    init = [tie_init(N, M, seed=r) for r in range(len(seeds))]
    batch = IA2CRunsMany(E, seeds, n_agents=N, n_models=M, steps_per_episode=T, max_episode_steps=T, init=init,
                         **{k: [v] * len(seeds) for k, v in SATURATED_HP.items()})
    alone = [IA2CTrainer(E, n_agents=N, n_models=M, steps_per_episode=T, max_episode_steps=T, seed=s, init=i, actor_kernel="columns",
                         **SATURATED_HP) for s, i in zip(seeds, init)]
    subjects = [buffers(batch, r) for r in range(len(seeds))]
    states = [oracle_state(b, SATURATED_HP, T, T) for b in subjects]
    batch.train_episode()
    for tr in alone:
        tr.train_episode()
    torch.cuda.synchronize()
    for r, (b, st) in enumerate(zip(subjects, states)):
        check_episode(b, st, seeds[r], 0, E, N, M, T, env_offset=getattr(batch, "env_offset", 0))
        assert_run_equals(batch, r, alone[r])
        act = host(b["act"])
        assert not act.any()
        u = np.stack([P.belief_uniforms(seeds[r], 0, t, belief_rows(E, N, 0), N - 1) for t in range(T + 1)])
        episode_bands(host(b["filter_action"]), act, u, philox=True).require(f"runs-many run {r}", half=E * N * (N - 1))
