"""Oracle pin for the recorded statistics: the fixed-order return sum against math.fsum, and the per-episode statistics of
oracle/history.py on the golden reference tapes (counts of the sampled actions, hits of each belief filter's predicted action
against the partner's sampled action, sums of the episode returns)."""
import math

import numpy as np
import pytest

from oracle import history as H


@pytest.mark.parametrize("E", [1, 37, 256, 4097])
def test_fixed_order_sum_against_fsum(E):
    rng = np.random.RandomState(E)
    x = rng.uniform(-100.0, 20.0, size=(3, E)) * rng.choice([1e-3, 1.0, 1e3], size=(3, E))
    s = H.fixed_order_sum(x)
    assert s.shape == (3,)
    for r in range(3):
        ref = math.fsum(x[r])
        assert abs(s[r] - ref) <= 1e-12 * max(abs(ref), np.abs(x[r]).sum() * 1e-3)


def test_fixed_order_sum_is_the_stated_order():
    """The lane sums and the tree written out with Python floats, one addition at a time."""
    rng = np.random.RandomState(7)
    x = rng.randn(600) * 1e6
    lanes = [0.0] * 256
    for e in range(600):
        lanes[e % 256] = lanes[e % 256] + float(x[e])
    w = 128
    while w:
        for j in range(w):
            lanes[j] = lanes[j] + lanes[j + w]
        w //= 2
    assert H.fixed_order_sum(x) == lanes[0]
    assert H.fixed_order_sum(np.zeros(5)) == 0.0 and not np.signbit(H.fixed_order_sum(-np.zeros(5)))


@pytest.mark.parametrize("name", ["ia2c_E10.npz", "ia2c_E64.npz"])
def test_statistics_of_the_golden_tapes(golden, name):
    g = golden(name)
    T, E = int(g["meta_T"]), int(g["meta_n_envs"])
    for ep in range(int(g["meta_episodes"])):
        sl = slice(ep * (T + 1), (ep + 1) * (T + 1))
        a1, a2 = g["act1/sampled"][sl], g["act2/sampled"][sl]                # [T+1, E]
        act = np.stack([a1, a2], axis=-1)
        partner_true = np.stack([a2, a1], axis=-1)                            # N = 2: the partner is the other agent
        partner_pred = np.stack([g["bf0/ap"][sl], g["bf1/ap"][sl]], axis=-1)  # bf0 = agent 1's filter over agent 2
        loss = np.arange(4, dtype=np.float32).reshape(2, 2)
        rec = H.record(act, partner_true, partner_pred, g["reward_lst"][ep], loss, 1, E, 2, T)
        for i, (own, other, f) in enumerate(((a1, a2, "bf0"), (a2, a1, "bf1"))):
            assert rec["action_counts"][i].tolist() == [int((own[:T] == k).sum()) for k in range(3)]
            assert rec["partner_hits"][i] == int((g[f"{f}/ap"][sl][:T] == other[:T]).sum())
        assert rec["action_counts"].sum() == 2 * T * E and rec["action_counts"].dtype == np.uint32
        assert abs(rec["return_sum"][0] - math.fsum(g["reward_lst"][ep])) <= 1e-12 * abs(math.fsum(np.abs(g["reward_lst"][ep])))
        assert np.array_equal(rec["loss"], loss)


def test_record_layout_of_a_batch():
    """R runs stacked on the env axis: run r's rows are the statistics of its own E envs."""
    rng = np.random.RandomState(3)
    R, E, N, T = 3, 5, 4, 6
    act = rng.randint(0, 3, size=(T + 1, R * E, N)).astype(np.uint8)
    pt, pp = rng.randint(0, 3, size=act.shape).astype(np.uint8), rng.randint(0, 3, size=act.shape).astype(np.uint8)
    ret = rng.randn(R * E)
    loss = rng.randn(2, R * N).astype(np.float32)
    rec = H.record(act, pt, pp, ret, loss, R, E, N, T)
    for r in range(R):
        es, ns = slice(r * E, (r + 1) * E), slice(r * N, (r + 1) * N)
        one = H.record(act[:, es], pt[:, es], pp[:, es], ret[es], loss[:, ns], 1, E, N, T)
        assert np.array_equal(rec["action_counts"][ns], one["action_counts"])
        assert np.array_equal(rec["partner_hits"][ns], one["partner_hits"])
        assert rec["return_sum"][r] == one["return_sum"][0]
