"""Cross-play on the GPU (ia2c_evaluate_lineups, evaluate_lineups, cross_play): a lineup computes byte for byte what
ia2c_evaluate computes for its gathered actors, the lineup of a run's own agents reproduces the run's evaluation, the
fixed-order statistics equal the oracle's, lineups beyond one grid dimension and out-of-range entries are handled, and the
sources are left untouched."""
import ctypes as C

import numpy as np
import pytest
import torch

from ia2c_b200 import _lib
from oracle import cross_play as XP
from oracle import evaluate as EV
from tests.test_gpu_runs import HYPER, SEEDS

pytestmark = pytest.mark.gpu


def h(t):
    return np.ascontiguousarray(t.detach().cpu().numpy())


def same_bytes(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def random_actors(rows, seed):
    return torch.from_numpy(np.random.RandomState(seed).normal(0.0, 0.6, size=(rows, _lib.ACTOR_P)).astype(np.float32)).cuda()


def lineup_call(pool, N, lineups, E, K, T, mes, greedy=False, seed=0, episode0=0, tape=None):
    """The C call through lineup_desc, every output copied back (returns included)."""
    from ia2c_b200.evaluate import lineup_desc
    lin = torch.as_tensor(np.asarray(lineups, dtype=np.int32)).cuda()
    P, nets = lin.shape[0], pool.shape[0]
    policy = torch.empty((nets, 9, 3), dtype=torch.float32, device="cuda")
    returns = torch.empty((P, K, E), dtype=torch.float64, device="cuda")
    counts = torch.empty((P * N, 3), dtype=torch.int64, device="cuda")
    stats = torch.empty((2, P), dtype=torch.float64, device="cuda")
    tp = torch.as_tensor(tape).cuda() if tape is not None else None
    d = lineup_desc(pool, nets, N, lin, E, K, T, mes, greedy, seed, episode0, policy, returns, counts, stats[0], stats[1], tp)
    _lib.check(_lib.load().ia2c_evaluate_lineups(C.byref(d), _lib.stream_ptr()), "ia2c_evaluate_lineups")
    torch.cuda.synchronize()
    return dict(returns=h(returns), action_counts=h(counts).view(np.uint64).reshape(P, N, 3), return_sum=h(stats[0]),
                return_m2=h(stats[1]), policy=h(policy))


def pseudo_runs(pool, N, lineups, E, K, T, mes, greedy=False, seed=0, episode0=0, tape=None):
    """ia2c_evaluate on the lineups' gathered actors, one pseudo-run per lineup (the tape layouts coincide)."""
    from ia2c_b200.evaluate import evaluate_actors
    idx = torch.as_tensor(np.asarray(lineups, dtype=np.int64).reshape(-1)).cuda()
    return evaluate_actors(pool[idx].contiguous(), len(lineups), N, E, K, T, mes, greedy, seed, episode0, pool.device,
                           u_action=tape)


def random_lineups(P, N, nets, seed):
    rs = np.random.RandomState(seed)
    lin = rs.randint(0, nets, size=(P, N))
    lin[0] = np.arange(N)                  # run 0 in its own seats
    lin[1] = np.arange(N)[::-1]            # run 0 with every seat swapped
    lin[2] = lin[2, 0]                     # one row in every seat
    return lin


@pytest.mark.parametrize("mode", ["philox", "tape", "greedy"])
@pytest.mark.parametrize("N", [2, 5, 8, 9, 64, 130])
def test_lineup_equals_evaluate_on_the_gathered_actors(N, mode):
    nets, P, T, mes, seed = 3 * N, 7, 30, 7, 0xC0FFEE1234
    E, K = (1, 1) if mode == "greedy" else (13, 3)
    pool = random_actors(nets, N)
    lin = random_lineups(P, N, nets, N + 1)
    tape = np.random.RandomState(N).rand(K, T, P * E, N).astype(np.float32) if mode == "tape" else None
    a = lineup_call(pool, N, lin, E, K, T, mes, greedy=mode == "greedy", seed=seed, episode0=5, tape=tape)
    b = pseudo_runs(pool, N, lin, E, K, T, mes, greedy=mode == "greedy", seed=seed, episode0=5, tape=tape)
    assert same_bytes(a["returns"], b["returns"])
    assert same_bytes(a["action_counts"], b["action_counts"])
    assert int(a["action_counts"].sum()) == P * N * E * K * T
    s, m2 = XP.lineup_stats(a["returns"])
    assert same_bytes(a["return_sum"], s) and same_bytes(a["return_m2"], m2)


@pytest.mark.parametrize("N", [2, 9])
def test_identity_lineups_reproduce_each_runs_evaluation(N):
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    cls = IA2CRuns if N <= 8 else IA2CRunsMany
    batch = cls(10, SEEDS, n_agents=N, **HYPER)
    for _ in range(3):
        batch.train_episode()
    R = batch.R
    ident = np.arange(R * N).reshape(R, N)
    for kw in (dict(K=2, seed=9, episode0=4), dict(K=1, greedy=True)):
        E = 1 if kw.get("greedy") else 10
        ev = batch.evaluate(episodes=kw["K"], num_envs=E, greedy=kw.get("greedy", False), seed=kw.get("seed", 0),
                            first_episode=kw.get("episode0", 0))
        a = lineup_call(batch.actor_params, N, ident, E, kw["K"], batch.T, 30, greedy=kw.get("greedy", False),
                        seed=kw.get("seed", 0), episode0=kw.get("episode0", 0))
        assert same_bytes(a["returns"], ev["returns"].reshape(R, kw["K"], E))
        assert same_bytes(a["action_counts"], ev["action_counts"])
    xp = batch.cross_play(episodes=2, seed=9, first_episode=4)
    ev = batch.evaluate(episodes=2, seed=9, first_episode=4)
    assert xp["mean_return"].shape == (R, R) and xp["action_freq"].shape == (R, R, N, 3)
    assert np.allclose(np.diag(xp["mean_return"]), ev["mean_return"], rtol=1e-12, atol=0)
    assert np.allclose(np.diag(xp["std_return"]), ev["std_return"], rtol=1e-12, atol=1e-12)
    assert same_bytes(xp["action_freq"][np.arange(R), np.arange(R)], ev["action_freq"])
    split = N // 2
    assert np.array_equal(xp["lineups"][1 * R + 2], np.r_[np.arange(split) + N, np.arange(split, N) + 2 * N])


@pytest.mark.parametrize("N", [3, 64])
def test_the_whole_call_against_the_oracle_under_a_tape(N):
    nets, P, E, K, T, mes = 2 * N, 5, 7, 2, 30, 11
    pool = random_actors(nets, 5 * N)
    lin = random_lineups(P, N, nets, N)
    tape = np.random.RandomState(3 * N).rand(K, T, P * E, N).astype(np.float32)
    a = lineup_call(pool, N, lin, E, K, T, mes, tape=tape)
    ref = XP.evaluate_lineups(h(pool), lin, E, K, T, mes, u=tape, table=a["policy"])
    for p in range(P):
        assert same_bytes(a["returns"][p], ref[p]["returns"]), p
        assert np.array_equal(a["action_counts"][p], ref[p]["counts"].astype(np.uint64)), p
    assert np.abs(a["policy"] - EV.policy_table(h(pool).astype(np.float64))).max() < 1e-6
    s, m2 = XP.lineup_stats(np.stack([r["returns"] for r in ref]))
    assert same_bytes(a["return_sum"], s) and same_bytes(a["return_m2"], m2)


def test_lineups_beyond_one_grid_dimension():
    N, nets, P = 2, 6, 70000
    pool = random_actors(nets, 1)
    lin = np.random.RandomState(2).randint(0, nets, size=(P, N))
    a = lineup_call(pool, N, lin, 1, 1, 4, 30, seed=5)
    for p in (P - 1, 65535, 65534):
        alone = lineup_call(pool, N, lin[p:p + 1], 1, 1, 4, 30, seed=5)
        for key in ("returns", "action_counts", "return_sum", "return_m2"):
            assert same_bytes(a[key][p:p + 1], alone[key]), (p, key)
    assert int(a["action_counts"].sum()) == P * N * 4


@pytest.mark.parametrize("N", [2, 64])
def test_an_out_of_range_entry_poisons_only_its_lineup(N):
    nets, P, E, K, T = 2 * N, 6, 9, 2, 30
    pool = random_actors(nets, 2)
    lin = random_lineups(P, N, nets, 4)
    bad = lin.copy()
    bad[3, N - 1] = nets
    bad[4, 0] = -1
    a, b = lineup_call(pool, N, bad, E, K, T, 30, seed=1), lineup_call(pool, N, lin, E, K, T, 30, seed=1)
    for p in (3, 4):
        assert np.isnan(a["returns"][p]).all() and np.isnan(a["return_sum"][p]) and np.isnan(a["return_m2"][p])
        assert not a["action_counts"][p].any()
    keep = [0, 1, 2, 5]
    for key in ("returns", "action_counts", "return_sum", "return_m2"):
        assert same_bytes(a[key][keep], b[key][keep]), key
    from ia2c_b200.evaluate import evaluate_lineups
    with pytest.raises(ValueError, match="outside the pool"):
        evaluate_lineups(pool, N, bad, E, K, T, 30, False, 1, 0, pool.device)


def _tensors(obj):
    """Every device tensor an object holds, its hyper-parameter dict and its rings included."""
    out = {}
    for name, v in vars(obj).items():
        if isinstance(v, torch.Tensor) and v.is_cuda:
            out[name] = h(v).view(np.uint8)
        elif isinstance(v, dict):
            out.update({f"{name}.{k}": h(t).view(np.uint8) for k, t in v.items() if isinstance(t, torch.Tensor) and t.is_cuda})
        elif v is not None and hasattr(v, "_dev") and isinstance(v._dev, torch.Tensor):
            out[name + "._dev"] = h(v._dev)
    return out


def test_cross_play_leaves_its_sources_untouched_and_is_deterministic():
    from ia2c_b200.evaluate import cross_play
    from ia2c_b200.runs import IA2CRuns
    from ia2c_b200.trainer import IA2CTrainer
    runs = IA2CRuns(10, SEEDS, **HYPER)
    runs.train_episodes(3)
    runs.exploit_explore(window=2, fraction=0.25)
    runs.train_episodes(1)
    tr = IA2CTrainer(10, seed=5)
    tr.train_episode()
    torch.cuda.synchronize()
    before = {**_tensors(runs), **{"trainer." + k: v for k, v in _tensors(tr).items()}}
    assert "_hyper.lr_actor" in before and "_history._dev" in before
    x1 = runs.cross_play(episodes=2, seed=3)
    x2 = runs.cross_play(episodes=2, seed=3)
    x3 = cross_play([runs, tr], episodes=2, seed=3)
    torch.cuda.synchronize()
    after = {**_tensors(runs), **{"trainer." + k: v for k, v in _tensors(tr).items()}}
    assert before.keys() == after.keys()
    for k in before:
        assert same_bytes(before[k], after[k]), k
    for key in x1:
        assert same_bytes(x1[key], x2[key]), key
    assert same_bytes(x3["mean_return"][:4, :4], x1["mean_return"])


def test_cross_play_across_sources_equals_one_batch():
    from ia2c_b200.evaluate import cross_play
    from ia2c_b200.runs import IA2CRuns
    from ia2c_b200.trainer import IA2CTrainer
    runs = IA2CRuns(10, SEEDS[:3], **{k: v[:3] for k, v in HYPER.items()})
    runs.train_episode()
    tr = IA2CTrainer(10, seed=77)
    tr.train_episode()
    one = IA2CRuns(10, SEEDS)
    one.actor_params[:3 * 2].copy_(runs.actor_params)
    one.actor_params[3 * 2:].copy_(tr.actor_params)
    a = cross_play([runs, tr], episodes=3, seed=8)
    b = one.cross_play(episodes=3, seed=8)
    assert a["mean_return"].shape == (4, 4)
    for key in a:
        assert same_bytes(a[key], b[key]), key
    g = cross_play([runs, tr], greedy=True)
    assert g["mean_return"].shape == (4, 4) and np.all(g["std_return"] == 0.0)
