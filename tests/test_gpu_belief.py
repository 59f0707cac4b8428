"""GPU parity: belief-filter kernels vs golden vectors of the real class and vs the oracle.  Bit-exact."""
import numpy as np
import pytest

from oracle import belief as B
from oracle import philox as P
from oracle.loops import mode3, others_of
from tests.helpers import dev, dptr, host

pytestmark = pytest.mark.gpu


def _dense(fa, lik, prev, u):
    import torch
    from ia2c_b200 import _lib
    lib = _lib.load()
    R, A = lik.shape
    M = prev.shape[1]
    ap = torch.empty(R, dtype=torch.int64, device="cuda")
    bp = torch.empty(R, M, dtype=torch.float64, device="cuda")
    pred = torch.empty(R, A, dtype=torch.float64, device="cuda")
    _lib.check(lib.ia2c_belief_update_dense(dptr((fa)), dptr((lik)), dptr((prev)), dptr((u.reshape(-1))),
                                            _lib.ptr(ap), _lib.ptr(bp), _lib.ptr(pred), R, M, A, _lib.stream_ptr()))
    return host(ap), host(bp), host(pred)


@pytest.mark.parametrize("tag", ["rand5", "rand3", "rand5x5", "org_known", "hvt_known"])
def test_dense_vs_golden_and_oracle(golden, tag):
    g = golden("belief_vectors.npz")
    fa = g[f"{tag}/filterAction"]
    for t in range(g[f"{tag}/obs"].shape[0]):
        lik, prev, u = g[f"{tag}/obs"][t], g[f"{tag}/prev"][t], g[f"{tag}/u"][t]
        ap, bp, pred = _dense(fa, lik, prev, u)
        assert np.array_equal(bp, g[f"{tag}/bprime"][t])                    # vs the real class: bit-exact
        assert np.array_equal(ap, g[f"{tag}/ap"][t])
        np.testing.assert_allclose(pred, g[f"{tag}/prediction"][t], rtol=2e-15, atol=0)
        oap, obp, opred = B.belief_update(fa, lik, prev, u)
        assert np.array_equal(pred, opred) and np.array_equal(ap, oap)      # vs the oracle: bit-exact incl. prediction


def test_dense_generic_dims_and_ragged_rows():
    rng = np.random.RandomState(0)
    for M, A, R in ((2, 2, 1), (4, 3, 257), (7, 8, 1000), (8, 2, 33)):
        fa = rng.rand(M, A)
        fa /= fa.sum(1, keepdims=True)
        prev = np.rint(rng.dirichlet(np.ones(M), R) * 100) / 100
        lik = rng.rand(R, A)
        u = rng.rand(R)
        ap, bp, pred = _dense(fa, lik, prev, u)
        oap, obp, opred = B.belief_update(fa, lik, prev, u)
        assert np.array_equal(bp, obp) and np.array_equal(ap, oap) and np.array_equal(pred, opred)


def test_class_api_consumes_numpy_stream_like_reference(golden):
    from ia2c_b200.belief import BeliefFilter
    g = golden("belief_vectors.npz")
    np.random.seed(11)
    bf = BeliefFilter(5, 3, 256)
    assert np.array_equal(bf.filterAction, g["rand5/filterAction"]) and np.array_equal(bf.prior, g["rand5/prior0"])
    assert np.array_equal(bf.filters, bf.filterAction.T)
    real_rand = np.random.rand
    for t in range(10):
        tape = g["rand5/u"][t]
        np.random.rand = lambda *shape: tape.copy()
        try:
            ap, bprime, pred = bf.update(g["rand5/obs"][t], g["rand5/prev"][t])
        finally:
            np.random.rand = real_rand
        assert ap.dtype == np.int64 and np.array_equal(ap, g["rand5/ap"][t]) and np.array_equal(bprime, g["rand5/bprime"][t])
    known = BeliefFilter(3, 3, 64, known="org")
    assert np.array_equal(known.filterAction, g["org_known/filterAction"])


def _pairs_oracle(fa, act, prior, u):
    """act [E,N]; prior [E,N,K,M]; u [E,N,K] -> ap [E,N,K], bprime [E,N,K,M] via the oracle."""
    E, N = act.shape
    K = N - 1
    ap = np.zeros((E, N, K), dtype=np.int64)
    bp = np.zeros_like(prior)
    M = prior.shape[-1]
    for i in range(N):   # one oracle call per agent: its K modelled others x E envs are independent rows sharing the agent's models
        others = np.asarray(list(others_of(i, N)))
        a, b, _ = B.belief_update(fa[i], B.likelihood_from_action(act[:, others].reshape(-1), 3), prior[:, i].reshape(-1, M), u[:, i].reshape(-1))
        ap[:, i], bp[:, i] = a.reshape(E, K), b.reshape(E, K, M)
    return ap, bp


@pytest.mark.parametrize("E,N,M", [(1, 2, 5), (37, 2, 5), (300, 3, 5), (9, 5, 3), (5, 64, 5), (2, 256, 5), (3, 7, 6), (4, 6, 2), (3, 65, 5), (70, 33, 5), (40, 130, 5),
                                   (2, 600, 5), (1, 1023, 3)])   # N > 512: only the per-step kernel exists
def test_pairs_kernel_vs_oracle(E, N, M):
    import torch
    from ia2c_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(E + N)
    K = N - 1
    fa = rng.rand(N, M, 3)
    fa /= fa.sum(-1, keepdims=True)
    rec = torch.zeros(E, N, K, 8, dtype=torch.uint8, device="cuda")
    prior = np.tile(B.uniform_prior(1, M)[0], (E, N, K, 1))
    for t in range(6):
        act = rng.randint(0, 3, size=(E, N)).astype(np.uint8)
        injected = t % 2 == 0
        if injected:
            u = rng.rand(E, N, K)
        else:
            u = P.belief_uniforms(77, 5, t, (np.arange(E)[:, None] + 1000) * N + np.arange(N)[None, :], K)
        pred = torch.empty(E, N, K, dtype=torch.uint8, device="cuda")
        bel = torch.empty(E, N, K, M, dtype=torch.uint8, device="cuda")
        partner = torch.empty(E, N, dtype=torch.uint8, device="cuda")
        _lib.check(lib.ia2c_belief_update_pairs(_lib.ptr(rec), dptr((fa)), dptr((act)), dptr((u)) if injected else None,
                                                _lib.ptr(pred), _lib.ptr(bel), _lib.ptr(partner), E, N, M, int(t == 0), 77, 5, t, 1000,
                                                _lib.stream_ptr()))
        oap, obp = _pairs_oracle(fa, act, prior, u)
        assert np.array_equal(host(pred), oap)
        assert np.array_equal(host(bel), B.to_hundredths(obp))
        assert np.array_equal(host(rec)[..., :M], B.to_hundredths(obp)) and np.array_equal(host(rec)[..., 6], oap)
        assert np.array_equal(host(partner), mode3(oap))
        prior = obp


def test_pairs_fast_path_vs_oracle_at_scale():
    """The steady-state template of the many-agent kernel (device Philox, no dumps: FAST) on 1.5 M records per step against the
    oracle: every stored posterior byte and every predicted action — i.e. every fp32-screened decision and every record deferred
    to the exact pass — must equal the reference's fp64 sequence."""
    import torch
    from ia2c_b200 import _lib
    lib = _lib.load()
    E, N, M = 96, 128, 5
    K = N - 1
    rng = np.random.RandomState(5)
    fa = rng.rand(N, M, 3)
    fa /= fa.sum(-1, keepdims=True)
    rec = torch.zeros(E, N, K, 8, dtype=torch.uint8, device="cuda")
    partner = torch.empty(E, N, dtype=torch.uint8, device="cuda")
    fa_d = dev(fa)
    prior = np.tile(B.uniform_prior(1, M)[0], (E, N, K, 1))
    rows = (np.arange(E)[:, None] + 7) * N + np.arange(N)[None, :]
    for t in range(4):
        act = rng.randint(0, 3, size=(E, N)).astype(np.uint8)
        if t == 0:   # start from the uniform prior through the non-FAST template (reset), then three FAST steps
            u = P.belief_uniforms(3, 9, t, rows, K)
            _lib.check(lib.ia2c_belief_update_pairs(_lib.ptr(rec), _lib.ptr(fa_d), dptr(act), None, None, None, _lib.ptr(partner), E, N, M, 1,
                                                    3, 9, t, 7, _lib.stream_ptr()))
        else:
            u = P.belief_uniforms(3, 9, t, rows, K)
            _lib.check(lib.ia2c_belief_update_pairs(_lib.ptr(rec), _lib.ptr(fa_d), dptr(act), None, None, None, _lib.ptr(partner), E, N, M, 0,
                                                    3, 9, t, 7, _lib.stream_ptr()))
        oap, obp = _pairs_oracle(fa, act, prior, u)
        r = host(rec)
        assert np.array_equal(r[..., :M], B.to_hundredths(obp)) and np.array_equal(r[..., 6], oap) and not r[..., 7].any()
        assert np.array_equal(host(partner), mode3(oap))
        prior = obp


@pytest.mark.parametrize("E,N,M,T1,injected", [(5, 36, 5, 6, True), (40, 64, 5, 5, False), (3, 132, 5, 4, True), (17, 256, 5, 4, False),
                                               (70, 36, 3, 5, False), (2, 512, 5, 2, False), (9, 260, 5, 3, False),
                                               (50, 12, 5, 4, False), (7, 16, 5, 3, True), (33, 32, 3, 4, False), (300, 20, 5, 5, False),
                                               # N % 4 != 0: byte-wise staging of the others' actions
                                               (11, 65, 5, 3, False), (4, 130, 5, 3, True), (60, 10, 5, 4, False), (5, 33, 3, 3, False), (3, 511, 5, 2, False)])
def test_episode_kernel_equals_the_per_step_kernel(E, N, M, T1, injected):
    """ia2c_belief_update_pairs_episode (records resident on the SM for the whole episode, every warp on its own) against T1 calls of the per-step
    kernel, which the oracle tests above pin: records, per-step predictions, per-step posteriors and partner modes, byte for byte."""
    import torch
    from ia2c_b200 import _lib
    lib = _lib.load()
    assert lib.ia2c_belief_supports_episode(N, M) == 1 and lib.ia2c_belief_supports_episode(516, 5) == 0 and lib.ia2c_belief_supports_episode(8, 5) == 0
    rng = np.random.RandomState(E * 7 + N)
    K = N - 1
    fa = rng.rand(N, M, 3)
    fa /= fa.sum(-1, keepdims=True)
    fa_d = dev(fa)
    act = dev(rng.randint(0, 3, size=(T1, E, N)).astype(np.uint8))
    u = dev(rng.rand(T1, E, N, K)) if injected else None
    z = lambda *shape: torch.zeros(*shape, dtype=torch.uint8, device="cuda")
    rec_s, pred_s, bel_s, part_s = z(E, N, K, 8), z(T1, E, N, K), z(T1, E, N, K, M), z(T1, E, N)
    for t in range(T1):
        _lib.check(lib.ia2c_belief_update_pairs(_lib.ptr(rec_s), _lib.ptr(fa_d), _lib.ptr(act[t]), _lib.ptr(u[t]) if injected else None,
                                                _lib.ptr(pred_s[t]), _lib.ptr(bel_s[t]), _lib.ptr(part_s[t]), E, N, M, int(t == 0), 21, 4, t, 100,
                                                _lib.stream_ptr()))
    rec_e, pred_e, bel_e, part_e = z(E, N, K, 8) + 7, z(T1, E, N, K), z(T1, E, N, K, M), z(T1, E, N)
    _lib.check(lib.ia2c_belief_update_pairs_episode(_lib.ptr(rec_e), _lib.ptr(fa_d), _lib.ptr(act), _lib.ptr(u) if injected else None,
                                                    _lib.ptr(pred_e), _lib.ptr(bel_e), _lib.ptr(part_e), E, N, M, T1, 21, 4, 100, _lib.stream_ptr()))
    assert torch.equal(part_e, part_s) and torch.equal(pred_e, pred_s) and torch.equal(bel_e, bel_s) and torch.equal(rec_e, rec_s)
    # the steady-state template (no dumps) writes the same records and partner modes
    rec_f, part_f = z(E, N, K, 8), z(T1, E, N)
    if not injected:
        _lib.check(lib.ia2c_belief_update_pairs_episode(_lib.ptr(rec_f), _lib.ptr(fa_d), _lib.ptr(act), None, None, None, _lib.ptr(part_f), E, N, M, T1,
                                                        21, 4, 100, _lib.stream_ptr()))
        assert torch.equal(rec_f, rec_s) and torch.equal(part_f, part_s)
