"""The class-API kernels against the fp64 oracle at the benchmark's shape and at every dispatch boundary.

The drop-in classes (ac_nets.py users, a2c_test.py, bench cfg3) run three groups of kernels: the single-pass update
(`net_update_dense_kernel` + `net_update_reduce_adam_kernel`, csrc/net_update.cu), the MLP forward / backward / sampler
kernels (csrc/mlp.cu) and the loss and Adam kernels (csrc/loss.cu).  Their boundaries, and what reaches them here:

  single pass     3 tiles of 32 rows in flight per block, grid min(148, tiles): 14208 rows never refill a stage, 14209
                  issue the first refill and wait on parity 1, 28417 wrap the parity back to 0, 65536 (cfg3) and 65553
                  give every block 13-14 uses, the last one a partial tile.  Applicability: rows >= 1024, 64 <= F <= 512,
                  F % 4 == 0, O <= 8, a 16-byte aligned x; the shapes just outside it must take the kernel sequence.
  OMAX buckets    4 / 9 / 32: O = 1, 4, 5, 9, 10, 31, 32.
  row mapping     F < 64 thread per row, F >= 64 warp per row, F = 8192 (opt-in shared memory) at the API limit.
  grid stride     losses and narrow kernels past 592 x 256 = 151552 rows (finish_mean_kernel adds 592 partials), wide
                  kernels past 4736 rows; dW1 chunks: 1024 chunks of 65 rows at 65537 rows, a second B3 round of slices
                  above 256 chunks (16385 rows).
  Adam            pow(b, t) from the device step counter, up to t = 2^30 + 1.

Rules: bytes where a kernel claims bit-identity (index vs dense kernels, fallback shapes with and without
IA2C_NO_SINGLE_PASS, sampled actions given the kernel's own probabilities), rel_err <= 1e-5 against fp64 otherwise.

Conditioning.  The first Adam step is about lr * g / (|g| + 1e-8): an entry whose sign rounding can flip moves by 2 lr,
and the parameter comparison would measure rounding.  `Oracle` computes, next to every gradient Adam sees, the sum of the
absolute values of its terms (the same backward on |W|, |x| and the absolute per-row loss terms); one fp32 rounding of
that sum, 2^-24 * sum|terms|, is the entry's bound, and an entry whose step scale (|g| at the first step, the RMS
sqrt(v / (1 - b2^t)) of its gradients after it) is within 8 x its bound is ill-conditioned.  Every
case asserts it has none and prints its count with the smallest scale / bound.  The post-Adam state is also checked
against a float64 Adam step applied to the kernel's own gradient and moments (1e-6 of the largest entry).  The same
margin, 8 x 2^-24 x sum|terms|, is kept around zero for the pre-activations z1 and z2 (`relu_margins`): the update cases
draw their inputs clear of it, because a ReLU that fp32 and fp64 decide differently moves one row's term."""
import numpy as np
import pytest

from oracle import nets as NN
from oracle import philox as PH
from tests.helpers import dev, host, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-5
H = NN.HIDDEN
U32 = 2.0 ** -24
COND = 8.0                 # ill-conditioned: |g| <= COND * U32 * sum|terms|
LR_C, LR_A, BETA = 5e-4, 1e-4, 0.01
BUCKETS = (1, 4, 5, 9, 10, 31, 32)


# ---------------------------------------------------------------- inputs


def linear_init(F, O, seed):
    """nn.Linear-style uniform(-1/sqrt(fan_in), 1/sqrt(fan_in)) parameters of an F -> 6 -> 6 -> O net."""
    rng = np.random.RandomState(seed)
    parts = []
    for fi, fo in ((F, H), (H, H), (H, O)):
        k = 1.0 / np.sqrt(fi)
        parts += [rng.uniform(-k, k, (fo, fi)), rng.uniform(-k, k, fo)]
    return NN.pack(parts).astype(np.float32)


def make_rows(rng, rows, F, style):
    """float32 rows: 'onehot' (a2c_test.py's one_hot(state, 500)), 'sparse' (one-hot, the first half with ~5 % extra dense
    entries) or 'dense' (every entry non-zero)."""
    if style == "dense":
        return rng.uniform(-1.0, 1.0, (rows, F)).astype(np.float32)
    x = np.zeros((rows, F), dtype=np.float32)
    x[np.arange(rows), rng.randint(0, F, rows)] = 1.0
    if style == "sparse":
        h = rows // 2
        x[:h] += ((rng.rand(h, F) < 0.05) * rng.rand(h, F)).astype(np.float32)
    return x


def one_hot(idx, F):
    x = np.zeros((len(idx), F), dtype=np.float32)
    x[np.arange(len(idx)), idx] = 1.0
    return x


def running_grad(rng, P):
    """The actor's running gradient sum before the first update (never zeroed, Q2): entries of magnitude 0.005..0.015, so
    that no entry of the accumulated gradient starts next to zero."""
    return (np.where(rng.rand(P) < 0.5, -1.0, 1.0) * (0.005 + 0.01 * rng.rand(P))).astype(np.float32)


def signals(rng, kind, rows):
    """Critic targets or actor advantages: 1 + randn.  With a zero mean (bench: randn) the rows' gradient terms cancel
    deeply enough at O <= 8 over fully dense rows that some entries are ill-conditioned (see Conditioning)."""
    return (1.0 + rng.randn(rows)).astype(np.float32)


# ---------------------------------------------------------------- oracle


def adam64(p, m, v, g, t, lr):
    b1, b2 = 0.9, 0.999
    p, m, v, g = (np.asarray(a, np.float64) for a in (p, m, v, g))
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    return p - lr / (1 - b1 ** t) * (m / (np.sqrt(v) / np.sqrt(1 - b2 ** t) + 1e-8)), m, v


def close(devv, ref, tol=1e-6):
    devv, ref = np.asarray(devv, np.float64), np.asarray(ref, np.float64)
    assert np.abs(devv - ref).max() <= tol * np.abs(ref).max()


def abs_terms(kind, flat, x, act, sig, beta, F, O, next_obs=None, next_act=None, gamma_mask=None):
    """sum over rows of |term| for every gradient entry: the oracle's backward on |W|, |x| and the absolute per-row loss
    terms, with the fp64 ReLU masks."""
    B = len(act)
    rows = np.arange(B)
    out, cache = NN.forward(flat, x, F, O, softmax=kind == 1, keep=True)
    xx, z1, h1, z2, h2, y = cache
    dy = np.zeros_like(y)
    if kind == 0:
        t = np.abs(sig)
        if next_obs is not None:
            qn = NN.forward(flat, next_obs, F, O)[rows, next_act]
            t = t + np.abs(gamma_mask * qn)
        dy[rows, act] = 2.0 * (t + np.abs(y[rows, act])) / B
    else:
        q = out / out.sum(-1, keepdims=True)
        eps = NN.EPS_CLAMP
        inside = (q >= eps) & (q <= 1 - eps)
        ga = beta * (np.abs(np.log(np.clip(q, eps, 1 - eps))) + inside)
        ga[rows, act] += np.abs(sig) * inside[rows, act] / q[rows, act]
        dy = q * (ga + (q * ga).sum(-1, keepdims=True)) / B
    absflat = np.abs(flat)
    ab = NN.backward(absflat, (np.abs(xx), z1, h1, z2, h2, y), dy, F, O)
    if next_obs is not None:
        _, cn = NN.forward(flat, next_obs, F, O, keep=True)
        dn = np.zeros_like(cn[5])
        dn[rows, next_act] = 2.0 * np.abs(gamma_mask) * (t + np.abs(y[rows, act])) / B
        ab = ab + NN.backward(absflat, (np.abs(cn[0]),) + tuple(cn[1:]), dn, F, O)
    return ab


def conditioning(scale, ab, what):
    """Count of ill-conditioned entries: Adam's step scale (|g| at the first step, sqrt(v / (1 - b2^t)) after it, the RMS of
    the gradients so far) within COND x the rounding bound 2^-24 * sum|terms| of this step's gradient.  Entries with no
    terms are exact zeros in fp32 and fp64."""
    live = ab > 0
    ratio = scale[live] / (U32 * ab[live])
    n_ill = int((ratio <= COND).sum())
    print(f"{what}: {n_ill} ill-conditioned of {int(live.sum())} entries, min scale/bound = {ratio.min() if ratio.size else np.inf:.3g}")
    return n_ill


def relu_margins(flat, x, F, O, what):
    """Count of pre-activations z1, z2 within COND * 2^-24 * sum|terms| of zero, where fp32 could take the other side of
    the ReLU than fp64.  Printed, not asserted: at 10^5 - 10^6 continuous pre-activations a few land there by density, and
    a flip moves a gradient by one row's term, which the 1e-5 rules then report."""
    W1, b1, W2, b2, _, _ = NN.unpack(np.asarray(flat, np.float64), F, O)
    x = np.asarray(x, np.float64)
    ax = x if x.min() >= 0 else np.abs(x)
    z1, a1 = x @ W1.T + b1, ax @ np.abs(W1).T + np.abs(b1)
    h1 = np.maximum(z1, 0)
    z2, a2 = h1 @ W2.T + b2, h1 @ np.abs(W2).T + np.abs(b2)
    n = int((np.abs(z1) <= COND * U32 * a1).sum() + (np.abs(z2) <= COND * U32 * a2).sum())
    if n:
        print(f"{what}: {n} pre-activations within the ReLU margin")
    return n


def update_case(kind, F, O, rows, style, seed, clear=True):
    """Parameters, rows, actions, signal, learning rate and the actor's running gradient of one ia2c_net_update case.  With
    `clear`, redrawn (next seed) until no pre-activation lies inside the ReLU margin: with ~131 rows per W1 column, one
    flipped ReLU moves the gradient by ~5e-5 of its largest entry (seen at 65536 rows, |z1| = 6e-9)."""
    for s in range(seed, seed + 20):
        rng = np.random.RandomState(s)
        flat = linear_init(F, O, s)
        x = make_rows(rng, rows, F, style)
        if not clear or relu_margins(flat, x, F, O, f"draw {s}") == 0:
            break
    else:
        raise AssertionError(f"no draw clears the ReLU margin from seed {seed}")
    act = rng.randint(0, O, rows)
    sig = signals(rng, kind, rows)
    lr = LR_C if kind == 0 else LR_A
    grad0 = running_grad(rng, flat.size) if kind == 1 else None
    return flat, x, act, sig, lr, grad0


def mlp_case(rows, F, O, seed):
    rng = np.random.RandomState(seed)
    flat = (rng.randn(NN.n_params(F, O)) * 0.4).astype(np.float32)
    if F == 8192:
        x = (rng.randn(rows, F) * 0.05).astype(np.float32)
    elif F < 500:
        x = rng.randn(rows, F).astype(np.float32)
    else:
        x = make_rows(rng, rows, F, "sparse")
    return flat, x, rng.randn(rows, O).astype(np.float32)


def class_case(F, O, rows, seed):
    """Observations (class indices for F = 500, dense rows otherwise), actions, targets, advantages, and the initial
    critic and actor parameters of a CriticNetwork / ActorNetwork pair."""
    rng = np.random.RandomState(seed)
    idx = rng.randint(0, F, rows)
    x = one_hot(idx, F) if F == 500 else make_rows(rng, rows, F, "dense")
    act = rng.randint(0, O, rows)
    return idx, x, act, signals(rng, 0, rows), signals(rng, 1, rows), (linear_init(F, O, seed), linear_init(F, O, seed + 1))


def alternating_case(T, E, F, O, n, seed):
    rng = np.random.RandomState(seed)
    out = []
    for _ in range(n):
        out.append(dict(x=make_rows(rng, T * E, F, "sparse"), xn=make_rows(rng, T * E, F, "sparse"), act=rng.randint(0, O, T * E),
                        cnext=rng.randint(0, O, T * E), rew=signals(rng, 0, T * E), mask=(rng.rand(T * E) < 0.9).astype(np.float32)))
    return linear_init(F, O, seed), out


class Oracle:
    """fp64 trajectory of one net under ia2c_net_update / batch_update: loss, the gradient Adam sees (the critic's own,
    the actor's running sum), parameters and moments after every update; asserts every such gradient well conditioned."""

    def __init__(self, kind, flat, F, O, lr, beta=0.0, grad0=None, m0=None, v0=None, step0=0):
        self.kind, self.F, self.O, self.lr, self.beta = kind, F, O, lr, beta
        self.p = flat.astype(np.float64)
        P = flat.size
        self.accum = np.zeros(P) if grad0 is None else grad0.astype(np.float64)
        self.acc_abs = np.abs(self.accum)
        self.m = np.zeros(P) if m0 is None else m0.astype(np.float64)
        self.v = np.zeros(P) if v0 is None else v0.astype(np.float64)
        self.t = step0
        self.n_ill = 0

    def update(self, x, act, sig, what="", **q8):
        x = np.asarray(x, dtype=np.float64)
        act = np.asarray(act).reshape(-1).astype(np.int64)
        sig = np.asarray(sig, dtype=np.float64).reshape(-1)
        if self.kind == 0:
            loss, g, _ = NN.critic_loss_grad(self.p, x, act, sig, self.F, self.O, **q8)
            ab = abs_terms(0, self.p, x, act, sig, 0.0, self.F, self.O, **q8)
        else:
            loss, g1, _ = NN.actor_loss_grad(self.p, x, act, sig, self.beta, self.F, self.O)
            self.accum = self.accum + g1
            self.acc_abs = self.acc_abs + abs_terms(1, self.p, x, act, sig, self.beta, self.F, self.O)
            g, ab = self.accum, self.acc_abs
        self.t += 1
        self.p, self.m, self.v = adam64(self.p, self.m, self.v, g, self.t, self.lr)
        self.n_ill += conditioning(np.sqrt(self.v / (1 - 0.999 ** self.t)), ab, f"{what} update {self.t}")
        relu_margins(self.p, x, self.F, self.O, what)
        assert self.n_ill == 0, what
        return dict(loss=float(loss), g=g, p=self.p.copy(), m=self.m.copy(), v=self.v.copy(), step=self.t, sig=sig)


def check_state(kind, pre, d, r, lr, what):
    """Device state d after one update (pre: before it) against the oracle's r: end to end within 1e-5, and the Adam step
    on the kernel's own gradient within 1e-6."""
    assert d["step"] == r["step"] and d["status"] == 0, (what, d["step"], r["step"], d["status"])
    if kind == 0:
        assert rel_err(d["loss"], r["loss"]) < RTOL, what
    else:
        assert abs(d["loss"] - r["loss"]) <= RTOL * max(abs(r["loss"]), float(np.abs(r["sig"]).mean())), what
    for k in ("g", "p", "m", "v"):
        assert rel_err(d[k], r[k]) < RTOL, (what, k, rel_err(d[k], r[k]))
    p, m, v = adam64(pre["p"], pre["m"], pre["v"], d["g"], r["step"], lr)
    close(d["p"], p), close(d["m"], m), close(d["v"], v)


# ---------------------------------------------------------------- device runs


def net_update_run(kind, flat, act, sig, n, F, O, lr, beta=0.0, x=None, grad0=None, m0=None, v0=None, step0=0, offset=0):
    """n calls of ia2c_net_update on one net; x is copied `offset` floats into a larger allocation.  -> n + 1 host snapshots."""
    import torch
    from ia2c_b200 import _lib
    lib = _lib.load()
    rows, P = len(act), flat.size
    z = np.zeros(P, np.float32)
    p, g = dev(flat), dev(z if grad0 is None else grad0)
    m, v = dev(z if m0 is None else m0), dev(z if v0 is None else v0)
    step = torch.full((1,), step0, dtype=torch.int32, device="cuda")
    loss, status = torch.zeros(1, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
    ws = torch.empty(int(lib.ia2c_net_update_workspace(rows, F, O)), dtype=torch.float32, device="cuda")
    ad, sd = dev(act.astype(np.int32)), dev(sig.astype(np.float32))
    buf = torch.empty(rows * F + offset, dtype=torch.float32, device="cuda")
    buf[offset:] = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32).reshape(-1)).cuda()

    def snap():
        torch.cuda.synchronize()
        return dict(p=host(p).copy(), g=host(g).copy(), m=host(m).copy(), v=host(v).copy(), step=int(step.item()),
                    loss=float(loss.item()), status=int(status.item()))
    out = [snap()]
    for _ in range(n):
        _lib.check(lib.ia2c_net_update(kind, p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), step.data_ptr(),
                                       buf.data_ptr() + 4 * offset, None,
                                       ad.data_ptr(), sd.data_ptr(), beta, lr, loss.data_ptr(), status.data_ptr(), ws.data_ptr(),
                                       rows, F, O, None))
        out.append(snap())
    return out


def class_snap(net):
    import torch
    torch.cuda.synchronize()
    st = net.optimizer.state[net.net.flat]
    return dict(p=host(net.net.flat).copy(), g=host(net.net.flat.grad).copy(), m=host(st["exp_avg"]).copy(),
                v=host(st["exp_avg_sq"]).copy(), step=int(st["step"].item()), loss=float(net.losses[-1]), status=0)


def class_init_snap(net, grad0=None):
    P = net.net.flat.numel()
    z = np.zeros(P)
    return dict(p=host(net.net.flat).copy(), g=z if grad0 is None else grad0, m=z, v=z, step=0)


def check_run(kind, states, oracle, x, act, sig, lr, what, **q8):
    for it in range(1, len(states)):
        r = oracle.update(x, act, sig, what=what, **q8)
        check_state(kind, states[it - 1], states[it], r, lr, f"{what} update {it}")


# ---------------------------------------------------------------- 1. single-pass update, steady state


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("rows", [14208, 14209, 28417, 65536, 65536 + 17])
def test_single_pass_steady_state(monkeypatch, kind, rows):
    """ia2c_net_update on 500 one-hot / sparse-dense features, 6 outputs, 3 updates: no refill (14208), the first refill and
    parity-1 wait (14209), parity back to 0 (28417), cfg3 (65536) and 13-14 uses per block with a partial last tile
    (65553).  At the cfg3-sized shapes also against the kernel sequence behind IA2C_NO_SINGLE_PASS."""
    F, O = 500, 6
    monkeypatch.delenv("IA2C_NO_SINGLE_PASS", raising=False)
    tiles = -(-rows // 32)
    assert -(-tiles // min(148, tiles)) == {14208: 3, 14209: 4, 28417: 7, 65536: 14, 65553: 14}[rows]   # most uses of a block
    flat, x, act, sig, lr, grad0 = update_case(kind, F, O, rows, "sparse", rows + kind)
    states = net_update_run(kind, flat, act, sig, 3, F, O, lr, BETA, x=x, grad0=grad0)
    check_run(kind, states, Oracle(kind, flat, F, O, lr, BETA, grad0), x, act, sig, lr, f"single pass kind {kind} rows {rows}")
    if rows >= 65536:
        monkeypatch.setenv("IA2C_NO_SINGLE_PASS", "1")
        seq = net_update_run(kind, flat, act, sig, 3, F, O, lr, BETA, x=x, grad0=grad0)
        for a, b in zip(states[1:], seq[1:]):
            assert a["step"] == b["step"] and rel_err(a["loss"], b["loss"]) < RTOL
            for k in ("g", "p", "m", "v"):
                assert rel_err(a[k], b[k]) < RTOL, k


# ---------------------------------------------------------------- 2. single-pass boundary shapes and fallbacks


@pytest.mark.parametrize("rows", [1024, 1024 + 31])
@pytest.mark.parametrize("O", [1, 2, 8])
@pytest.mark.parametrize("F", [64, 68, 480, 508, 512])
def test_single_pass_boundary_shapes(monkeypatch, F, O, rows):
    """Every lane-step count (F = 64 .. 512, tails 68 / 508 / 480), O = 1 / 2 / 8 and the smallest row counts, for both
    kinds and one-hot, sparse-dense and fully dense rows, 3 updates each, against the oracle."""
    monkeypatch.delenv("IA2C_NO_SINGLE_PASS", raising=False)
    for kind in (0, 1):
        for style in ("onehot", "sparse", "dense"):
            seed = F * 1000 + O * 100 + rows + 7 * kind + ("onehot", "sparse", "dense").index(style)
            flat, x, act, sig, lr, grad0 = update_case(kind, F, O, rows, style, seed)
            what = f"single pass {rows}x{F}x{O} {style} kind {kind}"
            states = net_update_run(kind, flat, act, sig, 3, F, O, lr, BETA, x=x, grad0=grad0)
            check_run(kind, states, Oracle(kind, flat, F, O, lr, BETA, grad0), x, act, sig, lr, what)


@pytest.mark.parametrize("rows,F,O,offset", [(1023, 500, 6, 0), (2048, 60, 6, 0), (2048, 502, 6, 0), (2048, 516, 6, 0),
                                             (2048, 500, 9, 0), (2048, 500, 6, 1)])
def test_single_pass_fallback_shapes(monkeypatch, rows, F, O, offset):
    """Shapes just outside the single pass (1023 rows, F = 60 / 502 / 516, O = 9, x 4 bytes off a 16-byte boundary) take the
    kernel sequence: the result is byte-identical with and without IA2C_NO_SINGLE_PASS, and matches the oracle."""
    for kind in (0, 1):
        flat, x, act, sig, lr, grad0 = update_case(kind, F, O, rows, "sparse", rows + F + O + offset + kind)
        runs = []
        for no_single in (False, True):
            if no_single:
                monkeypatch.setenv("IA2C_NO_SINGLE_PASS", "1")
            else:
                monkeypatch.delenv("IA2C_NO_SINGLE_PASS", raising=False)
            runs.append(net_update_run(kind, flat, act, sig, 3, F, O, lr, BETA, x=x, grad0=grad0, offset=offset))
        for a, b in zip(*runs):
            for k in a:
                assert np.array_equal(a[k], b[k]), (kind, k)
        what = f"fallback {rows}x{F}x{O} offset {offset} kind {kind}"
        check_run(kind, runs[0], Oracle(kind, flat, F, O, lr, BETA, grad0), x, act, sig, lr, what)


# ---------------------------------------------------------------- 3. MLP kernels at their OMAX buckets


def mlp_forward(lib, _lib, flat, x, rows, F, O, softmax, h1=None):
    import torch
    y = torch.empty(rows, O, device="cuda")
    xd, pd = dev(x), dev(flat)
    _lib.check(lib.ia2c_mlp_forward(pd.data_ptr(), xd.data_ptr(), y.data_ptr(), _lib.ptr(h1), rows, F, O, 1, softmax, None))
    return y


def check_mlp(rows, F, O, seed):
    """ia2c_mlp_forward / ia2c_mlp_backward with softmax off and on: outputs, gradient and dx against the oracle, and the
    backward again from the forward's saved layer-1 activations in accumulate mode."""
    import torch
    from ia2c_b200 import _lib
    lib = _lib.load()
    flat, x, dy = mlp_case(rows, F, O, seed)
    f64 = flat.astype(np.float64)
    relu_margins(f64, x, F, O, f"mlp {rows}x{F}x{O}")
    for softmax in (0, 1):
        y = mlp_forward(lib, _lib, flat, x, rows, F, O, softmax)
        ref, cache = NN.forward(f64, x, F, O, softmax=bool(softmax), keep=True)
        assert rel_err(host(y), ref) < RTOL, ("y", softmax)
        dyp = dy.astype(np.float64)
        if softmax:
            dyp = ref * (dyp - (ref * dyp).sum(-1, keepdims=True))
        gref = NN.backward(f64, cache, dyp, F, O)
        W1, _, W2, _, W3, _ = NN.unpack(f64, F, O)
        dxref = (((dyp @ W3) * (cache[4] > 0)) @ W2 * (cache[2] > 0)) @ W1
        grad = torch.full((flat.size,), 7.0, device="cuda")
        dx = torch.empty(rows, F, device="cuda")
        ws = torch.empty(lib.ia2c_mlp_backward_workspace(rows, F, O), device="cuda")
        xd, pd, dyd = dev(x), dev(flat), dev(dy)
        _lib.check(lib.ia2c_mlp_backward(pd.data_ptr(), xd.data_ptr(), dyd.data_ptr(), None, grad.data_ptr(), dx.data_ptr(),
                                         ws.data_ptr(), rows, F, O, softmax, 0, None))
        torch.cuda.synchronize()
        assert rel_err(host(grad), gref) < RTOL, ("grad", softmax)
        assert rel_err(host(dx), dxref) < RTOL, ("dx", softmax)
        h1 = torch.empty(rows, H, device="cuda")
        y2 = mlp_forward(lib, _lib, flat, x, rows, F, O, softmax, h1)
        assert np.array_equal(host(y2), host(y))
        assert rel_err(host(h1), cache[2]) < RTOL
        dx2 = torch.empty(rows, F, device="cuda")
        _lib.check(lib.ia2c_mlp_backward(pd.data_ptr(), xd.data_ptr(), dyd.data_ptr(), h1.data_ptr(), grad.data_ptr(),
                                         dx2.data_ptr(), ws.data_ptr(), rows, F, O, softmax, 1, None))
        torch.cuda.synchronize()
        assert rel_err(host(grad), 2 * gref) < RTOL, ("grad accumulate", softmax)
        assert rel_err(host(dx2), dxref) < RTOL, ("dx from h1", softmax)


def check_index_equals_dense(rows, F, O, seed):
    """ia2c_mlp_forward_index / ia2c_mlp_backward_index / ia2c_actor_sample_index on class indices against the dense kernels
    on the materialised one-hot rows, byte for byte."""
    import torch
    from ia2c_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(seed)
    flat = dev((rng.randn(NN.n_params(F, O)) * 0.4).astype(np.float32))
    idx = rng.randint(0, F, rows)
    idx[:2] = 0, F - 1
    x = dev(one_hot(idx, F))
    idd = dev(idx.astype(np.int64))
    dy = dev(rng.randn(rows, O).astype(np.float32))
    u = dev(rng.rand(rows).astype(np.float32))
    for softmax in (0, 1):
        res = {}
        for mode in ("dense", "index"):
            y, h1 = torch.empty(rows, O, device="cuda"), torch.empty(rows, H, device="cuda")
            grad = torch.empty(flat.numel(), device="cuda")
            ws = torch.empty(lib.ia2c_mlp_backward_workspace(rows, F, O), device="cuda")
            act, probs = torch.empty(rows, dtype=torch.int64, device="cuda"), torch.empty(rows, O, device="cuda")
            P_ = lambda t: t.data_ptr()
            if mode == "dense":
                _lib.check(lib.ia2c_mlp_forward(P_(flat), P_(x), P_(y), P_(h1), rows, F, O, 1, softmax, None))
                _lib.check(lib.ia2c_mlp_backward(P_(flat), P_(x), P_(dy), P_(h1), P_(grad), None, P_(ws), rows, F, O, softmax, 0, None))
                _lib.check(lib.ia2c_actor_sample(P_(flat), P_(x), P_(u), P_(act), P_(probs), rows, F, O, 0, 0, None))
            else:
                _lib.check(lib.ia2c_mlp_forward_index(P_(flat), P_(idd), P_(y), P_(h1), rows, F, O, softmax, None))
                _lib.check(lib.ia2c_mlp_backward_index(P_(flat), P_(idd), P_(dy), P_(h1), P_(grad), P_(ws), rows, F, O, softmax, 0, None))
                _lib.check(lib.ia2c_actor_sample_index(P_(flat), P_(idd), P_(u), P_(act), P_(probs), rows, F, O, 0, 0, None))
            torch.cuda.synchronize()
            res[mode] = dict(y=host(y), h1=host(h1), grad=host(grad), act=host(act), probs=host(probs))
        for k in res["dense"]:
            assert np.array_equal(res["dense"][k], res["index"][k]), (k, softmax)


@pytest.mark.parametrize("F", [6, 63, 64, 500])
@pytest.mark.parametrize("O", BUCKETS)
def test_mlp_kernels_at_every_bucket(O, F):
    """Forward, backward (dx, with and without h1_saved, accumulate) at O = 1 / 4 / 5 / 9 / 10 / 31 / 32 on both row
    mappings (F = 6, 63 thread per row; 64, 500 warp per row), and the index kernels byte for byte against them."""
    rows = 2053
    check_mlp(rows, F, O, 100 * O + F)
    check_index_equals_dense(rows, F, O, 100 * O + F + 1)


@pytest.mark.parametrize("O", [6, 32])
def test_mlp_kernels_at_the_widest_input(O):
    """F = 8192, the API limit: the wide kernels stage 197 KB of weights in opt-in shared memory."""
    check_mlp(3000, 8192, O, O)


# ---------------------------------------------------------------- 4. grid-stride loops and dW1 chunking


def class_pair_run(F, O, obs, act, target, adv, n, flats):
    """n CriticNetwork / ActorNetwork.batch_update pairs (no graph: ia2c_net_update) -> per-net snapshots."""
    from ia2c_b200.nets import ActorNetwork, CriticNetwork
    critic, actor = CriticNetwork("c", F, O, LR_C), ActorNetwork("a", F, O, LR_A, BETA)
    critic.net.load_flat(flats[0]), actor.net.load_flat(flats[1])
    snaps = [[class_init_snap(critic)], [class_init_snap(actor)]]
    for _ in range(n):
        critic.batch_update(obs, act, target)
        snaps[0].append(class_snap(critic))
        actor.batch_update(obs, act, adv)
        snaps[1].append(class_snap(actor))
    return snaps


def check_class_pair(F, O, x, act, target, adv, flats, snaps, what):
    check_run(0, snaps[0], Oracle(0, flats[0], F, O, LR_C), x, act, target, LR_C, f"{what} critic")
    check_run(1, snaps[1], Oracle(1, flats[1], F, O, LR_A, BETA), x, act, adv, LR_A, f"{what} actor")


@pytest.mark.parametrize("rows,F", [(300001, 6), (65537, 500), (16385, 500)])
def test_grid_stride_and_chunking(monkeypatch, rows, F):
    """300001 x 6: the narrow kernels and both losses stride past 151552 rows and the loss adds 592 block partials.
    65537 x 500: the wide kernels stride past 4736 rows, dW1 in 1024 chunks of 65 rows.  16385 x 500: 257 chunks, a second
    round of B3 slices.  Through the C ABI (mlp kernels; ia2c_net_update's kernel sequence, 3 updates of each kind) and
    through CriticNetwork / ActorNetwork.batch_update (index input for F = 500)."""
    import torch
    from ia2c_b200 import _lib
    O = 6
    chunks = min(1024, -(-rows // 64))
    assert (chunks, -(-rows // chunks)) == {300001: (1024, 293), 65537: (1024, 65), 16385: (257, 64)}[rows]
    check_mlp(rows, F, O, rows)
    monkeypatch.setenv("IA2C_NO_SINGLE_PASS", "1")
    for kind in (0, 1):
        flat, x, act, sig, lr, grad0 = update_case(kind, F, O, rows, "dense" if F < 64 else "sparse", rows + kind,
                                                     clear=rows < 300001)
        states = net_update_run(kind, flat, act, sig, 3, F, O, lr, BETA, x=x, grad0=grad0)
        check_run(kind, states, Oracle(kind, flat, F, O, lr, BETA, grad0), x, act, sig, lr, f"sequence {rows}x{F} kind {kind}")
    monkeypatch.delenv("IA2C_NO_SINGLE_PASS")
    idx, x, act, target, adv, flats = class_case(F, O, rows, rows + 7)
    obs = torch.from_numpy(idx if F == 500 else x).cuda()
    a_t = torch.from_numpy(act[:, None].astype(np.float32)).cuda()
    t_t, adv_t = torch.from_numpy(target[:, None]).cuda(), torch.from_numpy(adv[:, None]).cuda()
    snaps = class_pair_run(F, O, obs, a_t, t_t, adv_t, 3, flats)
    check_class_pair(F, O, x, act, target, adv, flats, snaps, f"class API {rows}x{F}")


# ---------------------------------------------------------------- 5. loss kernels


@pytest.mark.parametrize("O", [1, 32])
def test_loss_kernels_past_the_grid_stride(O):
    """ia2c_critic_loss / ia2c_actor_loss at 200003 rows (592 blocks striding, 592 partials): loss, dQ, dtarget, dprobs and
    dadv against the closed forms on the kernels' fp32 inputs."""
    import torch
    from ia2c_b200 import _lib
    lib = _lib.load()
    B = 200003
    rng = np.random.RandomState(O)
    act = rng.randint(0, O, B)
    ad = dev(act.astype(np.int32))
    ws = torch.empty(lib.ia2c_loss_workspace(B), device="cuda")
    loss = torch.zeros((), device="cuda")
    # critic: mean((target - Q[a])^2), dQ[a] = -2 delta / B, dtarget = 2 delta / B
    Q = rng.randn(B, O).astype(np.float32)
    tg = rng.randn(B).astype(np.float32)
    dQ, dT = torch.empty(B, O, device="cuda"), torch.empty(B, device="cuda")
    Qd, td = dev(Q), dev(tg)
    _lib.check(lib.ia2c_critic_loss(Qd.data_ptr(), ad.data_ptr(), td.data_ptr(), loss.data_ptr(), dQ.data_ptr(), dT.data_ptr(),
                                    ws.data_ptr(), B, O, None))
    torch.cuda.synchronize()
    delta = tg.astype(np.float64) - Q[np.arange(B), act]
    dQr = np.zeros((B, O))
    dQr[np.arange(B), act] = -2 * delta / B
    assert rel_err(float(loss.item()), np.mean(delta * delta)) < RTOL
    assert rel_err(host(dQ), dQr) < RTOL and rel_err(host(dT), 2 * delta / B) < RTOL
    # actor: Categorical(probs=p), beta = 0.01, advantages of mean 1
    y = rng.randn(B, O) * 2
    p = np.exp(y - y.max(-1, keepdims=True))
    p = (p / p.sum(-1, keepdims=True)).astype(np.float32)
    adv = signals(rng, 1, B)
    dP, dA = torch.empty(B, O, device="cuda"), torch.empty(B, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    pd, advd = dev(p), dev(adv)
    _lib.check(lib.ia2c_actor_loss(pd.data_ptr(), ad.data_ptr(), advd.data_ptr(), BETA, loss.data_ptr(), dP.data_ptr(), dA.data_ptr(),
                                   status.data_ptr(), ws.data_ptr(), B, O, None))
    torch.cuda.synchronize()
    p64, a64 = p.astype(np.float64), adv.astype(np.float64)
    s = p64.sum(-1, keepdims=True)
    q = p64 / s
    eps = NN.EPS_CLAMP
    inside = (q >= eps) & (q <= 1 - eps)
    logit = np.log(np.clip(q, eps, 1 - eps))
    rows = np.arange(B)
    neglogp = -logit[rows, act]
    lref = np.mean(a64 * neglogp + BETA * (logit * q).sum(-1))
    g = BETA * (logit + inside)
    g[rows, act] -= a64 * inside[rows, act] / q[rows, act]
    dPr = (g - (q * g).sum(-1, keepdims=True)) / s / B
    assert int(status.item()) == 0
    assert rel_err(float(loss.item()), lref) < RTOL
    assert rel_err(host(dP), dPr) < RTOL and rel_err(host(dA), neglogp / B) < RTOL


# ---------------------------------------------------------------- 6. samplers


def check_sampler(entry, flat, xin, x, rows, F, O, what):
    """Injected uniforms and Philox: probabilities within 1e-5 of the oracle, actions equal to the inverse CDF of the kernel's
    own probabilities at the oracle's uniforms."""
    import torch
    from ia2c_b200 import _lib
    rng = np.random.RandomState(rows + F + O)
    ref = NN.forward(flat.astype(np.float64), x, F, O, softmax=True)
    act, probs = torch.empty(rows, dtype=torch.int64, device="cuda"), torch.empty(rows, O, device="cuda")
    u = rng.rand(rows).astype(np.float32)
    seed, counter = 0x5EED0000 + O, (5 << 16) | 9
    fd = dev(flat)
    for uu in (u, None):
        ud = dev(uu) if uu is not None else None
        _lib.check(entry(fd.data_ptr(), xin.data_ptr(), None if ud is None else ud.data_ptr(), act.data_ptr(),
                         probs.data_ptr(), rows, F, O, seed, counter, None))
        torch.cuda.synchronize()
        if uu is None:
            uu = PH.uniform_f32(seed, PH.STREAM_ACTION, 5, 9, np.arange(rows))
        assert rel_err(host(probs), ref) < RTOL, what
        assert np.array_equal(host(act), NN.sample_inverse_cdf(host(probs), uu)), what
    if O > 1:
        assert len(np.unique(host(act))) > 1, what


@pytest.mark.parametrize("O", [1, 5, 32])
@pytest.mark.parametrize("F", [64, 500])
def test_wide_sampler_vs_oracle(F, O):
    """ia2c_actor_sample on the warp-per-row path (actor_sample_kernel<*, true>) against the oracle."""
    from ia2c_b200 import _lib
    rows = 20011
    rng = np.random.RandomState(F + O)
    flat = linear_init(F, O, F + O)
    flat[-O:] += rng.randn(O).astype(np.float32)
    x = make_rows(rng, rows, F, "dense" if F == 64 else "sparse")
    check_sampler(_lib.load().ia2c_actor_sample, flat, dev(x), x, rows, F, O, f"wide sampler {F}x{O}")


@pytest.mark.parametrize("O", BUCKETS)
def test_index_sampler_vs_oracle(O):
    from ia2c_b200 import _lib
    rows, F = 20011, 500
    rng = np.random.RandomState(O)
    flat = linear_init(F, O, O)
    flat[-O:] += rng.randn(O).astype(np.float32)
    idx = rng.randint(0, F, rows)
    check_sampler(_lib.load().ia2c_actor_sample_index, flat, dev(idx.astype(np.int64)), one_hot(idx, F), rows, F, O,
                  f"index sampler {O}")


# ---------------------------------------------------------------- 7. class-API Adam at large step counters


@pytest.mark.parametrize("step0", [0, 1, 9, 1000, 123456, 2 ** 30])
def test_class_api_adam_at_large_step_counters(step0):
    """adam_kernel (ia2c_adam_step, with and without grad_accum) and net_update_reduce_adam_kernel (the single pass) against
    a float64 Adam step from device step counters step0: pow(b, t) is taken in the kernels from the counter."""
    import torch
    from ia2c_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(step0 % 1000)
    nets, P = 2, 147
    for accumulate in (False, True):
        p0 = rng.randn(nets, P).astype(np.float32)
        m0 = (rng.randn(nets, P) * 1e-3).astype(np.float32)
        v0 = (rng.rand(nets, P) * 1e-5).astype(np.float32)
        g = (rng.randn(nets, P) * 1e-2).astype(np.float32)
        acc0 = (rng.randn(nets, P) * 1e-2).astype(np.float32)
        p, m, v, gd, acc = dev(p0), dev(m0), dev(v0), dev(g), dev(acc0)
        step = torch.full((nets,), step0, dtype=torch.int32, device="cuda")
        _lib.check(lib.ia2c_adam_step(p.data_ptr(), gd.data_ptr(), acc.data_ptr() if accumulate else None, m.data_ptr(),
                                      v.data_ptr(), step.data_ptr(), 2e-4, 0.9, 0.999, 1e-8, nets, P, None))
        torch.cuda.synchronize()
        assert (host(step) == step0 + 1).all()
        geff = g.astype(np.float64) + (acc0 if accumulate else 0)
        if accumulate:
            close(host(acc), geff)
        rp, rm, rv = adam64(p0, m0, v0, geff, step0 + 1, 2e-4)
        close(host(p), rp), close(host(m), rm), close(host(v), rv)
    rows, F, O = 1024, 64, 3
    for kind in (0, 1):
        flat, x, act, sig, lr, grad0 = update_case(kind, F, O, rows, "dense", kind)
        P = flat.size
        m0, v0 = (rng.randn(P) * 1e-3).astype(np.float32), (rng.rand(P) * 1e-5).astype(np.float32)
        d = net_update_run(kind, flat, act, sig, 1, F, O, lr, BETA, x=x, grad0=grad0, m0=m0, v0=v0, step0=step0)
        r = Oracle(kind, flat, F, O, lr, BETA, grad0, m0, v0, step0).update(x, act, sig, f"adam step0 {step0}")
        check_state(kind, d[0], d[1], r, lr, f"single pass at step0 {step0} kind {kind}")


# ---------------------------------------------------------------- 8. the cfg3 workload as users run it


@pytest.mark.parametrize("inp", ["dense", "index"])
def test_cfg3_pair_as_users_run_it(inp):
    """bench cfg3: CriticNetwork + ActorNetwork.batch_update on [64, 1024, 500] dense one-hot floats (the single pass) or
    int64 class indices (the index kernels), 3 update pairs against the oracle."""
    import torch
    T, E, F, O = 64, 1024, 500, 6
    idx, x, act, target, adv, flats = class_case(F, O, T * E, 33)
    it = torch.from_numpy(idx.reshape(T, E)).cuda()
    obs = torch.nn.functional.one_hot(it, F).float() if inp == "dense" else it
    a_t = torch.from_numpy(act.reshape(T, E, 1).astype(np.float32)).cuda()
    t_t = torch.from_numpy(target.reshape(T, E, 1)).cuda()
    adv_t = torch.from_numpy(adv.reshape(T, E, 1)).cuda()
    snaps = class_pair_run(F, O, obs, a_t, t_t, adv_t, 3, flats)
    check_class_pair(F, O, x, act, target, adv, flats, snaps, f"cfg3 {inp}")


def test_fused_and_autograd_critic_updates_share_the_optimizer():
    """_fused_update and the autograd path (a target with a graph through run_main(grad=True), Q8) alternate on one
    CriticNetwork: the same Adam moments and device step counter carry across."""
    import torch
    from ia2c_b200.nets import CriticNetwork
    T, E, F, O, gamma = 8, 512, 500, 6, 0.95
    flat, data = alternating_case(T, E, F, O, 4, 8)
    critic = CriticNetwork("c", F, O, LR_C)
    critic.net.load_flat(flat)
    oracle = Oracle(0, flat, F, O, LR_C)
    pre = class_init_snap(critic)
    for it, c in enumerate(data):
        x, xn, act, cnext, rew, mask = c["x"], c["xn"], c["act"], c["cnext"], c["rew"], c["mask"]
        obs = torch.from_numpy(x.reshape(T, E, F)).cuda()
        a_t = torch.from_numpy(act.reshape(T, E, 1)).cuda()
        if it % 2 == 0:   # no graph: one ia2c_net_update call
            tgt = (rew + gamma * mask * NN.forward(oracle.p, xn, F, O)[np.arange(T * E), cnext]).astype(np.float32)
            critic.batch_update(obs, a_t, torch.from_numpy(tgt.reshape(T, E, 1)).cuda())
            r = oracle.update(x, act, tgt, what=f"fused update {it}")
        else:             # the target keeps its graph through the second forward pass (ia2c.py:108-113)
            nobs = torch.from_numpy(xn.reshape(T, E, F)).cuda()
            qn = (critic.run_main(nobs, grad=True) * torch.nn.functional.one_hot(torch.from_numpy(cnext.reshape(T, E)).cuda(), O)).sum(-1, keepdims=True)
            target = torch.from_numpy(rew.reshape(T, E, 1)).cuda() + gamma * torch.from_numpy(mask.reshape(T, E, 1)).cuda() * qn
            assert target.requires_grad
            critic.batch_update(obs, a_t, target)
            r = oracle.update(x, act, rew, what=f"autograd update {it}", next_obs=xn, next_act=cnext,
                              gamma_mask=gamma * mask.astype(np.float64))
        d = class_snap(critic)
        check_state(0, pre, d, r, LR_C, f"alternating update {it}")
        pre = d
