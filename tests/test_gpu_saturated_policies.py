"""Every actor-gradient kernel against the fp64 oracle on saturated policies.

The actor loss is Categorical(probs=p): q = p / sum(p), logit = log(clamp(q, eps, 1 - eps)), eps = 2^-23, and its gradient
is zero through the clamp.  Each kernel writes that rule out by hand, and at reference-like weights every q is of order 1/A,
so the clamp is never reached.  Long training ends near-deterministic, and there it is reached all the time.  The actors
here keep a small W3 and set the output bias b3 so that whole agents (or, for A2C, joint actions) sit in chosen regimes,
measured as logit gaps below the top logit:

  R0 interior        reference weights;
  R1 clamped low     one action at a gap of 25 (q ~ 1e-11, a normal fp32 number), the others inside with q <= 0.9;
  R2 subnormal       one action at a gap of 95: its fp32 probability is subnormal (the build keeps subnormals);
  R3 exact zero      one action at a gap of 125: expf underflows to exactly 0 in fp32;
  R4 saturated       both minor actions at gaps of 20 or more: the dominant q lies above 1 - eps in fp32 and fp64.

`classify` is called on the oracle's fp64 q at the observations each test uses.  It asserts margins (no q and no 1 - q
within a factor 4 of eps, so the kernels' fp32 clamp decision is the oracle's) and conditioning (no inside q above 0.99,
where go - qg cancels to adv * (1 - q) and no fp32 implementation meets 1e-5), and it counts rows per regime and taken
clamped / zero-probability actions, so that a test fails rather than goes vacuous when its actors drift.

The GPU cases pin one kernel each: actor_loss_kernel (loss.cu, the kernel sequence of ia2c_net_update), the single-pass
update (net_update.cu), the column actor kernel standalone on every rollout path and in its RUNS instantiation (trainer.cu),
the pipelined actor kernel (actor_pipe.cu), the A2C actor kernel (a2c.cu), the inverse-CDF sampler and the evaluation."""
from collections import Counter

import numpy as np
import pytest

from oracle import a2c_envs as A2
from oracle import evaluate as EV
from oracle import loops as L
from oracle import nets as NN
from oracle import philox as P
from tests.helpers import dev, host, rel_err
from tests.test_gpu_trainer import _compare_with_oracle
from tests.test_gpu_trainer_oracle_scale import RUNS_HYPER, assert_path, buffers, check_episode, oracle_state

RTOL = 1e-5
EPS = NN.EPS_CLAMP
TINY32 = float(np.finfo(np.float32).tiny)
H = NN.HIDDEN
GAP = {"R1": 25.0, "R2": 95.0, "R3": 125.0}
CYCLE = ("R1", "R3", "R2", "R4", "R0")   # agent i of a trainer takes CYCLE[i % 5]: N = 2 gives R1 and R3

# Philox keys whose action stream draws x >> 8 == 0, i.e. u == 0, at (index, t) of episode 0: the inverse-CDF sampler then
# takes action 0 whenever p0 > 0, so a batch whose actors clamp action 0 low takes a clamped action there.  Found offline
# with oracle/philox.py over index < 64 and t < 4; the tests re-check the draw.
ZERO_DRAWS = ((0xC27B, 27, 0), (0x500006F98, 14, 1))


# ---------------------------------------------------------------- constructions


def w3_offset(F):
    return H * F + H + H * H + H


def linear_init(F, A, seed):
    """nn.Linear-style uniform(-1/sqrt(fan_in), 1/sqrt(fan_in)) parameters of an F -> 6 -> 6 -> A net."""
    rng = np.random.RandomState(seed)
    parts = []
    for fi, fo in ((F, H), (H, H), (H, A)):
        k = 1.0 / np.sqrt(fi)
        parts += [rng.uniform(-k, k, (fo, fi)), rng.uniform(-k, k, fo)]
    return NN.pack(parts).astype(np.float32)


def saturate(actor, regimes, F=6, A=3, low=None, seed=0):
    """Copies of actor parameters [n, P] (reference_init, a2c_reference_init) with net n in regimes[n]: W3 of scale 0.05
    and b3 holding the regime's logit gaps.  The clamped-low action of net n is `low` (default n % A); "R123" clamps
    three actions low at once (low, low + 1, low + 2: gaps 25, 95 and 125) and needs A >= 5."""
    a = np.array(actor, dtype=np.float32).reshape(len(regimes), -1).copy()
    rng = np.random.RandomState(seed)
    w3 = w3_offset(F)
    for n, reg in enumerate(regimes):
        if reg == "R0":
            continue
        lo = n % A if low is None else low
        lows = [(lo + k) % A for k in range(3)] if reg == "R123" else [lo]
        others = [o for o in range(A) if o not in lows]
        b = np.zeros(A)
        if reg == "R4":
            b[:] = -20.0 - 4.0 * rng.rand(A)
            b[others[0]] = 0.0
        else:
            for o, g in zip(lows, (GAP["R1"], GAP["R2"], GAP["R3"]) if reg == "R123" else (GAP[reg],)):
                b[o] = -g
            b[others] = -np.linspace(0.0, 0.7, len(others))
        a[n, w3:w3 + H * A] = rng.uniform(-0.05, 0.05, H * A)
        a[n, w3 + H * A:w3 + H * A + A] = b
    return a


def classify(flat, x, act, F=6, A=3, dev_flat=None):
    """Margins, conditioning and regime counts of the rows x [B, F] of one net with taken actions act [B].  q is the oracle's
    fp64 distribution at the parameters `flat`; the fp32 one (R1 / R2 / R3, taken zeros) is at `dev_flat`, the parameters
    the device held (default: flat rounded to fp32)."""
    x = np.asarray(x, dtype=np.float64).reshape(-1, F)
    act = np.asarray(act).reshape(-1).astype(np.int64)
    q = NN.forward(np.asarray(flat, dtype=np.float64), x, F, A, softmax=True)
    q = q / q.sum(-1, keepdims=True)
    p32 = NN.forward(np.asarray(flat if dev_flat is None else dev_flat, dtype=np.float32), x.astype(np.float32), F, A,
                     softmax=True)
    q32 = p32 / p32.sum(-1, keepdims=True)

    def band(v):
        return (v >= EPS / 4) & (v <= 4 * EPS)

    assert not band(q).any(), f"{int(band(q).sum())} probabilities within a factor 4 of eps"
    assert not band(1 - q).any(), f"{int(band(1 - q).sum())} probabilities within 4 eps of 1"
    assert not ((q > 0.99) & (q <= 1 - EPS)).any(), "an inside probability above 0.99 (ill-conditioned row)"
    low, high = q < EPS, q > 1 - EPS
    rows = np.arange(len(act))
    return Counter(R0=int((~low.any(-1) & ~high.any(-1)).sum()), R1=int((low & (q32 >= TINY32)).any(-1).sum()),
                   R2=int((low & (q32 > 0) & (q32 < TINY32)).any(-1).sum()), R3=int((low & (q32 == 0)).any(-1).sum()),
                   R4=int(high.any(-1).sum()), taken_low=int((q[rows, act] < EPS).sum()),
                   taken_zero=int((q32[rows, act] == 0).sum()))


def require(counts, regimes, taken_zero=True, what=""):
    """Every claimed regime and a taken clamped action (and, with taken_zero, a taken fp32 zero) occurred."""
    summary = f"{what}: " + ", ".join(f"{k}={counts[k]}" for k in ("R0", "R1", "R2", "R3", "R4", "taken_low", "taken_zero"))
    print(summary)
    for r in regimes:
        assert counts[r] > 0, f"no {r} row; {summary}"
    assert counts["taken_low"] > 0, f"no taken clamped action; {summary}"
    if taken_zero:
        assert counts["taken_zero"] > 0, f"no taken zero-probability action; {summary}"


def regimes_of(N):
    return [CYCLE[i % len(CYCLE)] for i in range(N)]


def claimed(N):
    return sorted(set(regimes_of(N)))


def ia2c_init(N, M, seed, regimes=None, low=None):
    from ia2c_b200.trainer import reference_init
    actor, critic, fa = reference_init(N, M, seed=seed)
    return saturate(actor, regimes or regimes_of(N), low=low, seed=seed), critic, fa


# ---------------------------------------------------------------- CPU: the constructions and the oracle


@pytest.mark.parametrize("N", [2, 5, 12])
def test_ia2c_constructions_hold_margins_and_regimes(N):
    """Every agent of a constructed trainer init sits in its regime at all 9 observations, with the margins."""
    from ia2c_b200.trainer import reference_init
    actor, _, _ = reference_init(N, 5, seed=N)
    sat = saturate(actor, regimes_of(N), seed=N)
    for i, reg in enumerate(regimes_of(N)):
        act = np.full(9, i % 3)
        c = classify(sat[i], EV.OBS9, act)
        assert c[reg] == 9, (i, reg, c)
        assert reg == "R4" or c["R4"] == 0, (i, c)   # (an R4 row's minor actions are clamped low as well)
        if reg in ("R1", "R2", "R3"):
            assert c["taken_low"] == 9 and c["taken_zero"] == (9 if reg == "R3" else 0), (i, c)
            q = NN.forward(sat[i].astype(np.float64), EV.OBS9, 6, 3, softmax=True)
            assert q.max() <= 0.9


def test_mixed_constructions_hold_margins():
    """The A = 6 and A = 9 (A2C joint) actors clamp three actions low at once, one of each fp32 kind."""
    from ia2c_b200.a2c import a2c_reference_init
    rng = np.random.RandomState(0)
    flat = saturate(linear_init(500, 6, 1)[None], ["R123"], F=500, A=6, low=2)[0]
    x = np.eye(500)[rng.randint(0, 500, 300)]
    c = classify(flat, x, np.arange(300) % 6, F=500, A=6)
    assert c["R1"] == c["R2"] == c["R3"] == 300 and c["taken_low"] == 150 and c["taken_zero"] == 50, c
    actor, _ = a2c_reference_init(0)
    sat = saturate(actor[None], ["R123"], A=9, low=4)[0]
    c = classify(sat, EV.OBS9, np.arange(9), A=9)
    assert c["R1"] == c["R2"] == c["R3"] == 9 and c["taken_low"] == 3 and c["taken_zero"] == 1, c


def test_classifier_refuses_rows_on_the_clamp():
    """A probability at eps, at 1 - eps or inside above 0.99 is refused: there the fp32 and fp64 decisions may differ."""
    flat = np.zeros(NN.n_params(6, 3))
    w3 = w3_offset(6)
    for b3 in ([0.0, -np.log(1 / EPS), 0.0], [0.0, -15.9 + 0.35, -30.0], [0.0, -6.0, -30.0]):
        flat[w3 + 18:] = b3
        with pytest.raises(AssertionError):
            classify(flat, EV.OBS9, np.zeros(9, int))


def test_oracle_gradient_is_torch_categorical_at_saturated_rows():
    """The oracle's closed form against torch autograd through Categorical(probs=softmax(y)) in fp32, the reference's
    precision, on rows with clamped-low, subnormal, zero and saturated actions, taken and not taken."""
    import torch
    from torch.distributions import Categorical
    rng = np.random.RandomState(3)
    beta = 0.05
    for F, A, reg, low in ((6, 3, "R1", 0), (6, 3, "R2", 1), (6, 3, "R3", 2), (6, 3, "R4", 1), (6, 9, "R123", 3)):
        flat = saturate(linear_init(F, A, 7)[None], [reg], F=F, A=A, low=low, seed=5)[0]
        x = rng.rand(64, F).astype(np.float32)
        act = rng.randint(0, A, 64)
        adv = rng.randn(64).astype(np.float32)
        c = classify(flat, x, act, F=F, A=A)
        require(c, [reg] if reg != "R123" else ["R1", "R2", "R3"], taken_zero=reg in ("R3", "R123"), what=f"oracle {reg}")
        loss, grad, _ = NN.actor_loss_grad(flat.astype(np.float64), x, act, adv, beta, F, A)
        w = torch.tensor(flat, requires_grad=True)
        W1, b1, W2, b2, W3, b3 = (w[o:o + int(np.prod(s))].reshape(s) for o, s in
                                  zip(np.cumsum([0, H * F, H, H * H, H, A * H]), ((H, F), (H,), (H, H), (H,), (A, H), (A,))))
        h = torch.relu(torch.relu(torch.from_numpy(x) @ W1.T + b1) @ W2.T + b2)
        d = Categorical(probs=torch.softmax(h @ W3.T + b3, -1))
        tl = (torch.from_numpy(adv) * -d.log_prob(torch.from_numpy(act)) - beta * d.entropy()).mean()
        tl.backward()
        assert abs(tl.item() - float(loss)) <= RTOL * max(abs(float(loss)), float(np.abs(adv).mean())), reg
        assert rel_err(w.grad.numpy(), grad) < RTOL, reg


# ---------------------------------------------------------------- a, b: loss.cu and the single-pass update


@pytest.mark.gpu
@pytest.mark.parametrize("F, A, rows, reg", [(6, 3, 600, "R1"), (6, 3, 600, "R2"), (6, 3, 600, "R3"), (500, 6, 1200, "R123")])
def test_actor_loss_kernel_via_batch_update(monkeypatch, F, A, rows, reg):
    """ActorNetwork.batch_update on the kernel sequence (forward, actor_loss_kernel, backward, Adam) over 3 updates: loss,
    the never-zeroed gradient sum (Q2) and parameters against NN.actor_loss_grad + AdamRef.  The org shape takes dense rows,
    the taxi shape one-hot class indices."""
    import torch
    from ia2c_b200.nets import ActorNetwork
    monkeypatch.setenv("IA2C_NO_SINGLE_PASS", "1")
    lr, beta = 1e-3, 0.02
    rng = np.random.RandomState(rows + F)
    flat = saturate(linear_init(F, A, F)[None], [reg], F=F, A=A, low=rng.randint(A), seed=F)[0]
    net = ActorNetwork("a", F, A, lr, beta)
    net.net.load_flat(flat)
    ref, adam, accum = flat.astype(np.float64), NN.AdamRef(flat.size, lr, np.float64), np.zeros(flat.size)
    counts = Counter()
    for it in range(3):
        if F == 500:
            idx = rng.randint(0, F, rows)
            obs, x = torch.from_numpy(idx), np.eye(F)[idx]
        else:
            x = rng.rand(rows, F).astype(np.float32)
            obs = torch.from_numpy(x)
        act = rng.randint(0, A, rows)
        adv = rng.randn(rows).astype(np.float32)
        counts += classify(ref, x, act, F=F, A=A, dev_flat=host(net.net.flat))
        net.batch_update(obs, torch.from_numpy(act).reshape(rows, 1), torch.from_numpy(adv).reshape(rows, 1))
        loss, grad, _ = NN.actor_loss_grad(ref, x, act, adv.astype(np.float64), beta, F, A)
        accum = accum + grad
        ref = adam.step(ref, accum)
        scale = max(abs(float(loss)), float(np.abs(adv).mean()))
        assert abs(float(net.losses[-1]) - float(loss)) <= RTOL * scale, it
        assert rel_err(host(net.net.flat.grad), accum) < RTOL, it
        assert rel_err(host(net.net.flat), ref) < RTOL, it
    require(counts, ["R1", "R2", "R3"] if reg == "R123" else [reg], taken_zero=reg in ("R3", "R123"), what=f"loss.cu {F}x{A} {reg}")


@pytest.mark.gpu
@pytest.mark.parametrize("rows", [4100, 5000])
def test_single_pass_actor_update_vs_oracle(monkeypatch, rows):
    """ia2c_net_update kind 1 on wide dense rows (the single-pass kernel) against the oracle directly, 2 updates, from a
    non-zero running gradient sum."""
    import torch
    from ia2c_b200 import _lib
    monkeypatch.delenv("IA2C_NO_SINGLE_PASS", raising=False)
    lib = _lib.load()
    F, A, lr, beta = 500, 6, 5e-4, 0.01
    rng = np.random.RandomState(rows)
    flat = saturate(linear_init(F, A, rows)[None], ["R123"], F=F, A=A, low=1, seed=rows)[0]
    x = np.zeros((rows, F), dtype=np.float32)
    x[np.arange(rows), rng.randint(0, F, rows)] = 1.0
    x[: rows // 2] += (rng.rand(rows // 2, F) < 0.05) * rng.rand(rows // 2, F).astype(np.float32)
    act = rng.randint(0, A, rows).astype(np.int32)
    sig = rng.randn(rows).astype(np.float32)
    grad0 = (rng.randn(flat.size) * 0.01).astype(np.float32)
    p, g = dev(flat.copy()), dev(grad0.copy())
    m, v = dev(np.zeros(flat.size, np.float32)), dev(np.zeros(flat.size, np.float32))
    step = torch.zeros(1, dtype=torch.int32, device="cuda")
    loss, status = torch.zeros(1, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
    ws = torch.empty(int(lib.ia2c_net_update_workspace(rows, F, A)), dtype=torch.float32, device="cuda")
    xd, ad, sd = dev(x), dev(act), dev(sig)
    ref, adam, accum = flat.astype(np.float64), NN.AdamRef(flat.size, lr, np.float64), grad0.astype(np.float64)
    counts = Counter()
    for it in range(2):
        counts += classify(ref, x, act, F=F, A=A, dev_flat=host(p))
        _lib.check(lib.ia2c_net_update(1, p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), step.data_ptr(), xd.data_ptr(),
                                       None, ad.data_ptr(), sd.data_ptr(), beta, lr, loss.data_ptr(), status.data_ptr(),
                                       ws.data_ptr(), rows, F, A, None))
        torch.cuda.synchronize()
        lr_, grad, _ = NN.actor_loss_grad(ref, x, act, sig.astype(np.float64), beta, F, A)
        accum = accum + grad
        ref = adam.step(ref, accum)
        assert int(status.item()) == 0
        assert abs(float(loss.item()) - float(lr_)) <= RTOL * max(abs(float(lr_)), float(np.abs(sig).mean())), it
        assert rel_err(host(g), accum) < RTOL and rel_err(host(p), ref) < RTOL, it
    require(counts, ["R1", "R2", "R3"], what=f"net_update single pass {rows}x{F}")


# ---------------------------------------------------------------- c, d: column and pipelined actor kernels, injected actions


def injected_episodes(tr, st, E, N, T, episodes, seed):
    """`episodes` injected episodes of tr against the oracle state st (_compare_with_oracle), with uniformly drawn actions,
    so a third of an agent's rows take its clamped action.  Returns the regime counts of the rows the losses covered."""
    rng = np.random.RandomState(seed)
    counts = Counter()
    for _ in range(episodes):
        actions = rng.randint(0, 3, size=(T + 1, E, N))
        u = rng.rand(T + 1, E, N, N - 1)
        before, dev_actor = st.actor.copy(), host(tr.actor_params).copy()
        tr.inject(actions=actions, u_belief=u)
        tr.train_episode(sync_stats=True)
        traj, upd = L.ia2c_episode(st, E, actions=actions, u_belief=u)
        _compare_with_oracle(tr, st, traj, upd, N)
        for i in range(N):
            counts += classify(before[i], traj["obs"][:T], traj["act"][:T, :, i], dev_flat=dev_actor[i])
    return counts


def injected_trainer(E, N, M, T, **kw):
    from ia2c_b200.trainer import IA2CTrainer
    actor, critic, fa = ia2c_init(N, M, seed=N + M)
    st = L.IA2CState(actor=actor.astype(np.float64), critic=critic.astype(np.float64), filter_action=fa, T=T, max_episode_steps=T)
    tr = IA2CTrainer(E, n_agents=N, n_models=M, steps_per_episode=T, max_episode_steps=T, init=(actor, critic, fa), dumps=True,
                     beta=0.01, **kw)
    st.beta = float(np.float32(0.01))
    return tr, st


@pytest.mark.gpu
@pytest.mark.parametrize("path, N, M, E, T, kw", [
    ("fused", 2, 5, 64, 30, {}), ("fused", 5, 5, 33, 12, {}), ("step", 2, 2, 64, 30, {}),
    ("many", 12, 4, 8, 6, {}), ("many", 64, 5, 3, 4, {}), ("table", 36, 2, 4, 4, dict(belief_kernel="step"))])
def test_column_actor_kernel(path, N, M, E, T, kw):
    """trainer.cu's column actor kernel (standalone instantiation) behind every rollout path, two injected episodes."""
    tr, st = injected_trainer(E, N, M, T, actor_kernel="columns", **kw)
    assert_path(tr, N, M, path, "columns")
    counts = injected_episodes(tr, st, E, N, T, 2, seed=N)
    require(counts, claimed(N), what=f"columns {path} N={N}")


@pytest.mark.gpu
@pytest.mark.parametrize("N, M, E, T", [(2, 5, 64, 30), (130, 5, 2, 3)])
def test_pipelined_actor_kernel(N, M, E, T):
    """actor_pipe.cu, two injected episodes; its one division adv / q runs for every row, so a taken q == 0 must leave
    no inf or NaN behind."""
    from ia2c_b200 import _lib
    tr, st = injected_trainer(E, N, M, T, actor_kernel="pipe")
    if N <= 8:
        assert_path(tr, N, M, "fused", "pipe")
    assert not tr.desc.flags & _lib.FLAG_ACTOR_COLUMNS
    counts = injected_episodes(tr, st, E, N, T, 2, seed=N)
    require(counts, claimed(N), what=f"pipe N={N}")
    assert np.isfinite(host(tr.actor_grad)).all() and np.isfinite(host(tr.adv_dump)).all()


# ---------------------------------------------------------------- e: A2C


def a2c_saturated(seed):
    from ia2c_b200.a2c import a2c_reference_init
    actor, critic = a2c_reference_init(seed)
    return saturate(actor[None], ["R123"], A=9, low=seed % 9, seed=seed)[0], critic


@pytest.mark.gpu
@pytest.mark.parametrize("E", [37, 300])
def test_a2c_actor_kernel(E):
    """a2c.cu with injected joint actions against a2c_org_update_envs, 2 updates.  The Q7 term's neglogp is the clamped
    -log eps at every taken clamped action."""
    from ia2c_b200.a2c import A2COrgTrainer
    from tests.test_gpu_a2c import kernel_slots
    T, beta = 20, 0.01
    actor, critic = a2c_saturated(E)
    tr = A2COrgTrainer(E, seeds=1, steps_per_update=T, beta=beta, init=[(actor, critic)])
    st = A2.A2COrgEnvsState(actor=actor.astype(np.float64), critic=critic.astype(np.float64), E=E, T=T,
                            beta=float(np.float32(beta)))
    rng = np.random.RandomState(E)
    counts = Counter()
    for upd in range(2):
        slots = rng.randint(0, 9, size=(T + 1, E))
        before, dev_actor = st.actor.copy(), host(tr.actor_params)[0].copy()
        tr.inject(slots)
        tr.train_update(sync_stats=True)
        got = kernel_slots(tr, upd == 0)
        assert np.array_equal(got[1:], slots[1:]) and (upd > 0 or np.array_equal(got[0], slots[0]))
        out = A2.a2c_org_update_envs(st, actions=got)
        assert np.array_equal(host(tr.obs), out["states"]) and np.array_equal(host(tr.act), out["actions"])
        counts += classify(before, out["states"], out["actions"], A=9, dev_flat=dev_actor)
        assert rel_err(host(tr.critic_params)[0], st.critic) < RTOL
        scale = max(abs(float(out["actor_loss"])), float(np.abs(out["adv"]).mean()))
        assert abs(host(tr.loss_out)[1, 0] - out["actor_loss"]) <= RTOL * scale, upd
        assert rel_err(host(tr.actor_grad)[0, :147], out["actor_grad"]) < RTOL, upd
        assert rel_err(host(tr.actor_grad_accum)[0], out["actor_grad_accum"]) < RTOL, upd
        assert rel_err(host(tr.actor_params)[0], st.actor) < RTOL, upd
    require(counts, ["R1", "R2", "R3"], what=f"a2c E={E}")


@pytest.mark.gpu
def test_a2c_batch_equals_single_runs_when_saturated():
    from ia2c_b200.a2c import A2COrgTrainer
    from tests.test_gpu_a2c import BUFFERS, same_bytes
    E, T, seeds = 37, 20, [5, 9, 11]
    lr_a, lr_c, beta = [1e-4, 3e-4, 1e-3], [5e-5, 1e-4, 5e-4], [0.01, 0.05, 0.002]
    init = [a2c_saturated(s) for s in seeds]
    batch = A2COrgTrainer(E, seeds=seeds, steps_per_update=T, lr_actor=lr_a, lr_critic=lr_c, beta=beta, init=init)
    single = [A2COrgTrainer(E, seeds=s, steps_per_update=T, lr_actor=a, lr_critic=c, beta=b, init=[i])
              for s, a, c, b, i in zip(seeds, lr_a, lr_c, beta, init)]
    for _ in range(3):
        batch.train_update()
        for tr in single:
            tr.train_update()
    for r, tr in enumerate(single):
        view = batch.run_view(r)
        for k in BUFFERS:
            assert same_bytes(view[k], getattr(tr, k)), (r, k)


# ---------------------------------------------------------------- f: batches of runs (the RUNS instantiation)


def adv_rounding_sensitivity(b, st, actor0, accum0, N, T):
    """rel_err by which rounding the advantages to fp32 moves the agents' accumulated oracle gradients (worst agent).  b holds
    the device's episode and st the oracle after it (its updated critic gives the advantages); actor0 and accum0 are the
    actor parameters and the running gradient sum before it."""
    obs, rew = host(b["obs"]).astype(np.float64), host(b["reward"]).astype(np.float64).reshape(-1)
    act, pp = host(b["act"]).astype(np.int64), host(b["partner_pred"]).astype(np.int64)
    worst = 0.0
    for i in range(N):
        nja = L.joint_index(i, N, act[1:T + 1, :, i], pp[1:T + 1, :, i]).reshape(-1)
        ja = L.joint_index(i, N, act[:T, :, i], pp[:T, :, i]).reshape(-1)
        rows = np.arange(ja.size)
        adv = (rew + st.gamma * NN.forward(st.critic[i], obs[1:T + 1], 6, 9)[rows, nja]) - NN.forward(st.critic[i], obs[:T], 6, 9)[rows, ja]
        g64, g32 = (NN.actor_loss_grad(actor0[i], obs[:T], act[:T, :, i], a, st.beta, 6, 3)[1]
                    for a in (adv, adv.astype(np.float32).astype(np.float64)))
        worst = max(worst, rel_err(accum0[i] + g32, accum0[i] + g64))
    return worst


# Sampled actions make the actor gradient a sum of score terms adv * (q - onehot(a)) that cancel in expectation, and in
# Org-N the advantages at these inits are large against what is left.  At few rows per agent the cancellation can be deep
# enough that fp32 rounding of the advantages alone moves the gradient by 1e-6 or more, and then no fp32 kernel meets 1e-5
# on the Adam moments.  The shapes below were chosen well conditioned, and the test asserts that they stay so.
ADV_SENSITIVITY = 1.5e-6


@pytest.mark.gpu
@pytest.mark.parametrize("kind, N, M, E, T, episodes", [("runs", 2, 5, 37, 30, 2), ("runs", 3, 5, 37, 30, 2), ("runs", 8, 5, 37, 30, 2),
                                                         ("many", 12, 4, 24, 10, 2), ("many", 130, 5, 1, 4, 1)])
def test_runs_take_clamped_actions(kind, N, M, E, T, episodes):
    """Batches refuse injected tapes, so the taken clamped action comes from a Philox zero draw on action 0, which every
    agent clamps low (R1).  Each run against the oracle (check_episode) and byte for byte against a standalone trainer
    with its seed, init and hyper-parameters."""
    import torch
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    from ia2c_b200.trainer import IA2CTrainer
    from tests.test_gpu_runs import assert_run_equals
    R = len(ZERO_DRAWS)
    seeds = [s for s, _, _ in ZERO_DRAWS]
    for s, idx, t in ZERO_DRAWS:
        assert idx < E * N and t < T and P.uniform_f32(s, P.STREAM_ACTION, 0, t, np.array([idx]))[0] == 0.0
    assert any(s >> 32 for s in seeds)
    hyper = {k: v[:R] for k, v in RUNS_HYPER.items()}
    init = [ia2c_init(N, M, seed=r, regimes=["R1"] * N, low=0) for r in range(R)]
    cls = IA2CRuns if kind == "runs" else IA2CRunsMany
    batch = cls(E, seeds, n_agents=N, n_models=M, steps_per_episode=T, max_episode_steps=T, init=init, **hyper)
    alone = [IA2CTrainer(E, n_agents=N, n_models=M, steps_per_episode=T, max_episode_steps=T, seed=seeds[r], init=init[r],
                         actor_kernel="columns", **{k: v[r] for k, v in hyper.items()}) for r in range(R)]
    counts = [Counter() for _ in range(R)]
    for ep in range(episodes):
        subjects = [(buffers(batch, r), {k: v[r] for k, v in hyper.items()}) for r in range(R)]
        states = [oracle_state(b, hp, T, T) for b, hp in subjects]
        before = [(st.actor.copy(), host(b["actor_params"]).copy(), st.actor_grad_accum.copy()) for st, (b, _) in zip(states, subjects)]
        batch.train_episode()
        for tr in alone:
            tr.train_episode()
        torch.cuda.synchronize()
        for r, ((b, _), st) in enumerate(zip(subjects, states)):
            check_episode(b, st, seeds[r], ep, E, N, M, T, env_offset=getattr(batch, "env_offset", 0))
            sens = adv_rounding_sensitivity(b, st, before[r][0], before[r][2], N, T)
            assert sens < ADV_SENSITIVITY, f"run {r} episode {ep}: fp32 advantages alone move the gradient by {sens:.2e}"
            obs, act = host(b["obs"])[:T], host(b["act"])[:T]
            for i in range(N):
                counts[r] += classify(before[r][0][i], obs, act[:, :, i], dev_flat=before[r][1][i])
            assert_run_equals(batch, r, alone[r])
    for r in range(R):
        require(counts[r], ["R1"], taken_zero=False, what=f"{kind} N={N} run {r}")


# ---------------------------------------------------------------- g, h: sampler and evaluation


def passthrough_actor(F=6, A=3):
    """Parameters whose logits are x[:3] for x >= 0 (identity layers, zero biases)."""
    flat = np.zeros(NN.n_params(F, A), dtype=np.float32)
    W1, _, W2, _, W3, _ = NN.unpack(flat, F, A)
    W1[:3, :3] = np.eye(3)
    W2[:3, :3] = np.eye(3)
    W3[:, :3] = np.eye(3)
    return flat


@pytest.mark.gpu
def test_sampler_on_zero_probabilities_and_extreme_uniforms():
    """ia2c_actor_sample with injected uniforms 0, 2^-24, 1 - 2^-24 and one fp32 step either side of every CDF boundary,
    on rows with zeros first, in the middle, last, all but one, and a subnormal: the kernel's draw is NN.sample_inverse_cdf
    on its own probabilities, and no zero-probability action is ever returned."""
    import torch
    from ia2c_b200 import _lib
    lib = _lib.load()
    flat = passthrough_actor()
    logits = np.array([[0, 200, 200], [200, 0, 200], [200, 200, 0], [200, 0, 0], [0, 200, 0], [0, 0, 200], [100, 0, 100.5],
                       [0, 0, 0], [0, 125, 0.3]], dtype=np.float32)
    x = np.zeros((len(logits), 6), dtype=np.float32)
    x[:, :3] = logits

    def sample(xr, u):
        act = torch.empty(len(xr), dtype=torch.int64, device="cuda")
        probs = torch.empty(len(xr), 3, device="cuda")
        _lib.check(lib.ia2c_actor_sample(dev(flat).data_ptr(), dev(xr).data_ptr(), dev(u).data_ptr(), act.data_ptr(),
                                         probs.data_ptr(), len(xr), 6, 3, 0, 0, _lib.stream_ptr()), "ia2c_actor_sample")
        torch.cuda.synchronize()
        return host(act), host(probs)

    _, p = sample(x, np.zeros(len(x), np.float32))
    assert (p == 0).sum() >= 9 and ((p > 0) & (p < TINY32)).any()
    us = []
    for row in p:
        s = np.float32(0)
        for v in row:
            s = np.float32(s + v)
        c = np.float32(0)
        cands = [np.float32(0), np.float32(2.0 ** -24), np.float32(1 - 2.0 ** -24)]
        for v in row:
            c = np.float32(c + v)
            b = np.float32(c / s)
            cands += [np.nextafter(b, np.float32(0)), b, np.nextafter(b, np.float32(1))]
        us.append([u for u in cands if 0 <= u < 1])
    rows = np.concatenate([np.full(len(u), i) for i, u in enumerate(us)])
    u = np.concatenate(us).astype(np.float32)
    act, probs = sample(x[rows], u)
    assert np.array_equal(act, NN.sample_inverse_cdf(probs, u))
    assert (probs[np.arange(len(act)), act] > 0).all()


@pytest.mark.gpu
def test_greedy_evaluation_on_saturated_tables_and_ties():
    """Greedy evaluation takes the argmax of each table row, ties to the lowest index (torch.argmax, oracle/evaluate.py)."""
    from ia2c_b200.evaluate import evaluate_actors
    b3s = np.array([[-125, 0, -125], [-30, -30, 0], [0, 0, 0], [-200, 3, 3], [3, -200, 3], [5, 5, -200], [0, -22, -24],
                    [-95, -95, 0]], dtype=np.float32)
    N = len(b3s)
    params = np.zeros((N, 105), dtype=np.float32)
    params[:, 102:] = b3s
    d = dev(params)
    out = evaluate_actors(d, 1, N, 1, 1, 30, 30, True, 0, 0, d.device)
    want = np.argmax(b3s, -1)
    assert np.array_equal(out["greedy_actions"][0], np.repeat(want[:, None], 9, 1))
    assert np.array_equal(out["greedy_actions"], out["policy"].argmax(-1))
    ref = EV.evaluate(np.zeros((N, 105)), 1, 1, 30, 30, greedy=True, table=out["policy"][0])
    assert np.array_equal(out["returns"][0], ref["returns"]) and np.array_equal(out["action_counts"][0], ref["counts"].astype(np.uint64))


@pytest.mark.gpu
def test_philox_evaluation_never_takes_zero_probability_actions():
    """Actors with exact-zero (and subnormal) actions under the stream-4 sampler: the table is ia2c_actor_sample's
    distribution byte for byte, the zero-probability actions never appear, and the counts follow the table."""
    import torch
    from ia2c_b200 import _lib
    from ia2c_b200.evaluate import evaluate_actors
    lib = _lib.load()
    b3s = np.array([[0, -125, 0.5], [-130, 0, 0], [0, 0.3, -140], [-125, -125, 0], [-95, 0, 0.2], [0, -25, -125]], dtype=np.float32)
    N, E, K, T = len(b3s), 64, 2, 30
    params = np.zeros((N, 105), dtype=np.float32)
    params[:, 102:] = b3s
    d = dev(params)
    out = evaluate_actors(d, 1, N, E, K, T, 30, False, 77, 0, d.device)
    x = dev(EV.OBS9.astype(np.float32))
    u = torch.zeros(9, device="cuda")
    act = torch.empty(9, dtype=torch.int64, device="cuda")
    probs = torch.empty(9, 3, device="cuda")
    for i in range(N):
        _lib.check(lib.ia2c_actor_sample(d[i].data_ptr(), x.data_ptr(), u.data_ptr(), act.data_ptr(), probs.data_ptr(),
                                         9, 6, 3, 0, 0, _lib.stream_ptr()), "ia2c_actor_sample")
        assert np.array_equal(out["policy"][0, i].view(np.uint8), host(probs).view(np.uint8)), i
    pol = out["policy"][0, :, 0]
    counts = out["action_counts"][0].astype(np.int64)
    assert (pol == 0).sum() == 6
    assert not counts[pol == 0].any()
    assert np.abs(counts / counts.sum(-1, keepdims=True) - pol).max() < 0.03
    ref = EV.evaluate(np.zeros((N, 105)), E, K, T, 30, seed=77, table=out["policy"][0])
    assert np.array_equal(out["returns"][0], ref["returns"]) and np.array_equal(counts, ref["counts"])
