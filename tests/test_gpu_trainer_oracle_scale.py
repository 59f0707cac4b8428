"""The IA2C trainer against the oracle as users run it: default kernel selection, device Philox sampling, no dumps, at the shapes
of the benchmark and the many-agent configs, with time limits inside the episode, hyper-parameters other than the defaults and
several episodes, for IA2CTrainer and for every run of IA2CRuns / IA2CRunsMany.

Before each episode the oracle is loaded from the device (parameters, Adam moments and steps, the actor's running gradient sum),
so every episode is checked from exactly the inputs its kernels had; the end state of the previous episode was itself compared
with the oracle.  The oracle regenerates the episode's Philox uniforms (oracle/philox.py), checks every sampled action against
its inverse CDF at the device's observations, replays the device's actions and compares the rest: trajectory, belief records,
env state and step counters bit for bit, gradients, losses, parameters and Adam moments per agent within 1e-5."""
import numpy as np
import pytest
import torch

from oracle import belief as B
from oracle import loops as L
from oracle import nets as NN
from oracle import philox as P
from tests.helpers import host, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-5
SAMPLER_TOL, SAMPLER_FLIPS = 1e-5, 1e-3   # |u - CDF boundary| of an action that differs from the oracle's; share of such draws
DEFAULTS = dict(gamma=0.9, beta=0.001, lr_actor=0.0001, lr_critic=0.0002)
SHARED = ("obs", "reward", "act", "partner_true", "partner_pred", "belief_records", "env_state", "env_hist", "env_cls", "env_elapsed",
          "ep_return", "loss_out", "actor_params", "critic_params", "actor_grad", "critic_grad", "actor_grad_accum", "actor_m", "actor_v",
          "critic_m", "critic_v", "actor_step", "critic_step")


def chunk_len(T, E, N):
    """Time-chunk length of the gradient kernels (chunk_plan in csrc/trainer.cu): one resident wave of 148 x 2 x 128 threads."""
    c = min(max(148 * 2 * 128 // (E * N), 1), T)
    return -(-T // c)


def assert_path(tr, N, M, path, actor):
    """The kernels a case claims to pin are the ones its trainer selected."""
    from ia2c_b200 import _lib
    f = tr.desc.flags
    fused = bool(tr.lib.ia2c_rollout_fused_supported(N, M))
    if path == "fused":      # rollout_fused_kernel<N, M> with the critic-gradient stage
        assert fused and f & _lib.FLAG_FUSED_ROLLOUT and f & _lib.FLAG_FUSED_CRITIC
    elif path == "step":     # env_step_kernel, actor_step_kernel, belief_pairs_kernel, critic_grad_kernel
        assert N <= 8 and not fused and not f & (_lib.FLAG_FUSED_ROLLOUT | _lib.FLAG_FUSED_CRITIC)
    elif path == "many":     # rollout_many_kernel, belief_pairs_episode_kernel, critic_grad_kernel
        assert 9 <= N <= 256 and tr.lib.ia2c_belief_supports_episode(N, M)
        assert not f & (_lib.FLAG_FUSED_ROLLOUT | _lib.FLAG_ROLLOUT_PER_STEP | _lib.FLAG_BELIEF_PER_STEP)
    elif path == "table":    # per-step kernels with belief_pairs_table_kernel (K >= 32)
        assert N - 1 >= 32 and f & _lib.FLAG_BELIEF_PER_STEP and not f & _lib.FLAG_FUSED_ROLLOUT
    else:
        raise ValueError(path)
    assert bool(f & _lib.FLAG_ACTOR_COLUMNS) == (actor == "columns")


def buffers(obj, r=None):
    """Device buffers of a trainer, or of run r of a batch, under the trainer's names."""
    return obj.run_view(r) if r is not None else {k: getattr(obj, k) for k in SHARED + ("filter_action",)}


def oracle_state(b, hp, T, max_steps):
    """An fp64 oracle holding exactly what the device holds before the episode."""
    g = {k: host(b[k]).astype(np.float64) for k in ("actor_params", "critic_params", "actor_grad_accum", "actor_m", "actor_v",
                                                     "critic_m", "critic_v")}
    st = L.IA2CState(actor=g["actor_params"], critic=g["critic_params"], filter_action=host(b["filter_action"]),
                     lr_c=float(hp["lr_critic"]), lr_a=float(hp["lr_actor"]),
                     beta=float(np.float32(hp["beta"])), gamma=float(np.float32(hp["gamma"])),   # the kernels take them as float32
                     T=T, max_episode_steps=max_steps or None, actor_grad_accum=g["actor_grad_accum"])
    a_step, c_step = host(b["actor_step"]), host(b["critic_step"])
    for i in range(st.actor.shape[0]):
        st.adam_a[i].m, st.adam_a[i].v, st.adam_a[i].t = g["actor_m"][i], g["actor_v"][i], int(a_step[i])
        st.adam_c[i].m, st.adam_c[i].v, st.adam_c[i].t = g["critic_m"][i], g["critic_v"][i], int(c_step[i])
    return st


def check_sampler(probs, u, act):
    """Every sampled action is the oracle's inverse-CDF draw, except where the uniform lies on a CDF boundary to within fp32
    rounding of the probabilities."""
    u = u.astype(np.float64)
    flip = NN.sample_inverse_cdf(probs, u) != act
    if flip.any():
        cdf = np.cumsum(probs, -1)[..., :2] / probs.sum(-1, keepdims=True)
        gap = np.abs(cdf[flip] - u[flip][:, None]).min(-1)
        assert gap.max() < SAMPLER_TOL, f"{int(flip.sum())} actions differ from the oracle's, max distance to a boundary {gap.max():.3g}"
    assert flip.mean() <= SAMPLER_FLIPS, f"{flip.mean():.2e} of the actions differ from the oracle's"


def check_episode(b, st, seed, episode, E, N, M, T, env_offset=0):
    """One finished episode of the device (buffers b) against the oracle state st taken before it."""
    d = {k: host(v) for k, v in b.items()}
    idx = (env_offset + np.arange(E))[:, None] * N + np.arange(N)[None, :]
    u_act = np.stack([P.uniform_f32(seed, P.STREAM_ACTION, episode, t, idx) for t in range(T + 1)])
    u_bel = np.stack([P.belief_uniforms(seed, episode, t, idx, N - 1) for t in range(T + 1)])
    act = d["act"].astype(np.int64)
    assert act.max() <= 2
    traj, upd = L.ia2c_episode(st, E, actions=act, u_belief=u_bel)
    # bit for bit: trajectory, sampler, final belief records, env state, step counters
    assert np.array_equal(d["obs"], traj["obs"])
    check_sampler(traj["probs"], u_act, act)
    assert np.array_equal(d["reward"], traj["reward"].astype(np.float32))
    true_p, pred_p = L.partner_actions(traj, N)
    assert np.array_equal(d["partner_true"], true_p) and np.array_equal(d["partner_pred"], pred_p)
    assert np.array_equal(d["ep_return"], traj["ep_return"])
    rec = d["belief_records"]
    assert np.array_equal(rec[..., :M], B.to_hundredths(traj["belief"][T]))
    assert np.array_equal(rec[..., 6], traj["pred"][T])
    assert not rec[..., M:6].any() and not rec[..., 7].any()
    for k in ("env_state", "env_hist", "env_cls", "env_elapsed"):
        assert np.array_equal(d[k], traj[k]), k
    assert np.array_equal(d["actor_step"], [a.t for a in st.adam_a]) and np.array_equal(d["critic_step"], [a.t for a in st.adam_c])
    # per agent within 1e-5: gradients (with their loss entries), parameters, Adam moments, losses
    err = {}

    def worst(name, value):
        err[name] = max(err.get(name, 0.0), value)

    for i in range(N):
        worst("critic_grad", rel_err(d["critic_grad"][i, :-1], upd["critic_grad"][i]))
        worst("critic_grad_loss", rel_err(d["critic_grad"][i, -1], upd["critic_loss"][i]))
        worst("critic_loss", rel_err(d["loss_out"][0, i], upd["critic_loss"][i]))
        worst("critic_params", rel_err(d["critic_params"][i], st.critic[i]))
        worst("critic_m", rel_err(d["critic_m"][i], st.adam_c[i].m))
        worst("critic_v", rel_err(d["critic_v"][i], st.adam_c[i].v))
        worst("actor_grad_accum", rel_err(d["actor_grad_accum"][i], upd["actor_grad"][i]))
        worst("actor_params", rel_err(d["actor_params"][i], st.actor[i]))
        worst("actor_m", rel_err(d["actor_m"][i], st.adam_a[i].m))
        worst("actor_v", rel_err(d["actor_v"][i], st.adam_a[i].v))
        # the actor loss is a mean of signed terms that cancel at many rows: judged on the scale of its terms
        scale = max(abs(float(upd["actor_loss"][i])), float(np.abs(upd["adv"][i]).mean()))
        for got in (d["loss_out"][1, i], d["actor_grad"][i, -1]):
            worst("actor_loss", abs(float(got) - float(upd["actor_loss"][i])) / scale)
    assert max(err.values()) < RTOL, {k: f"{v:.2e}" for k, v in err.items()}


def check_episodes(obj, subjects, episodes, E, N, M, T, max_steps):
    """Trains `episodes` episodes of obj (a trainer or a batch of runs) and checks each subject (buffers, seed, hyper-parameters)
    after each of them."""
    for _ in range(episodes):
        episode = obj.episode
        states = [oracle_state(b, hp, T, max_steps) for b, _, hp in subjects]
        obj.train_episode()
        torch.cuda.synchronize()
        for (b, seed, hp), st in zip(subjects, states):
            check_episode(b, st, seed, episode, E, N, M, T, env_offset=getattr(obj, "env_offset", 0))


# id: (N, M, E, T, max_episode_steps, episodes, kernel path, actor kernel, chunk length of the gradient kernels or None,
#      hyper-parameters and trainer options other than the defaults)
CASES = {
    # the bench headline: fused rollout + fused critic stage, column actor kernel; 256 critic and 128 actor partial rows per net
    # (chunks of 8, 8, 8 and 6 steps)
    "4096x2": (2, 5, 4096, 30, 30, 3, "fused", "columns", 8, {}),
    "4096x2-pipe": (2, 5, 4096, 30, 30, 3, "fused", "pipe", None, dict(actor_kernel="pipe")),
    # autoresets at t = 12 and 24, hyper-parameters other than the defaults
    "4096x2-reset": (2, 5, 4096, 30, 12, 3, "fused", "columns", 8, dict(gamma=0.99, beta=0.05, lr_actor=1e-3, lr_critic=2e-3)),
    "2048x2-M3": (2, 3, 2048, 30, 30, 3, "fused", "columns", 4, {}),
    # every fused instantiation, E not a multiple of the block's 8 (N <= 4) or 4 envs
    "1001x3": (3, 5, 1001, 30, 30, 3, "fused", "columns", 3, {}),
    "1001x4": (4, 5, 1001, 30, 30, 3, "fused", "columns", 4, {}),
    "1001x5": (5, 5, 1001, 30, 30, 3, "fused", "columns", 5, {}),
    "1001x6-reset": (6, 5, 1001, 30, 7, 3, "fused", "columns", 5, dict(gamma=0.5)),
    "1001x7": (7, 5, 1001, 30, 30, 3, "fused", "columns", 6, {}),
    "1001x8": (8, 5, 1001, 30, 30, 3, "fused", "columns", 8, {}),
    # N <= 8 without a fused instantiation: the per-step kernels
    "4096x2-M2": (2, 2, 4096, 30, 30, 3, "step", "columns", 8, {}),
    "1001x4-M4": (4, 4, 1001, 30, 30, 3, "step", "columns", 4, {}),
    "1001x7-M6": (7, 6, 1001, 30, 30, 3, "step", "columns", 6, {}),
    # N > 8: rollout_many_kernel and the whole-episode belief kernel in its steady-state (no dumps, Philox) form
    "600x9-reset": (9, 2, 600, 30, 12, 3, "many", "columns", 5, {}),
    "1050x12": (12, 4, 1050, 30, 30, 3, "many", "columns", 10, {}),
    "4736x16": (16, 6, 4736, 30, 30, 2, "many", "columns", 30, {}),   # cfg4 / cfg5 regime: one chunk of 30 per thread
    "200x33": (33, 3, 200, 10, 10, 3, "many", "columns", 2, {}),
    "1184x64": (64, 5, 1184, 8, 8, 2, "many", "columns", 8, {}),       # cfg4's agent count
    "40x130": (130, 5, 40, 4, 4, 2, "many", "pipe", None, {}),         # N > 64: pipelined actor kernel by default
    "24x256": (256, 5, 24, 3, 3, 2, "many", "pipe", None, {}),         # cfg5's agent count
    # belief_pairs_table_kernel (K >= 32), the per-step belief form, for the model counts the whole-episode cases above leave out
    "64x36-M2-table": (36, 2, 64, 6, 6, 2, "table", "columns", 1, dict(belief_kernel="step")),
    "64x40-M4-table": (40, 4, 64, 6, 6, 2, "table", "columns", 1, dict(belief_kernel="step")),
    "64x44-M6-table": (44, 6, 64, 6, 6, 2, "table", "columns", 1, dict(belief_kernel="step")),
}


@pytest.mark.parametrize("case", list(CASES))
def test_trainer_matches_oracle(case):
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    N, M, E, T, max_steps, episodes, path, actor, chunk, opts = CASES[case]
    hp = {**DEFAULTS, **{k: v for k, v in opts.items() if k in DEFAULTS}}
    kw = {k: v for k, v in opts.items() if k not in DEFAULTS}
    seed = 1000 + 16 * N + M
    tr = IA2CTrainer(E, n_agents=N, n_models=M, steps_per_episode=T, max_episode_steps=max_steps, seed=seed,
                     init=reference_init(N, M, seed=seed), **hp, **kw)
    assert_path(tr, N, M, path, actor)
    if chunk is not None:
        assert chunk_len(T, E, N) == chunk
    check_episodes(tr, [(buffers(tr), seed, hp)], episodes, E, N, M, T, max_steps)


RUNS_HYPER = dict(gamma=[0.9, 0.97, 0.6], beta=[0.001, 0.02, 0.1], lr_actor=[1e-4, 5e-4, 2e-3], lr_critic=[2e-4, 1e-3, 5e-5])


@pytest.mark.parametrize("kind, N, M, E, max_steps, R", [("runs", 3, 5, 333, 30, 3), ("many", 12, 4, 300, 12, 2)])
def test_runs_match_oracle(kind, N, M, E, max_steps, R):
    """Each run of a batch against the oracle directly, with its own seed and hyper-parameters."""
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    from ia2c_b200.trainer import reference_init
    T = 30
    seeds = [41, 2 ** 40 + 3, 7][:R]   # a Philox key with a non-zero high word (reference_init itself takes 32-bit seeds)
    hyper = {k: v[:R] for k, v in RUNS_HYPER.items()}
    cls = IA2CRuns if kind == "runs" else IA2CRunsMany
    batch = cls(E, seeds, n_agents=N, n_models=M, steps_per_episode=T, max_episode_steps=max_steps,
                init=[reference_init(N, M, seed=r) for r in range(R)], **hyper)
    subjects = [(buffers(batch, r), seeds[r], {k: v[r] for k, v in hyper.items()}) for r in range(R)]
    check_episodes(batch, subjects, 3 if kind == "runs" else 2, E, N, M, T, max_steps)


@pytest.mark.parametrize("N, M, E", [(2, 5, 4096), (4, 4, 1001), (12, 4, 1050), (40, 4, 64)])
def test_dumps_change_no_bytes(N, M, E):
    """Parity dumps select the other form of the belief kernels (and add stores to the others): a trainer with dumps must
    write the same bytes as one without into every buffer the two share."""
    from ia2c_b200.trainer import IA2CTrainer, reference_init
    init = reference_init(N, M, seed=N)
    kw = dict(belief_kernel="step") if N - 1 >= 32 else {}
    a = IA2CTrainer(E, n_agents=N, n_models=M, seed=77, init=init, **kw)
    b = IA2CTrainer(E, n_agents=N, n_models=M, seed=77, init=init, dumps=True, **kw)
    assert a.desc.flags == b.desc.flags
    for ep in range(3):
        a.train_episode(), b.train_episode()
        torch.cuda.synchronize()
        for name in SHARED:
            assert np.array_equal(host(getattr(a, name)), host(getattr(b, name))), (name, ep)
