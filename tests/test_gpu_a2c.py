"""GPU tests of the native A2C trainer (ia2c_b200/a2c.py, csrc/a2c.cu) for the a2c_org_test.py loop: the recorded reference
run replayed through it, Philox sampling against the E-env oracle (oracle/a2c_envs.py), batches of runs against single
runs byte for byte, checkpoint / resume, determinism and the launch count."""
import re

import numpy as np
import pytest

from oracle import a2c_envs as A
from oracle import nets as NN
from oracle.loops import N_FEAT, N_JOINT
from tests.helpers import host, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-5
BUFFERS = ("actor_params", "critic_params", "actor_grad", "critic_grad", "actor_grad_accum", "actor_m", "actor_v", "critic_m",
           "critic_v", "actor_step", "critic_step", "env_state", "env_hist", "env_cls", "env_elapsed", "pending_action",
           "ep_return", "obs", "act", "reward", "loss_out")


def golden_slots(g, update, T):
    """The reference's recorded draws of one update in slot order [T+1, 1]; slot 0 (update 0 only) is a placeholder later."""
    s = g["act1/sampled"]
    if update == 0:
        return s[:T + 1].reshape(T + 1, 1)
    lo = T + 1 + (update - 1) * T
    return np.concatenate([[0], s[lo:lo + T]]).reshape(T + 1, 1)


def kernel_slots(tr, first):
    """The actions the trainer drew in its last update, in slot order [T+1, R*E] (slot 0 is meaningful at update 0 only)."""
    act = host(tr.act).astype(np.int64)
    return np.concatenate([act[:1] if first else np.zeros_like(act[:1]), act[1:], host(tr.pending_action)[None].astype(np.int64)])


def same_bytes(a, b):
    return host(a).tobytes() == host(b).tobytes()


def test_golden_replay():
    """E = 1, R = 1 with the reference's 401 recorded draws injected: env bit-exact over all 400 steps, losses, gradients and
    parameters within 1e-5, returns and loss windows as the reference printed them."""
    from ia2c_b200.a2c import A2COrgTrainer
    from tests.conftest import load_golden
    g = load_golden("a2c_org.npz")
    lr_c, lr_a, beta, _gamma = g["meta_hyper"]
    T = int(g["meta_T"])
    tr = A2COrgTrainer(1, seeds=0, steps_per_update=T, lr_actor=lr_a, lr_critic=lr_c, beta=beta,
                       init=[(g["act1/init"][0], g["main1/init"][0])])
    printed = [line.split() for line in str(g["stdout"]).strip().splitlines()]
    for upd in range(int(g["meta_updates"])):
        tr.inject(golden_slots(g, upd, T))
        stats = tr.train_update(sync_stats=True)
        es = slice(upd * T, (upd + 1) * T)
        assert np.array_equal(host(tr.act)[:, 0], g["org/action"][es])
        assert np.array_equal(host(tr.obs)[:, 0], g["main1/upd_obs"][upd][:, 0])
        assert np.array_equal(host(tr.reward)[:, 0], g["org/reward"][es].astype(np.float32))
        assert host(tr.env_hist)[0] == g["org/reward"][es][-1] and host(tr.env_state)[0] == g["org/state"][es][-1]
        ret = 0.0
        for r in g["org/reward"][es]:
            ret += float(r)
        assert stats["ep_return"][0, 0] == ret                                     # fp64, summed in step order
        assert rel_err(stats["critic_loss"][0], g["main1/upd_loss"][upd]) < RTOL
        assert rel_err(host(tr.critic_grad)[0, :147], g["main1/upd_grad"][upd]) < RTOL
        assert rel_err(host(tr.critic_params)[0], g["main1/upd_params"][upd]) < RTOL
        assert rel_err(stats["actor_loss"][0], g["act1/upd_loss"][upd]) < RTOL
        assert rel_err(host(tr.actor_grad_accum)[0], g["act1/upd_grad"][upd]) < RTOL   # running sum, Q7 term included
        assert rel_err(host(tr.actor_params)[0], g["act1/upd_params"][upd]) < RTOL
        ep, ret_s, crit_w, act_w = printed[upd]
        assert int(ep) == upd
        printed_ret = float(re.search(r"tensor\((.*)\)", ret_s).group(1))   # the reference's float32 sum, 4 decimals
        assert abs(stats["ep_return"][0, 0] - printed_ret) <= 1e-6 * abs(printed_ret) + 5e-5
        # windows are means of losses that may cancel (the actor's): judge them on the scale of the losses averaged
        crit_scale, act_scale = np.abs(g["main1/upd_loss"][:upd + 1]).max(), np.abs(g["act1/upd_loss"][:upd + 1]).max()
        assert abs(stats["critic_loss_window"][0] - float(crit_w)) <= RTOL * crit_scale
        assert abs(stats["actor_loss_window"][0] - float(act_w)) <= RTOL * act_scale
    assert abs(stats["critic_loss_window"][0] - g["critic_loss_window"]) <= RTOL * crit_scale
    assert abs(stats["actor_loss_window"][0] - g["actor_loss_window"]) <= RTOL * act_scale


@pytest.mark.parametrize("E", [1, 37, 300])
def test_philox_mode_is_replayable_by_the_oracle(E):
    """Performance mode: the kernel's draws against the oracle's inverse CDF at the regenerated Philox uniforms (ulp-level
    flips only), then the kernel's own draws fed to the oracle as a tape: env bit-exact, everything else within 1e-5."""
    from ia2c_b200.a2c import A2COrgTrainer, a2c_reference_init
    T, seed = 100, 1234
    actor, critic = a2c_reference_init(0)
    tr = A2COrgTrainer(E, seeds=seed, steps_per_update=T, init=[(actor, critic)])
    st = A.A2COrgEnvsState(actor=actor.astype(np.float64), critic=critic.astype(np.float64), E=E, T=T)
    flips, draws = 0, 0
    for upd in range(5):
        obs0 = np.concatenate([np.eye(3)[st.env.prev_cls], np.eye(3)[st.env.cls]], -1)
        tr.train_update(sync_stats=True)
        got = kernel_slots(tr, upd == 0)
        u = A.action_uniforms(seed, upd, T, E)
        obs = host(tr.obs).astype(np.float64)
        probs = NN.forward(st.actor, obs, N_FEAT, N_JOINT, softmax=True).reshape(T, E, N_JOINT)
        resampled = NN.sample_inverse_cdf(probs, u[1:])
        flips += int((resampled != got[1:]).sum())
        draws += resampled.size
        if upd == 0:
            p0 = NN.forward(st.actor, obs0, N_FEAT, N_JOINT, softmax=True)
            flips += int((NN.sample_inverse_cdf(p0, u[0]) != got[0]).sum())
            draws += E
        out = A.a2c_org_update_envs(st, actions=got)
        assert np.array_equal(host(tr.obs), out["states"])
        assert np.array_equal(host(tr.act), out["actions"])
        assert np.array_equal(host(tr.reward), out["reward"].astype(np.float32))
        assert np.array_equal(host(tr.env_hist), out["env_hist"]) and np.array_equal(host(tr.env_state), out["env_state"])
        assert np.allclose(host(tr.ep_return), out["ep_return"], rtol=1e-12, atol=0)
        assert rel_err(host(tr.loss_out)[0, 0], out["critic_loss"]) < RTOL
        assert rel_err(host(tr.critic_grad)[0, :147], out["critic_grad"]) < RTOL
        assert rel_err(host(tr.critic_params)[0], st.critic) < RTOL
        # the actor loss is a mean of T * E signed terms of size |adv|: judge its error on that scale
        scale = max(abs(float(out["actor_loss"])), float(np.abs(out["adv"]).mean()))
        assert abs(host(tr.loss_out)[1, 0] - out["actor_loss"]) <= RTOL * scale
        assert rel_err(host(tr.actor_grad)[0, :147], out["actor_grad"]) < RTOL
        assert rel_err(host(tr.actor_grad_accum)[0], out["actor_grad_accum"]) < RTOL
        assert rel_err(host(tr.actor_params)[0], st.actor) < RTOL
    assert flips / draws < 2e-3, (flips, draws)


@pytest.mark.parametrize("E", [1, 37])
def test_runs_are_byte_identical_to_single_runs(E):
    """R = 4 runs with a repeated seed and distinct hyper-parameters: every run's slice of every buffer is byte for byte the
    single run with its seed and hyper-parameters; scalar and per-run-list hyper-parameters give identical bytes."""
    from ia2c_b200.a2c import A2COrgTrainer
    T, seeds = 20, [5, 5, 9, 11]
    lr_a, lr_c, beta = [1e-4, 3e-4, 2e-4, 1e-3], [5e-5, 1e-4, 2e-5, 5e-4], [0.01, 0.05, 0.0, 0.02]
    batch = A2COrgTrainer(E, seeds=seeds, steps_per_update=T, lr_actor=lr_a, lr_critic=lr_c, beta=beta)
    single = [A2COrgTrainer(E, seeds=s, steps_per_update=T, lr_actor=a, lr_critic=c, beta=b)
              for s, a, c, b in zip(seeds, lr_a, lr_c, beta)]
    for _ in range(3):
        batch.train_update()
        for tr in single:
            tr.train_update()
    for r, tr in enumerate(single):
        view = batch.run_view(r)
        for k in BUFFERS:
            assert same_bytes(view[k], getattr(tr, k)), (r, k)
    assert not same_bytes(batch.run_view(0)["actor_params"], batch.run_view(1)["actor_params"])   # same seed, other lr
    scalar = A2COrgTrainer(E, seeds=seeds, steps_per_update=T, lr_actor=2e-4, lr_critic=1e-4, beta=0.03)
    listed = A2COrgTrainer(E, seeds=seeds, steps_per_update=T, lr_actor=[2e-4] * 4, lr_critic=[1e-4] * 4, beta=[0.03] * 4)
    for _ in range(2):
        scalar.train_update(), listed.train_update()
    for k in BUFFERS:
        assert same_bytes(getattr(scalar, k), getattr(listed, k)), k


def test_checkpoint_resume_is_byte_identical(tmp_path):
    """state_dict after k updates, then continuing in a fresh trainer, gives the bytes of never stopping (pending action,
    reward history, Adam state, gradient running sum and update counter included)."""
    from ia2c_b200.a2c import A2COrgTrainer
    E, T, seeds = 37, 30, [3, 4]
    straight = A2COrgTrainer(E, seeds=seeds, steps_per_update=T)
    first = A2COrgTrainer(E, seeds=seeds, steps_per_update=T)
    for _ in range(4):
        ref = straight.train_update(sync_stats=True)
    for _ in range(2):
        first.train_update(sync_stats=True)
    path = tmp_path / "a2c.pt"
    first.save(path)
    resumed = A2COrgTrainer(E, seeds=[0, 0], steps_per_update=T)   # other seeds and init: the checkpoint restores them
    resumed.load(path)
    for _ in range(2):
        stats = resumed.train_update(sync_stats=True)
    for k in BUFFERS:
        assert same_bytes(getattr(resumed, k), getattr(straight, k)), k
    assert np.array_equal(stats["critic_loss_window"], ref["critic_loss_window"])


def test_same_seed_twice_gives_identical_bytes():
    from ia2c_b200.a2c import A2COrgTrainer
    a, b = A2COrgTrainer(64, seeds=[7, 8]), A2COrgTrainer(64, seeds=[7, 8])
    for _ in range(3):
        a.train_update(), b.train_update()
    for k in BUFFERS:
        assert same_bytes(getattr(a, k), getattr(b, k)), k


def test_four_launches_per_update():
    from ia2c_b200 import _lib
    from ia2c_b200.a2c import A2COrgTrainer
    tr = A2COrgTrainer(300, seeds=[1, 2, 3])
    tr.train_update()
    before = _lib.launch_count()
    for _ in range(3):
        tr.train_update()
    assert _lib.launch_count() - before == 12
