"""Oracle pin of the E-env form of the a2c_org_test.py update (oracle/a2c_envs.py) against the unmodified reference's run
(tests/golden/a2c_org.npz), and of the trainer's default initialisation against the run's initial parameters."""
import numpy as np
import pytest

from oracle import a2c_envs as A
from oracle import philox as PX
from tests.helpers import rel_err

RTOL = 1e-5


def golden_slots(g, update, T):
    """The reference's recorded draws of one update in slot order [T+1, 1]; slot 0 only exists at update 0."""
    s = g["act1/sampled"]
    if update == 0:
        return s[:T + 1].reshape(T + 1, 1)
    lo = T + 1 + (update - 1) * T
    return np.concatenate([[-1], s[lo:lo + T]]).reshape(T + 1, 1)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_envs_form_at_one_env_reproduces_the_reference(golden, dtype):
    g = golden("a2c_org.npz")
    lr_c, lr_a, beta, _gamma = g["meta_hyper"]
    T = int(g["meta_T"])
    st = A.A2COrgEnvsState(actor=g["act1/init"][0].astype(dtype), critic=g["main1/init"][0].astype(dtype), E=1,
                           lr_c=lr_c, lr_a=lr_a, beta=beta, T=T)
    for upd in range(int(g["meta_updates"])):
        out = A.a2c_org_update_envs(st, actions=golden_slots(g, upd, T))
        es = slice(upd * T, (upd + 1) * T)
        assert np.array_equal(out["actions"][:, 0], g["org/action"][es])
        assert np.array_equal(out["reward"][:, 0], g["org/reward"][es])          # fp64 bit-exact
        assert np.array_equal(out["states"][:, 0], g["main1/upd_obs"][upd][:, 0])
        assert rel_err(out["critic_loss"], g["main1/upd_loss"][upd]) < RTOL
        assert rel_err(out["critic_grad"], g["main1/upd_grad"][upd]) < RTOL
        assert rel_err(st.critic, g["main1/upd_params"][upd]) < RTOL
        assert rel_err(out["adv"][:, 0], g["act1/upd_adv"][upd][:, 0, 0]) < RTOL
        assert rel_err(out["actor_loss"], g["act1/upd_loss"][upd]) < RTOL
        assert rel_err(out["actor_grad_accum"], g["act1/upd_grad"][upd]) < RTOL
        assert rel_err(st.actor, g["act1/upd_params"][upd]) < RTOL


def test_envs_are_independent_rows():
    """E envs with distinct action tapes are E one-env runs: the trajectory of env e equals a one-env run on column e."""
    rng = np.random.RandomState(5)
    T, E = 12, 3
    init = rng.randn(2, 147).astype(np.float32) * 0.3
    tapes = rng.randint(0, 9, size=(2, T + 1, E))
    st = A.A2COrgEnvsState(actor=init[0].copy(), critic=init[1].copy(), E=E, T=T)
    outs = [A.a2c_org_update_envs(st, actions=tapes[k]) for k in range(2)]
    for e in range(E):
        one = A.A2COrgEnvsState(actor=init[0].copy(), critic=init[1].copy(), E=1, T=T)
        for k in range(2):
            o = A.a2c_org_update_envs(one, actions=tapes[k][:, e:e + 1])
            assert np.array_equal(o["reward"][:, 0], outs[k]["reward"][:, e])
            assert np.array_equal(o["states"][:, 0], outs[k]["states"][:, e])


def test_action_uniforms_follow_the_counter_layout():
    u = A.action_uniforms(7, 3, T=4, E=5)
    assert u.shape == (5, 5) and u.dtype == np.float32
    for s in range(5):
        for e in range(5):
            x0 = PX.draw(7, 3, 3, s, np.array([e], dtype=np.uint64))[0][0]
            assert u[s, e] == np.float32(int(x0) >> 8) * np.float32(2.0 ** -24)
    assert np.all((u >= 0) & (u < 1))


def test_reference_init_reproduces_the_recorded_run(golden):
    from ia2c_b200.a2c import a2c_reference_init
    g = golden("a2c_org.npz")
    actor, critic = a2c_reference_init(int(g["meta_seed"]))
    assert np.array_equal(actor, g["act1/init"][0])
    assert np.array_equal(critic, g["main1/init"][0])
