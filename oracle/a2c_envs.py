"""CPU restatement of one a2c_org_test.py update for E independent envs.  TEST INFRASTRUCTURE (see oracle/__init__.py).

``loops.a2c_org_update`` restates the reference exactly: ONE Org instance whose state fills both of the script's buffer
rows (SURVEY.md Q6).  This is the same update with one row per env for E envs, the form the native trainer
(ia2c_b200/a2c.py, csrc/a2c.cu) computes: a mean over the reference's duplicated rows equals the mean over one row, so at
E = 1 it reproduces the reference run (tests/test_oracle_a2c.py pins it to tests/golden/a2c_org.npz).

Randomness is injected in the native trainer's slot order: slot 0 is update 0's first draw (from the reset observation),
slot t + 1 the draw after step t.  Either the actions themselves (replay) or the uniforms of the inverse-CDF sampler;
``action_uniforms`` regenerates the Philox uniforms the kernel draws (stream 3, DESIGN.md §4).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import nets as NN
from . import philox as PX
from .loops import N_FEAT, N_JOINT
from .org import OrgBatchRef

STREAM_A2C_ACTION = 3


def action_uniforms(seed, update, T, E):
    """float32 [T+1, E]: the uniform of slot s for env e (its index within its run) at ``update``: Philox key = seed,
    counter = (e, s | 3 << 16, update), the 24-bit float of the action sampler."""
    return np.stack([PX.uniform_f32(seed, STREAM_A2C_ACTION, update, s, np.arange(E, dtype=np.uint64)) for s in range(T + 1)])


@dataclass
class A2COrgEnvsState:
    actor: np.ndarray            # [147]
    critic: np.ndarray           # [147]
    E: int = 1
    lr_c: float = 0.00005        # a2c_org_test.py:32
    lr_a: float = 0.0001         # a2c_org_test.py:31
    beta: float = 0.01           # a2c_org_test.py:30
    T: int = 100                 # a2c_org_test.py:24

    def __post_init__(self):
        dt = self.actor.dtype
        self.actor_grad_accum = np.zeros_like(self.actor)
        self.adam_a = NN.AdamRef(self.actor.size, self.lr_a, dt)
        self.adam_c = NN.AdamRef(self.critic.size, self.lr_c, dt)
        self.env = OrgBatchRef(self.E, max_episode_steps=None)   # reset once, never again (Q6)
        self.pending_action = None
        self.update = 0


def a2c_org_update_envs(st: A2COrgEnvsState, actions=None, u=None):
    """One update of all E envs.  ``actions`` int[T+1, E] or ``u`` float[T+1, E] (inverse-CDF uniforms), both in slot
    order; slot 0 is used at update 0 only.  Mutates ``st``; returns the trajectory, the sampled slots and diagnostics."""
    dt = st.actor.dtype
    T, E = st.T, st.E

    def draw(slot, obs):
        if actions is not None:
            return np.asarray(actions[slot], dtype=np.int64).reshape(E)
        p = NN.forward(st.actor, obs, N_FEAT, N_JOINT, softmax=True)
        return NN.sample_inverse_cdf(p, np.asarray(u[slot]).reshape(E))

    slots = np.full((T + 1, E), -1, dtype=np.int64)
    if st.pending_action is None:   # a2c_org_test.py:56-60 (update 0 only)
        obs0 = np.concatenate([np.eye(3, dtype=np.float32)[st.env.prev_cls], np.eye(3, dtype=np.float32)[st.env.cls]], -1)
        st.pending_action = draw(0, obs0)
        slots[0] = st.pending_action
    S = np.zeros((T, E, N_FEAT), dtype=np.float32)
    ACT = np.zeros((T, E), dtype=np.int64)
    REW = np.zeros((T, E), dtype=np.float64)
    for t in range(T):
        obs, r, _ = st.env.step_joint(st.pending_action)
        S[t], ACT[t], REW[t] = obs, st.pending_action, r   # stored pair: (post-step obs, action taken) (Q4)
        st.pending_action = draw(t + 1, obs)
        slots[t + 1] = st.pending_action
    rew = REW.astype(np.float32).astype(dt)
    # masks == 0 (Q5): the critic target is the reward
    closs, cgrad, _ = NN.critic_loss_grad(st.critic, S, ACT, rew, N_FEAT, N_JOINT)
    st.critic = st.adam_c.step(st.critic, cgrad)
    # actor: adv = Q[a] - V, V = sum(Q * d), gradient through d (Q7); loops.a2c_org_update spells out the two passes
    rows = np.arange(T * E)
    Q = NN.forward(st.critic, S, N_FEAT, N_JOINT)
    d = NN.forward(st.actor, S, N_FEAT, N_JOINT, softmax=True)
    V = (Q * d).sum(-1)
    adv = Q[rows, ACT.reshape(-1)] - V
    _, _, dl_dadv = NN.actor_loss_grad(st.actor, S, ACT, adv, st.beta, N_FEAT, N_JOINT)
    extra_dy = (-dl_dadv)[:, None] * d * (Q - V[:, None])
    aloss, agrad, _ = NN.actor_loss_grad(st.actor, S, ACT, adv, st.beta, N_FEAT, N_JOINT, adv_extra_dy=extra_dy)
    st.actor_grad_accum = st.actor_grad_accum + agrad           # never zeroed (Q2)
    st.actor = st.adam_a.step(st.actor, st.actor_grad_accum)
    st.update += 1
    return dict(states=S, actions=ACT, reward=REW, slots=slots, ep_return=REW.sum(0), adv=adv.reshape(T, E),
                critic_loss=closs, critic_grad=cgrad, actor_loss=aloss, actor_grad=agrad,
                actor_grad_accum=st.actor_grad_accum.copy(), env_state=st.env.state.copy(), env_hist=st.env.reward.copy(),
                pending_action=st.pending_action.copy())
