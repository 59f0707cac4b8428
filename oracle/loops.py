"""CPU restatement of the reference's two training loops.  TEST INFRASTRUCTURE (see oracle/__init__.py).

  * ``ia2c_episode``  — one episode of ia2c.py:62-131 (rollout :72-102, critic phase :104-114,
    actor phase :116-129), generalised from 2 to N agents per SURVEY.md Appendix B
    ("Org-N", builder-defined; identical to the reference at N=2, which is what the goldens pin).
  * ``a2c_org_update`` — one update of a2c_org_test.py:43-92 (single joint agent, 9 actions, quirks Q4-Q7).

Randomness is injected: sampled actions (or the uniforms the CUDA sampler would consume) and the
belief filter's uniforms come from a tape, exactly as the CUDA path consumes them under replay.

Pinned against: tests/golden/ia2c_E10.npz, ia2c_E64.npz, a2c_org.npz (unmodified reference runs).
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from . import belief as B
from . import nets as NN
from .org import OrgBatchRef

N_ACT = 3      # actions per agent            (ia2c.py:44)
N_JOINT = 9    # critic outputs               (ia2c.py:45)
N_FEAT = 6     # observation features         (ia2c.py:43)


def others_of(i, n):
    """Modelled others of agent i in pair order (all other agents, ascending)."""
    return [j for j in range(n) if j != i]


def mode3(actions):
    """Most frequent action along the last axis, ties -> lowest action index (Appendix B)."""
    a = np.asarray(actions)
    counts = np.stack([(a == k).sum(-1) for k in range(N_ACT)], axis=-1)
    return counts.argmax(-1)


def joint_index(i, n, own, other):
    """Joint-action index for agent i: lower agent index is the high digit, partner (i+1) mod n (Q9)."""
    if i < (i + 1) % n:
        return own * N_ACT + other % N_ACT
    return other * N_ACT + own % N_ACT


@dataclass
class IA2CState:
    actor: np.ndarray            # [N, 105]
    critic: np.ndarray           # [N, 147]
    filter_action: np.ndarray    # [N, M, A] f64
    lr_c: float = 0.0002         # ia2c.py:26
    lr_a: float = 0.0001         # ia2c.py:27
    beta: float = 0.001          # ia2c.py:28
    gamma: float = 0.9           # ia2c.py:29
    T: int = 30                  # ia2c.py:31
    max_episode_steps: int = 30  # ia2c.py:37
    actor_grad_accum: np.ndarray = None  # Q2
    adam_a: list = field(default_factory=list)
    adam_c: list = field(default_factory=list)

    def __post_init__(self):
        n = self.actor.shape[0]
        dt = self.actor.dtype
        if self.actor_grad_accum is None:
            self.actor_grad_accum = np.zeros_like(self.actor)
        if not self.adam_a:
            self.adam_a = [NN.AdamRef(self.actor.shape[1], self.lr_a, dt) for _ in range(n)]
            self.adam_c = [NN.AdamRef(self.critic.shape[1], self.lr_c, dt) for _ in range(n)]


def ia2c_rollout(st: IA2CState, E, actions=None, u_act=None, u_belief=None):
    """Rollout of one episode.  actions int[T+1,E,N] (replay) or u_act [T+1,E,N] (inverse-CDF sampler);
    u_belief f64[T+1,E,N,K].  Returns the trajectory dict."""
    n = st.actor.shape[0]
    K = n - 1
    M = st.filter_action.shape[1]
    T = st.T
    env = OrgBatchRef(E, max_episode_steps=st.max_episode_steps)
    obs = env.reset()
    OBS = np.zeros((T + 1, E, N_FEAT), dtype=np.float32)
    REW = np.zeros((T, E), dtype=np.float64)
    STATE = np.zeros((T, E), dtype=np.int32)
    ACT = np.zeros((T + 1, E, n), dtype=np.int64)
    PRED = np.zeros((T + 1, E, n, K), dtype=np.int64)
    BEL = np.zeros((T + 1, E, n, K, M), dtype=np.float64)
    PROBS = np.zeros((T + 1, E, n, N_ACT), dtype=st.actor.dtype)
    prior = np.tile(B.uniform_prior(E, M)[:, None, None, :], (1, n, K, 1))  # Q12
    for t in range(T + 1):
        if t > 0:
            if n == 2:
                joint = ACT[t - 1, :, 0] * N_ACT + ACT[t - 1, :, 1] % N_ACT  # ia2c.py:84
                obs, r, _ = env.step_joint(joint)
            else:
                obs, r, _ = env.step_agents(ACT[t - 1])
            REW[t - 1] = r
            STATE[t - 1] = env.state_pre_reset
        OBS[t] = obs
        for i in range(n):
            p = NN.forward(st.actor[i], obs, N_FEAT, N_ACT, softmax=True)
            PROBS[t, :, i] = p
            if actions is not None:
                ACT[t, :, i] = actions[t, :, i]
            else:
                ACT[t, :, i] = NN.sample_inverse_cdf(p, u_act[t, :, i])
        for i in range(n):
            for jj, j in enumerate(others_of(i, n)):
                lik = B.likelihood_from_action(ACT[t, :, j], N_ACT)       # ia2c.py:53-58
                ap, bprime, _ = B.belief_update(st.filter_action[i], lik, prior[:, i, jj], u_belief[t, :, i, jj])
                PRED[t, :, i, jj] = ap
                BEL[t, :, i, jj] = bprime
                prior[:, i, jj] = bprime                                    # rounded posterior is next prior (Q10)
    return dict(obs=OBS, reward=REW, state=STATE, act=ACT, pred=PRED, belief=BEL, probs=PROBS,
                ep_return=REW.sum(0),
                # env state after the episode's T steps (and their autoresets), in the device's layout
                env_state=env.state.astype(np.int32), env_hist=env.reward.copy(),
                env_cls=np.stack([env.prev_cls, env.cls], axis=-1).astype(np.uint8), env_elapsed=env.elapsed.astype(np.int32))


def partner_actions(traj, n):
    """true / predicted partner action per agent: mode over the modelled others."""
    ACT, PRED = traj["act"], traj["pred"]
    true_p = np.zeros_like(ACT)
    pred_p = np.zeros_like(ACT)
    for i in range(n):
        true_p[:, :, i] = mode3(ACT[:, :, others_of(i, n)])
        pred_p[:, :, i] = mode3(PRED[:, :, i, :])
    return true_p, pred_p


def ia2c_update(st: IA2CState, traj):
    """Critic phase then actor phase (ia2c.py:104-129).  Mutates ``st``; returns diagnostics."""
    n = st.actor.shape[0]
    dt = st.actor.dtype
    T = st.T
    OBS, ACT = traj["obs"], traj["act"]
    obs, nobs = OBS[:T], OBS[1:T + 1]
    rew = traj["reward"].astype(np.float32).astype(dt)  # reward enters the trajectory as float32 (ia2c.py:99)
    true_p, pred_p = partner_actions(traj, n)
    E = obs.shape[1]
    out = dict(critic_loss=[], critic_grad=[], critic_target=[], adv=[], actor_loss=[], actor_grad=[])
    idx = {}
    for i in range(n):
        idx[i] = dict(
            nja=joint_index(i, n, ACT[1:T + 1, :, i], pred_p[1:T + 1, :, i]),   # ia2c.py:104-105
            jt=joint_index(i, n, ACT[:T, :, i], true_p[:T, :, i]),              # ia2c.py:112
            ja=joint_index(i, n, ACT[:T, :, i], pred_p[:T, :, i]),              # ia2c.py:120-121
        )
    for i in range(n):  # critic phase (residual gradient: target carries grad, Q8)
        loss, grad, target = NN.critic_loss_grad(st.critic[i], obs, idx[i]["jt"], rew, N_FEAT, N_JOINT,
                                                 next_obs=nobs, next_act=idx[i]["nja"], gamma_mask=st.gamma)
        st.critic[i] = st.adam_c[i].step(st.critic[i], grad)
        out["critic_loss"].append(loss), out["critic_grad"].append(grad)
        out["critic_target"].append(target.reshape(T, E))
    for i in range(n):  # actor phase, advantage from the UPDATED critic (ia2c.py:116-127)
        rows = np.arange(T * E)
        Qn = NN.forward(st.critic[i], nobs, N_FEAT, N_JOINT)[rows, idx[i]["nja"].reshape(-1)]
        Qc = NN.forward(st.critic[i], obs, N_FEAT, N_JOINT)[rows, idx[i]["ja"].reshape(-1)]
        adv = (rew.reshape(-1) + dt.type(st.gamma) * Qn) - Qc
        loss, grad, _ = NN.actor_loss_grad(st.actor[i], obs, ACT[:T, :, i], adv, st.beta, N_FEAT, N_ACT)
        st.actor_grad_accum[i] = st.actor_grad_accum[i] + grad          # no zero_grad (Q2)
        st.actor[i] = st.adam_a[i].step(st.actor[i], st.actor_grad_accum[i])
        out["adv"].append(adv.reshape(T, E)), out["actor_loss"].append(loss)
        out["actor_grad"].append(st.actor_grad_accum[i].copy())
    return {k: np.stack(v) for k, v in out.items()}


def ia2c_episode(st, E, actions=None, u_act=None, u_belief=None):
    traj = ia2c_rollout(st, E, actions=actions, u_act=u_act, u_belief=u_belief)
    upd = ia2c_update(st, traj)
    return traj, upd


# ----------------------------------------------------------------------------------------------
# a2c_org_test.py: single joint agent on ONE Org instance (rows duplicated, Q6)

@dataclass
class A2COrgState:
    actor: np.ndarray            # [147]  (6 -> 6 -> 6 -> 9, softmax)
    critic: np.ndarray           # [147]
    lr_c: float = 0.00005        # a2c_org_test.py:32
    lr_a: float = 0.0001         # a2c_org_test.py:31
    beta: float = 0.01           # a2c_org_test.py:30
    gamma: float = 0.99          # a2c_org_test.py:29
    T: int = 100                 # a2c_org_test.py:24
    rows: int = 2                # n_envs buffer rows (a2c_org_test.py:22)

    def __post_init__(self):
        dt = self.actor.dtype
        self.actor_grad_accum = np.zeros_like(self.actor)
        self.adam_a = NN.AdamRef(self.actor.size, self.lr_a, dt)
        self.adam_c = NN.AdamRef(self.critic.size, self.lr_c, dt)
        self.env = OrgBatchRef(1, max_episode_steps=None)
        self.env.reset()
        self.pending_action = None


def a2c_org_update(st: A2COrgState, sampled):
    """One update.  ``sampled``: the T (first update: T+1) joint actions drawn by the reference's sampler,
    in call order.  Returns diagnostics; mutates ``st``."""
    dt = st.actor.dtype
    T, Rr = st.T, st.rows
    sampled = list(sampled)
    if st.pending_action is None:
        st.pending_action = sampled.pop(0)  # a2c_org_test.py:56-60 (ep == 0 only)
    S = np.zeros((T, Rr, N_FEAT), dtype=np.float32)
    ACT = np.zeros((T, Rr), dtype=np.int64)
    REW = np.zeros((T, Rr), dtype=np.float64)
    for t in range(T):
        obs, r, _ = st.env.step_joint(np.array([st.pending_action]))
        nxt = sampled.pop(0)
        REW[t] = r[0]
        S[t] = obs[0]            # in-place aliasing: stored "state" is already the post-step obs (Q4)
        ACT[t] = st.pending_action
        st.pending_action = nxt
    rew = REW.astype(np.float32).astype(dt)
    # masks == 0 (Q5): critic target is the reward; the second forward pass gets zero gradient
    closs, cgrad, target = NN.critic_loss_grad(st.critic, S, ACT, rew, N_FEAT, N_JOINT)
    st.critic = st.adam_c.step(st.critic, cgrad)
    # actor: adv = Q_cur - V with V = sum(Q * d), d from a second, differentiable forward (Q7)
    rows = np.arange(T * Rr)
    Q = NN.forward(st.critic, S, N_FEAT, N_JOINT)
    d = NN.forward(st.actor, S, N_FEAT, N_JOINT, softmax=True)
    V = (Q * d).sum(-1)
    Qcur = Q[rows, ACT.reshape(-1)]
    adv = Qcur - V
    # first pass to get dL/dadv = neglogp/B, then the extra term through V: dV/dy_k = d_k (Q_k - V)
    _, _, dl_dadv = NN.actor_loss_grad(st.actor, S, ACT, adv, st.beta, N_FEAT, N_JOINT)
    extra_dy = (-dl_dadv)[:, None] * d * (Q - V[:, None])
    aloss, agrad, _ = NN.actor_loss_grad(st.actor, S, ACT, adv, st.beta, N_FEAT, N_JOINT, adv_extra_dy=extra_dy)
    st.actor_grad_accum = st.actor_grad_accum + agrad
    st.actor = st.adam_a.step(st.actor, st.actor_grad_accum)
    return dict(states=S, actions=ACT, reward=REW, target=target.reshape(T, Rr), adv=adv.reshape(T, Rr),
                critic_loss=closs, critic_grad=cgrad, actor_loss=aloss, actor_grad=st.actor_grad_accum.copy())
