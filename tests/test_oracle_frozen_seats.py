"""oracle/frozen_seats.py: the trained seats of a frozen episode are those of the unfrozen oracle episode, and the frozen seats'
per-net state is what it was before it."""
import copy

import numpy as np
import pytest

from oracle import frozen_seats as FS
from oracle import loops as L
from ia2c_b200.trainer import reference_init


def _state(N, M, seed):
    actor, critic, fa = reference_init(N, M, seed=seed)
    return L.IA2CState(actor=actor.astype(np.float64), critic=critic.astype(np.float64), filter_action=fa, T=6)


@pytest.mark.parametrize("N, frozen", [(2, {1}), (3, {0, 2}), (9, {4})])
def test_frozen_oracle_matches_unfrozen_on_trained_seats(N, frozen):
    E, M, rng = 12, 5, np.random.RandomState(N)
    st = _state(N, M, seed=N)
    for _ in range(2):   # a second episode starts from Adam state the first one left
        act = rng.randint(0, 3, size=(st.T + 1, E, N))
        u = rng.rand(st.T + 1, E, N, N - 1)
        before, free = copy.deepcopy(st), copy.deepcopy(st)
        traj, upd = FS.frozen_episode(st, E, frozen, actions=act, u_belief=u)
        traj_f, upd_f = L.ia2c_episode(free, E, actions=act, u_belief=u)
        pred_f = L.partner_actions(traj_f, N)[1]
        for i in range(N):
            if i in frozen:
                assert np.array_equal(st.actor[i], before.actor[i]) and np.array_equal(st.critic[i], before.critic[i])
                assert np.array_equal(st.actor_grad_accum[i], before.actor_grad_accum[i])
                for a, b in ((st.adam_a[i], before.adam_a[i]), (st.adam_c[i], before.adam_c[i])):
                    assert a.t == b.t and np.array_equal(a.m, b.m) and np.array_equal(a.v, b.v)
                assert np.isnan(upd["critic_loss"][i]) and np.isnan(upd["actor_loss"][i])
                want = FS.NO_PREDICTION if N >= 9 else pred_f[:, :, i]
                assert np.all(traj["partner_pred"][:, :, i] == want)
            else:
                assert np.array_equal(st.actor[i], free.actor[i]) and np.array_equal(st.critic[i], free.critic[i])
                assert st.adam_a[i].t == free.adam_a[i].t and np.array_equal(st.adam_c[i].m, free.adam_c[i].m)
                assert upd["critic_loss"][i] == upd_f["critic_loss"][i] and upd["actor_loss"][i] == upd_f["actor_loss"][i]
                assert np.array_equal(traj["partner_pred"][:, :, i], pred_f[:, :, i])
        for i in frozen:   # the unfrozen twin, with the frozen rows copied back, is the frozen oracle
            free.actor[i], free.critic[i], free.actor_grad_accum[i] = st.actor[i], st.critic[i], st.actor_grad_accum[i]
            free.adam_a[i], free.adam_c[i] = copy.deepcopy(st.adam_a[i]), copy.deepcopy(st.adam_c[i])
        assert np.array_equal(np.stack(st.actor), np.stack(free.actor))
