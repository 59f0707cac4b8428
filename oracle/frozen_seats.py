"""Frozen seats (ia2c_train_episode_frozen): the oracle episode with some seats frozen.

A frozen seat acts as before, and nothing of it is updated.  Every seat's critic, actor gradient and beliefs read only the
trajectory and that seat's own state, so the episode is the unfrozen episode (``loops.ia2c_episode``; with a per-env pool,
``env_partners`` supplies the actions it replays) followed by:
  * the frozen seats' per-net state restored (parameters, Adam moments and steps, actor gradient sum);
  * their losses set to NaN;
  * for N >= 9, their partner predictions set to 0xFF ("no prediction": the whole-episode belief kernel skips their rows).
"""
import copy

import numpy as np

from . import loops as L

NO_PREDICTION = 0xFF


def frozen_episode(st, E, frozen, **episode_kw):
    """One episode of ``st`` (mutated) with the seats in ``frozen`` frozen.  ``episode_kw`` goes to ``loops.ia2c_episode``.
    Returns (traj, upd) as it does, with ``traj["partner_pred"]`` [T+1, E, N] added."""
    n = st.actor.shape[0]
    keep = {i: (st.actor[i].copy(), st.critic[i].copy(), st.actor_grad_accum[i].copy(), copy.deepcopy(st.adam_a[i]),
                copy.deepcopy(st.adam_c[i])) for i in frozen}
    traj, upd = L.ia2c_episode(st, E, **episode_kw)
    traj["partner_pred"] = L.partner_actions(traj, n)[1]
    for i, (a, c, g, adam_a, adam_c) in keep.items():
        st.actor[i], st.critic[i], st.actor_grad_accum[i], st.adam_a[i], st.adam_c[i] = a, c, g, adam_a, adam_c
        upd["critic_loss"][i] = upd["actor_loss"][i] = np.nan
        if n >= 9:
            traj["partner_pred"][:, :, i] = NO_PREDICTION
    return traj, upd
