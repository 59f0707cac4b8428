"""Execute an UNMODIFIED reference script (ia2c.py / a2c_org_test.py) against the drop-in modules on the GPU.

Launched by tests/test_gpu_reference_scripts.py in a fresh interpreter whose module search path starts with
ia2c_b200/compat and ia2c_b200/compat_gym, so the script's own ``from ac_nets import *``, ``from belief_filter
import BeliefFilter``, ``import gymnasium`` and the gym entry point ``"Org:Org"`` (ia2c.py:20-38,
a2c_org_test.py:16-19) resolve to the product's drop-in modules — the reference's module files are never on the path.
The script source is read from oracle/_ref (or the reference checkout), its loop length is set by text substitution on
the in-memory source exactly as oracle/gen_golden.py did when it recorded the golden tapes, and it is exec'd as
``__main__``.

Replay (SURVEY.md §8 c4): the golden run's sampled actions and ``np.random.rand`` draws are injected through thin
wrappers around the PRODUCT classes (the wrapped method is always called), and the same wrappers record what the
script computed: env outputs, beliefs, losses, gradients and post-Adam parameters -> an .npz the test compares
with tests/golden/*.npz.

    python -P tests/reference_script_driver.py ia2c.py tests/golden/ia2c_E10.npz /tmp/out.npz
"""
import os
import re
import sys
from collections import defaultdict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    script, golden_path, out_path = sys.argv[1:4]
    for sub in ("compat_gym", "compat"):
        sys.path.insert(0, os.path.join(ROOT, "ia2c_b200", sub))
    sys.path.insert(0, ROOT)
    import torch

    from ia2c_b200 import belief as belief_mod
    from ia2c_b200 import nets, org_env
    from oracle import ref_runner   # only to locate + verify the staged reference sources

    ref, origin = ref_runner.find_reference()
    if ref is None:
        print("NO_REFERENCE", origin)
        sys.exit(3)
    g = np.load(golden_path, allow_pickle=False)
    rec = defaultdict(list)
    h = lambda t: t.detach().cpu().numpy().copy()

    # ---- actors: replay the recorded samples, record initial parameters
    a_init = nets.ActorNetwork.__init__

    def actor_init(self, name, *a, **k):
        a_init(self, name, *a, **k)
        self._tape_name = name
        rec[f"{name}/init"].append(h(self.net.flat))
        self.replay(g[f"{name}/sampled"])

    nets.ActorNetwork.__init__ = actor_init
    c_init = nets.CriticNetwork.__init__

    def critic_init(self, name, *a, **k):
        c_init(self, name, *a, **k)
        self._tape_name = name
        rec[f"{name}/init"].append(h(self.net.flat))

    nets.CriticNetwork.__init__ = critic_init
    c_upd, a_upd = nets.CriticNetwork.batch_update, nets.ActorNetwork.batch_update

    def critic_update(self, obs, act, target, *a, **k):
        n = self._tape_name
        rec[f"{n}/upd_obs"].append(h(obs))
        rec[f"{n}/upd_target"].append(h(target))
        rec[f"{n}/target_requires_grad"].append(np.asarray(bool(target.requires_grad)))
        c_upd(self, obs, act, target, *a, **k)
        rec[f"{n}/upd_loss"].append(np.asarray(self.losses[-1]))
        rec[f"{n}/upd_grad"].append(h(self.net.flat.grad))
        rec[f"{n}/upd_params"].append(h(self.net.flat))

    def actor_update(self, obs, act, adv, *a, **k):
        n = self._tape_name
        rec[f"{n}/upd_adv"].append(h(adv))
        rec[f"{n}/adv_requires_grad"].append(np.asarray(bool(adv.requires_grad)))
        a_upd(self, obs, act, adv, *a, **k)
        rec[f"{n}/upd_loss"].append(np.asarray(self.losses[-1]))
        rec[f"{n}/upd_grad"].append(h(self.net.flat.grad))   # running sum (Q2)
        rec[f"{n}/upd_params"].append(h(self.net.flat))

    nets.CriticNetwork.batch_update = critic_update
    nets.ActorNetwork.batch_update = actor_update

    # ---- belief filters: inject the recorded np.random.rand draws, record outputs
    b_init, b_upd = belief_mod.BeliefFilter.__init__, belief_mod.BeliefFilter.update
    n_filters = [0]
    real_rand = np.random.rand

    def bf_init(self, *a, **k):
        b_init(self, *a, **k)
        self._tape_idx = n_filters[0]
        n_filters[0] += 1
        self._u_tape = iter(g[f"bf{self._tape_idx}/u"])
        rec[f"bf{self._tape_idx}/filterAction"].append(np.array(self.filterAction))

    def bf_update(self, obs, prev):
        np.random.rand = lambda *shape: next(self._u_tape)
        try:
            ap, bprime, pred = b_upd(self, obs, prev)
        finally:
            np.random.rand = real_rand
        rec[f"bf{self._tape_idx}/ap"].append(np.array(ap))
        rec[f"bf{self._tape_idx}/bprime"].append(np.array(bprime))
        return ap, bprime, pred

    belief_mod.BeliefFilter.__init__ = bf_init
    belief_mod.BeliefFilter.update = bf_update

    # ---- envs: record outputs
    v_step, v_reset = org_env.OrgVecEnv.step, org_env.OrgVecEnv.reset

    def vec_step(self, actions):
        out = v_step(self, actions)
        if self.num_envs > 1:
            rec["env/obs"].append(np.array(out[0]))
            rec["env/reward"].append(np.array(out[1]))
            rec["env/truncated"].append(np.array(out[3]))
        return out

    def vec_reset(self, *a, **k):
        out = v_reset(self, *a, **k)
        if self.num_envs > 1:
            rec["env/reset_obs"].append(np.array(out[0]))
        return out

    org_env.OrgVecEnv.step, org_env.OrgVecEnv.reset = vec_step, vec_reset
    o_step = org_env.Org.step

    def org_step(self, action):
        out = o_step(self, action)
        rec["org/state"].append(np.asarray(self.state))
        rec["org/reward"].append(np.asarray(float(out[1])))
        rec["org/obs"].append(np.array(out[0], dtype=np.float64))
        return out

    org_env.Org.step = org_step

    seed = int(g["meta_seed"])
    torch.manual_seed(seed)
    np.random.seed(seed)
    if script == "ia2c.py":
        subs = [(r"^NUM_EPISODES = \d+", f"NUM_EPISODES = {int(g['meta_episodes'])}"), (r"^n_envs=\d+", f"n_envs={int(g['meta_n_envs'])}")]
    else:
        subs = [(r"^n_updates = \d+", f"n_updates = {int(g['meta_updates'])}")]
    src = open(os.path.join(ref, script)).read()
    for pat, rep in subs:
        src, n = re.subn(pat, rep, src, count=1, flags=re.M)
        assert n == 1, (script, pat)
    ns = {"__name__": "__main__", "__file__": os.path.join(ref, script)}
    exec(compile(src, os.path.join(ref, script), "exec"), ns)

    # the script resolved the drop-in modules, not the reference's
    import ac_nets
    import Org as org_module
    assert os.path.dirname(os.path.abspath(ac_nets.__file__)).endswith(os.path.join("ia2c_b200", "compat")), ac_nets.__file__
    assert os.path.dirname(os.path.abspath(org_module.__file__)).endswith(os.path.join("ia2c_b200", "compat")), org_module.__file__
    out = {k: np.stack(v) for k, v in rec.items()}
    if script == "ia2c.py":
        out["reward_lst"] = np.stack(ns["reward_lst"])
        out["critic_loss_window"] = np.array([ns["critic1"].critic_loss, ns["critic2"].critic_loss])
        out["actor_loss_window"] = np.array([ns["actor1"].actor_loss, ns["actor2"].actor_loss])
    else:
        out["critic_loss_window"] = np.array(ns["critic"].critic_loss)
        out["actor_loss_window"] = np.array(ns["actor"].actor_loss)
    out["origin"] = np.array(origin)
    np.savez_compressed(out_path, **out)
    print("REFERENCE_SCRIPT_DONE", script, origin)


if __name__ == "__main__":
    main()
