"""Generate the golden fixtures under tests/golden/ by EXECUTING THE UNMODIFIED REFERENCE.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Run in the build container only:

    python -m oracle.gen_golden            # needs /root/reference, writes tests/golden/*.npz

The reference files are imported / exec'd from where they lie under
/root/reference; nothing is copied into this repo.  Two fixtures make them run
(SURVEY.md §8 c1): ``oracle.gym_standin`` stands in for the missing gymnasium
package, and ``belief_filter_deprecated`` is aliased as ``belief_filter``
(ia2c.py:23 imports a module the reference does not ship, SURVEY.md Q1).
Script-level constants (NUM_EPISODES, n_envs, n_updates) are changed by text
substitution on the assignment line of the in-memory source, never on disk.

Instrumentation wraps the reference's own classes (the wrapped method is always
called) and records, in call order: initial state_dicts, every sampled action,
every ``np.random.rand`` draw, env outputs, belief inputs/outputs, and for each
``batch_update`` its inputs, loss, gradients and post-step parameters.  These
tapes are both the replay stream injected into the CUDA path and the expected
outputs it is compared with.
"""
from __future__ import annotations

import os
import re
import sys
from collections import defaultdict

import numpy as np

REF = os.environ.get("IA2C_REFERENCE", "/root/reference")
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


class Tape:
    def __init__(self):
        self.d = defaultdict(list)

    def add(self, key, value):
        self.d[key].append(np.array(value))

    def save(self, path, **extra):
        out = {k: np.stack(v) for k, v in self.d.items()}
        out.update({k: np.asarray(v) for k, v in extra.items()})
        np.savez_compressed(path, **out)
        print(f"wrote {path}: {len(out)} arrays, {os.path.getsize(path)/1024:.1f} KiB")


def _import_reference():
    from oracle import gym_standin

    gym_standin.install()
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import torch  # noqa: F401
    import ac_nets
    import belief_filter_deprecated
    import Org as org_mod

    sys.modules["belief_filter"] = belief_filter_deprecated  # Q1 alias
    return ac_nets, belief_filter_deprecated, org_mod


def _sd(net):
    return {k: v.detach().clone().numpy() for k, v in net.state_dict().items()}


SD_KEYS = ["l1.weight", "l1.bias", "l2.weight", "l2.bias", "l3.weight", "l3.bias"]


def _flat(sd):
    return np.concatenate([np.asarray(sd[k]).reshape(-1) for k in SD_KEYS])


def _flat_grads(net):
    g = dict(net.named_parameters())
    return np.concatenate([g[k].grad.detach().numpy().reshape(-1) for k in SD_KEYS])


class Instrument:
    """Wraps the reference's classes so that every call lands on a Tape."""

    def __init__(self, tape, ac_nets, bfd, org_mod):
        import torch

        self.tape, self.ac_nets, self.bfd, self.org_mod, self.torch = tape, ac_nets, bfd, org_mod, torch
        self.names = {}
        self.bf_index = {}
        self.saved = []

    def _patch(self, obj, attr, new):
        self.saved.append((obj, attr, getattr(obj, attr)))
        setattr(obj, attr, new)

    def restore(self):
        for obj, attr, old in reversed(self.saved):
            setattr(obj, attr, old)
        self.saved.clear()

    def install(self):
        tape, torch = self.tape, self.torch
        A, C, B = self.ac_nets.ActorNetwork, self.ac_nets.CriticNetwork, self.bfd.BeliefFilter
        inst = self

        c_init, a_init = C.__init__, A.__init__

        def critic_init(self_, name, *a, **k):
            c_init(self_, name, *a, **k)
            inst.names[id(self_)] = name
            tape.add(f"{name}/init", _flat(_sd(self_.net)))

        def actor_init(self_, name, *a, **k):
            a_init(self_, name, *a, **k)
            inst.names[id(self_)] = name
            tape.add(f"{name}/init", _flat(_sd(self_.net)))

        self._patch(C, "__init__", critic_init)
        self._patch(A, "__init__", actor_init)

        sample = A.sample_action

        def sample_action(self_, obs, grad=False):
            act = sample(self_, obs, grad=grad)
            tape.add(f"{inst.names[id(self_)]}/sampled", act.detach().numpy())
            return act

        self._patch(A, "sample_action", sample_action)

        c_upd, a_upd = C.batch_update, A.batch_update

        def critic_update(self_, obs, act, target, *a, **k):
            n = inst.names[id(self_)]
            tape.add(f"{n}/upd_obs", obs.detach().numpy())
            tape.add(f"{n}/upd_act", act.detach().numpy())
            tape.add(f"{n}/upd_target", target.detach().numpy())
            c_upd(self_, obs, act, target, *a, **k)
            tape.add(f"{n}/upd_loss", np.asarray(self_.losses[-1]))
            tape.add(f"{n}/upd_grad", _flat_grads(self_.net))
            tape.add(f"{n}/upd_params", _flat(_sd(self_.net)))

        def actor_update(self_, obs, act, adv, *a, **k):
            n = inst.names[id(self_)]
            tape.add(f"{n}/upd_obs", obs.detach().numpy())
            tape.add(f"{n}/upd_act", act.detach().numpy())
            tape.add(f"{n}/upd_adv", adv.detach().numpy())
            a_upd(self_, obs, act, adv, *a, **k)
            tape.add(f"{n}/upd_loss", np.asarray(self_.losses[-1]))
            tape.add(f"{n}/upd_grad", _flat_grads(self_.net))  # running sum (Q2)
            tape.add(f"{n}/upd_params", _flat(_sd(self_.net)))

        self._patch(C, "batch_update", critic_update)
        self._patch(A, "batch_update", actor_update)

        b_init, b_upd = B.__init__, B.update

        def bf_init(self_, *a, **k):
            b_init(self_, *a, **k)
            idx = len(inst.bf_index)
            inst.bf_index[id(self_)] = idx
            tape.add(f"bf{idx}/filterAction", self_.filterAction)
            tape.add(f"bf{idx}/prior0", self_.prior)

        def bf_update(self_, obs, prev):
            idx = inst.bf_index[id(self_)]
            tape.add(f"bf{idx}/obs", obs)
            tape.add(f"bf{idx}/prev", prev)
            inst.rand_log = []
            ap, bprime, pred = b_upd(self_, obs, prev)
            (u,) = inst.rand_log
            inst.rand_log = None
            tape.add(f"bf{idx}/u", u)
            tape.add(f"bf{idx}/ap", ap)
            tape.add(f"bf{idx}/bprime", bprime)
            tape.add(f"bf{idx}/prediction", pred)
            return ap, bprime, pred

        self._patch(B, "__init__", bf_init)
        self._patch(B, "update", bf_update)

        self.rand_log = None
        np_rand = np.random.rand

        def rand(*shape):
            out = np_rand(*shape)
            if inst.rand_log is not None:
                inst.rand_log.append(out.copy())
            return out

        self._patch(np.random, "rand", rand)

        from oracle import gym_standin

        v_step, v_reset = gym_standin.SyncVectorEnv.step, gym_standin.SyncVectorEnv.reset

        def vec_step(self_, actions):
            tape.add("env/action", np.array([int(a) for a in actions]))
            out = v_step(self_, actions)
            tape.add("env/obs", out[0])
            tape.add("env/reward", out[1])
            tape.add("env/truncated", out[3])
            tape.add("env/state_pre_reset", self_.last_pre_reset_state)
            tape.add("env/state_post", np.array([e.state for e in self_.envs]))
            return out

        def vec_reset(self_, *a, **k):
            out = v_reset(self_, *a, **k)
            tape.add("env/reset_obs", out[0])
            return out

        self._patch(gym_standin.SyncVectorEnv, "step", vec_step)
        self._patch(gym_standin.SyncVectorEnv, "reset", vec_reset)

        o_step = self.org_mod.Org.step

        def org_step(self_, action):
            out = o_step(self_, action)
            if inst.record_single_env:
                tape.add("org/action", np.asarray(int(action)))
                tape.add("org/state", np.asarray(self_.state))
                tape.add("org/reward", np.asarray(float(out[1])))
                tape.add("org/obs", np.array(out[0], dtype=np.float64))
            return out

        self.record_single_env = False
        self._patch(self.org_mod.Org, "step", org_step)
        return self


def _run_script(fname, subs, capture_stdout=True):
    """exec a reference script as __main__ with constants substituted in memory."""
    import contextlib
    import io

    src = open(os.path.join(REF, fname)).read()
    for pat, rep in subs:
        src, n = re.subn(pat, rep, src, count=1, flags=re.M)
        assert n == 1, (fname, pat)
    code = compile(src, os.path.join(REF, fname), "exec")
    ns = {"__name__": "__main__", "__file__": os.path.join(REF, fname)}
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf) if capture_stdout else contextlib.nullcontext():
        exec(code, ns)
    return ns, buf.getvalue()


def gen_ia2c(n_envs, episodes, seed, out_name):
    import torch

    ac_nets, bfd, org_mod = _import_reference()
    tape = Tape()
    inst = Instrument(tape, ac_nets, bfd, org_mod).install()
    try:
        torch.manual_seed(seed)
        np.random.seed(seed)
        ns, stdout = _run_script(
            "ia2c.py",
            [(r"^NUM_EPISODES = \d+", f"NUM_EPISODES = {episodes}"), (r"^n_envs=\d+", f"n_envs={n_envs}")],
        )
    finally:
        inst.restore()
    reward_lst = np.stack(ns["reward_lst"])  # [episodes, E] float64 episode returns (ia2c.py:102,131)
    tape.save(
        os.path.join(OUT, out_name),
        reward_lst=reward_lst,
        stdout=np.array(stdout),
        meta_n_envs=n_envs,
        meta_episodes=episodes,
        meta_seed=seed,
        meta_T=ns["STEPS_PER_EPISODE"],
        meta_hyper=np.array([ns["LR_C"], ns["LR_A"], ns["BETA"], ns["GAMMA"]]),
        critic_loss_window=np.array([ns["critic1"].critic_loss, ns["critic2"].critic_loss]),
        actor_loss_window=np.array([ns["actor1"].actor_loss, ns["actor2"].actor_loss]),
    )


def gen_a2c_org(updates, seed, out_name):
    import torch

    ac_nets, bfd, org_mod = _import_reference()
    tape = Tape()
    inst = Instrument(tape, ac_nets, bfd, org_mod).install()
    inst.record_single_env = True
    try:
        torch.manual_seed(seed)
        np.random.seed(seed)
        ns, stdout = _run_script("a2c_org_test.py", [(r"^n_updates = \d+", f"n_updates = {updates}")])
    finally:
        inst.restore()
    tape.save(
        os.path.join(OUT, out_name),
        stdout=np.array(stdout),
        meta_updates=updates,
        meta_seed=seed,
        meta_T=ns["n_steps_per_update"],
        meta_hyper=np.array([ns["critic_lr"], ns["actor_lr"], ns["ent_coef"], ns["gamma"]]),
        critic_loss_window=np.array(ns["critic"].critic_loss),
        actor_loss_window=np.array(ns["actor"].actor_loss),
    )


def gen_org_table(out_name):
    """Exhaustive truth table of Org.step + a long random walk on one real Org instance."""
    _, _, org_mod = _import_reference()
    hist = [0.0, 1.0, -100.0, 6.6, -111.11, 0.123456789, 5.55]
    rows = []
    for s in range(5):
        for a in range(-2, 12):  # includes unknown action codes (Q16)
            for r in hist:
                for prev_cls in range(3):
                    env = org_mod.Org()
                    env.reset()
                    env.state, env.reward = s, r
                    env.observation[3:6] = np.eye(3)[prev_cls]
                    o, r2, d1, d2, _ = env.step(a)
                    rows.append((s, a, r, prev_cls, env.state, float(r2), *o, float(d1)))
    table = np.array(rows, dtype=np.float64)
    rng = np.random.RandomState(7)
    env = org_mod.Org()
    o0, _ = env.reset()
    acts = rng.randint(0, 9, size=4000)
    acts[rng.rand(4000) < 0.02] = 11  # sprinkle unknown codes
    ws, wr, wo = [], [], []
    for a in acts:
        o, r, _, _, _ = env.step(int(a))
        ws.append(env.state), wr.append(float(r)), wo.append(np.array(o))
    np.savez_compressed(
        os.path.join(OUT, out_name),
        table=table,
        table_cols=np.array("s,a,r,prev_cls,s2,r2,o0,o1,o2,o3,o4,o5,done"),
        reset_obs=np.array(o0, dtype=np.float64),
        walk_actions=acts,
        walk_state=np.array(ws),
        walk_reward=np.array(wr, dtype=np.float64),
        walk_obs=np.stack(wo),
    )
    print("wrote", out_name, table.shape)


def gen_belief(out_name):
    """Chained BeliefFilter.update calls on the real class: random models (M=5) and the papers' known models."""
    _, bfd, _ = _import_reference()
    out = {}
    for tag, M, A, E, known in (("rand5", 5, 3, 256, None), ("rand3", 3, 3, 64, None), ("rand5x5", 5, 5, 32, None),
                                ("org_known", 3, 3, 64, "org"), ("hvt_known", 5, 5, 32, "hvt")):
        np.random.seed(11)
        bf = bfd.BeliefFilter(M, A, E)
        if known == "org":  # constants quoted in comments at belief_filter_deprecated.py:32-33
            bf.filterAction = np.array([[0.8, 0.1, 0.1], [0.6, 0.2, 0.2], [0.4, 0.3, 0.3]])
            bf.filters = bf.filterAction.transpose()
        if known == "hvt":  # belief_filter_deprecated.py:36-37
            bf.filterAction = np.array([[0.8, 0.05, 0.05, 0.05, 0.05], [0.6, 0.1, 0.1, 0.1, 0.1],
                                        [0.4, 0.15, 0.15, 0.15, 0.15], [0.2, 0.2, 0.2, 0.2, 0.2],
                                        [0.1, 0.225, 0.225, 0.225, 0.225]])
            bf.filters = bf.filterAction.transpose()
        rng = np.random.RandomState(5)
        prior = bf.prior
        steps = 120
        obs_l, prev_l, u_l, ap_l, b_l, p_l, act_l = [], [], [], [], [], [], []
        np_rand = np.random.rand
        for t in range(steps):
            other = rng.randint(0, A, size=E)
            lik = np.ones((E, A)) * 0.1  # the likelihood of ia2c.py:53-58
            lik[np.arange(E), other] = 0.8
            if t % 7 == 3:  # also exercise general (non 0.8/0.1) likelihood rows
                lik = rng.rand(E, A)
            log = []

            def rec(*shape):
                x = np_rand(*shape)
                log.append(x.copy())
                return x

            np.random.rand = rec
            try:
                ap, bprime, pred = bf.update(lik, prior)
            finally:
                np.random.rand = np_rand
            obs_l.append(lik), prev_l.append(prior), u_l.append(log[0]), ap_l.append(ap)
            b_l.append(bprime), p_l.append(pred), act_l.append(other)
            prior = bprime
            if t % 30 == 29:
                prior = bf.prior  # episode boundary (Q12)
        out[f"{tag}/filterAction"] = bf.filterAction
        out[f"{tag}/prior0"] = bf.prior
        out[f"{tag}/other_action"] = np.stack(act_l)
        out[f"{tag}/obs"] = np.stack(obs_l)
        out[f"{tag}/prev"] = np.stack(prev_l)
        out[f"{tag}/u"] = np.stack(u_l)
        out[f"{tag}/ap"] = np.stack(ap_l)
        out[f"{tag}/bprime"] = np.stack(b_l)
        out[f"{tag}/prediction"] = np.stack(p_l)
        keep_envs(out, tag, BELIEF_KEEP_ENVS[tag])
    np.savez_compressed(os.path.join(OUT, out_name), **out)
    print("wrote", out_name)


# envs stored per belief case: the class updates every env row on its own, so a fixed subset of rows is a complete record
# of those rows, and it keeps belief_vectors.npz under 1 MB
BELIEF_KEEP_ENVS = {"rand5": 64, "rand3": 32, "rand5x5": 16, "org_known": 32, "hvt_known": 16}


def keep_envs(out, tag, n, seed=0):
    """Keep a fixed, seeded subset of n envs (the second axis) in every per-step array of one belief case; prior0 stays
    whole (it pins the class's initial prior), {tag}/env_index records the envs kept."""
    keep = np.sort(np.random.RandomState(seed).choice(out[f"{tag}/obs"].shape[1], n, replace=False))
    for k in ("other_action", "obs", "prev", "u", "ap", "bprime", "prediction"):
        out[f"{tag}/{k}"] = out[f"{tag}/{k}"][:, keep]
    out[f"{tag}/env_index"] = keep


def gen_acnets(out_name):
    """Direct batch_update / forward calls on the real ac_nets classes at several shapes."""
    import torch
    import torch.nn.functional as F

    ac_nets, _, _ = _import_reference()
    out = {}
    cases = [  # tag, T, E, F, critic outs, actor outs, one-hot input?
        ("org", 30, 8, 6, 9, 3, False),
        ("org9", 20, 4, 6, 9, 9, False),
        ("taxi", 16, 8, 500, 6, 6, True),
        ("dense", 12, 6, 11, 5, 4, False),
    ]
    for tag, T, E, Fd, J, A, onehot in cases:
        torch.manual_seed(3)
        rng = np.random.RandomState(9)
        critic = ac_nets.CriticNetwork("c", Fd, J, 2e-4)
        actor = ac_nets.ActorNetwork("a", Fd, A, 1e-4, 0.01)
        out[f"{tag}/critic_init"] = _flat(_sd(critic.net))
        out[f"{tag}/actor_init"] = _flat(_sd(actor.net))
        for it in range(3):
            if onehot:
                idx = torch.from_numpy(rng.randint(0, Fd, size=(T, E)))
                obs = F.one_hot(idx, Fd).float()
                idx2 = torch.from_numpy(rng.randint(0, Fd, size=(T, E)))
                nobs = F.one_hot(idx2, Fd).float()
            else:
                obs = torch.from_numpy(rng.randn(T, E, Fd).astype(np.float32))
                nobs = torch.from_numpy(rng.randn(T, E, Fd).astype(np.float32))
            cact = torch.from_numpy(rng.randint(0, J, size=(T, E, 1)).astype(np.float32))
            cnext = torch.from_numpy(rng.randint(0, J, size=(T, E)))
            aact = torch.from_numpy(rng.randint(0, A, size=(T, E)).astype(np.float32))
            rew = torch.from_numpy(rng.randn(T, E).astype(np.float32))
            mask = torch.from_numpy((rng.rand(T, E) < 0.8).astype(np.float32))
            gamma = 0.9
            # forward values (run_main / action_distribution)
            out[f"{tag}/{it}/Q"] = critic.run_main(obs).numpy()
            out[f"{tag}/{it}/P"] = actor.action_distribution(obs).numpy()
            # critic update with a target that carries its graph (ia2c.py:108-113, Q8)
            with_grad = it != 1
            qn = (critic.run_main(nobs, grad=with_grad) * F.one_hot(cnext, J).float()).sum(-1, keepdims=True)
            target = rew.unsqueeze(-1) + gamma * mask.unsqueeze(-1) * qn
            critic.batch_update(obs, cact, target)
            adv = torch.from_numpy(rng.randn(T, E, 1).astype(np.float32))
            actor.batch_update(obs, aact, adv)
            for k, v in dict(obs=obs, nobs=nobs, cact=cact, cnext=cnext, aact=aact, rew=rew, mask=mask, adv=adv,
                             target=target.detach()).items():
                out[f"{tag}/{it}/{k}"] = v.numpy()
            out[f"{tag}/{it}/target_has_grad"] = np.asarray(with_grad)
            out[f"{tag}/{it}/critic_loss"] = np.asarray(critic.losses[-1])
            out[f"{tag}/{it}/actor_loss"] = np.asarray(actor.losses[-1])
            out[f"{tag}/{it}/critic_grad"] = _flat_grads(critic.net)
            out[f"{tag}/{it}/actor_grad_accum"] = _flat_grads(actor.net)  # Σ of all grads so far (Q2)
            out[f"{tag}/{it}/critic_params"] = _flat(_sd(critic.net))
            out[f"{tag}/{it}/actor_params"] = _flat(_sd(actor.net))
        out[f"{tag}/dims"] = np.array([T, E, Fd, J, A, int(onehot)])
        out[f"{tag}/hyper"] = np.array([2e-4, 1e-4, 0.01, 0.9])
    np.savez_compressed(os.path.join(OUT, out_name), **out)
    print("wrote", out_name)


def main():
    os.makedirs(OUT, exist_ok=True)
    gen_org_table("org_table.npz")
    gen_belief("belief_vectors.npz")
    gen_acnets("acnets_updates.npz")
    gen_ia2c(n_envs=10, episodes=3, seed=0, out_name="ia2c_E10.npz")
    gen_ia2c(n_envs=64, episodes=2, seed=1, out_name="ia2c_E64.npz")
    gen_a2c_org(updates=4, seed=0, out_name="a2c_org.npz")


if __name__ == "__main__":
    main()
