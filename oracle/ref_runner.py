"""Run and time the UNMODIFIED reference scripts (thinclab/IA2C) on the host CPU.

TEST / MEASUREMENT INFRASTRUCTURE (see oracle/__init__.py): used by ``bench.py --impl reference``, by
bench.py's ``cpu_baseline`` leg and by the tests.  The reference files are executed from where they
lie — ``oracle/_ref/`` (staged by oracle/make_ref.py, digests verified) or the reference checkout
make_ref.REF_SRC names — with the two fixtures SURVEY.md §8 c1 names: ``oracle.gym_standin`` for the missing
gymnasium package (an in-process synchronous vector env; gymnasium's AsyncVectorEnv is not available)
and ``belief_filter_deprecated`` aliased as ``belief_filter`` (ia2c.py:23 imports a module the reference
does not ship, SURVEY.md Q1).  Script-level constants (NUM_EPISODES, n_envs, n_updates) are changed by
text substitution on the assignment line of the in-memory source, never on disk — the same mechanism
oracle/gen_golden.py uses to record the golden tapes.

    python -m oracle.ref_runner ia2c --envs 4096 --warmup 1 --episodes 3      # prints one JSON line
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import re
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def find_reference():
    """-> (directory, origin) of the unmodified reference files, or (None, reason)."""
    from oracle import make_ref

    try:
        make_ref.verify()
        return make_ref.REF_DST, "oracle/_ref (staged copy, sha256 verified)"
    except FileNotFoundError as exc:   # no manifest: a plain copy of the reference's files placed there is used as it is
        staged_err = str(exc)
        if all(os.path.exists(os.path.join(make_ref.REF_DST, f)) for f in make_ref.FILES):
            return make_ref.REF_DST, "oracle/_ref (copy without a manifest)"
    except Exception as exc:
        staged_err = str(exc)
    if os.path.isdir(make_ref.REF_SRC) and os.path.exists(os.path.join(make_ref.REF_SRC, "ia2c.py")):
        return make_ref.REF_SRC, make_ref.REF_SRC
    return None, staged_err


def import_reference(ref):
    """Import the reference's modules from ``ref`` (with the gymnasium stand-in and the Q1 alias)."""
    from oracle import gym_standin

    gym_standin.install()
    if ref not in sys.path:
        sys.path.insert(0, ref)
    import ac_nets
    import belief_filter_deprecated
    import Org as org_mod

    for m in (ac_nets, belief_filter_deprecated, org_mod):
        assert os.path.dirname(os.path.abspath(m.__file__)) == os.path.abspath(ref), (m.__file__, ref)
    sys.modules["belief_filter"] = belief_filter_deprecated  # Q1 alias
    return ac_nets, belief_filter_deprecated, org_mod


def run_script(ref, fname, subs, capture_stdout=True):
    """exec a reference script as __main__ with constants substituted in memory -> (namespace, stdout)."""
    src = open(os.path.join(ref, fname)).read()
    for pat, rep in subs:
        src, n = re.subn(pat, rep, src, count=1, flags=re.M)
        assert n == 1, (fname, pat)
    code = compile(src, os.path.join(ref, fname), "exec")
    ns = {"__name__": "__main__", "__file__": os.path.join(ref, fname)}
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf) if capture_stdout else contextlib.nullcontext():
        exec(code, ns)
    return ns, buf.getvalue()


def _threads():
    import torch

    try:
        from threadpoolctl import threadpool_info
        blas = max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
    except Exception:
        blas = 1
    return dict(torch_threads=torch.get_num_threads(), blas_threads=blas, host_logical_cpus=os.cpu_count())


def time_ia2c(n_envs, warmup, episodes, seed=0, warm_envs=0):
    """The reference's own ia2c.py main block (ia2c.py:41-134) at ``n_envs`` envs for warmup+episodes episodes.
    Episode boundaries are the script's ``envs.reset()`` calls (ia2c.py:72), time-stamped by a hook on the
    stand-in vector env (the fixture, not the reference).  ``warm_envs`` > 0 first runs the script once for one
    small episode (torch's lazy initialisation) so that a bounded run needs fewer full-size warm-up episodes.
    -> dict with per-episode seconds of the timed part."""
    import numpy as np
    import torch

    ref, origin = find_reference()
    if ref is None:
        raise FileNotFoundError(f"reference not available: {origin}")
    import_reference(ref)
    from oracle import gym_standin

    stamps = []
    v_reset = gym_standin.SyncVectorEnv.reset

    def stamped_reset(self_, *a, **k):
        stamps.append(time.perf_counter())
        return v_reset(self_, *a, **k)

    if warm_envs:
        run_script(ref, "ia2c.py", [(r"^NUM_EPISODES = \d+", "NUM_EPISODES = 1"), (r"^n_envs=\d+", f"n_envs={int(warm_envs)}")])
    gym_standin.SyncVectorEnv.reset = stamped_reset
    try:
        torch.manual_seed(seed)
        np.random.seed(seed)
        total = warmup + episodes
        run_script(ref, "ia2c.py", [(r"^NUM_EPISODES = \d+", f"NUM_EPISODES = {total}"), (r"^n_envs=\d+", f"n_envs={n_envs}")])
        stamps.append(time.perf_counter())
    finally:
        gym_standin.SyncVectorEnv.reset = v_reset
    assert len(stamps) == total + 1, (len(stamps), total)
    per_episode = [stamps[k + 1] - stamps[k] for k in range(total)][warmup:]
    agent_steps = n_envs * 2 * 30   # ia2c.py: 2 agents, STEPS_PER_EPISODE = 30
    sec = sum(per_episode)
    out = dict(script="ia2c.py", origin=origin, n_envs=n_envs, warmup=warmup, episodes=episodes, seconds=sec,
               per_episode_s=per_episode, ms_per_step=1e3 * sec / episodes, value=agent_steps * episodes / sec,
               unit="agent-steps/s")
    out.update(_threads())
    return out


def time_a2c_org(warmup, updates, seed=0):
    """The reference's a2c_org_test.py main block (a2c_org_test.py:27-92: one Org, 100 steps + critic and actor update
    per iteration).  Update boundaries are the script's per-update ``print`` (a2c_org_test.py:92)."""
    import builtins

    import numpy as np
    import torch

    ref, origin = find_reference()
    if ref is None:
        raise FileNotFoundError(f"reference not available: {origin}")
    import_reference(ref)
    stamps = [None]
    real_print = builtins.print

    def stamped_print(*a, **k):
        stamps.append(time.perf_counter())

    total = warmup + updates
    torch.manual_seed(seed)
    np.random.seed(seed)
    builtins.print = stamped_print
    try:
        stamps[0] = time.perf_counter()
        run_script(ref, "a2c_org_test.py", [(r"^n_updates = \d+", f"n_updates = {total}")], capture_stdout=False)
    finally:
        builtins.print = real_print
    assert len(stamps) == total + 1, (len(stamps), total)
    per_update = [stamps[k + 1] - stamps[k] for k in range(total)][warmup:]
    sec = sum(per_update)
    out = dict(script="a2c_org_test.py", origin=origin, warmup=warmup, updates=updates, seconds=sec,
               ms_per_step=1e3 * sec / updates, value=100 * updates / sec, unit="env-steps/s")
    out.update(_threads())
    return out


def time_acnets(rows_t, rows_e, n_features, n_critic, n_actor, warmup, updates, seed=0):
    """The reference's CriticNetwork/ActorNetwork.batch_update (ac_nets.py:62-80,112-127) on a2c_test.py's shapes
    (a2c_test.py:29-36,57,67: one-hot observations): one critic update + one actor update per iteration."""
    import numpy as np
    import torch
    import torch.nn.functional as F

    ref, origin = find_reference()
    if ref is None:
        raise FileNotFoundError(f"reference not available: {origin}")
    ac_nets, _, _ = import_reference(ref)
    torch.manual_seed(seed)
    rng = np.random.RandomState(seed)
    critic = ac_nets.CriticNetwork("c", n_features, n_critic, 5e-4)
    actor = ac_nets.ActorNetwork("a", n_features, n_actor, 1e-4, 0.01)
    T, E = rows_t, rows_e
    obs = F.one_hot(torch.from_numpy(rng.randint(0, n_features, size=(T, E))), n_features).float()
    act_c = torch.from_numpy(rng.randint(0, n_critic, size=(T, E, 1)).astype(np.float32))
    act_a = torch.from_numpy(rng.randint(0, n_actor, size=(T, E)).astype(np.float32))
    target = torch.from_numpy(rng.randn(T, E, 1).astype(np.float32))
    adv = torch.from_numpy(rng.randn(T, E, 1).astype(np.float32))
    times = []
    for k in range(warmup + updates):
        t0 = time.perf_counter()
        critic.batch_update(obs, act_c, target)
        actor.batch_update(obs, act_a, adv)
        times.append(time.perf_counter() - t0)
    sec = sum(times[warmup:])
    out = dict(script="ac_nets.py batch_update (critic + actor)", origin=origin, rows=T * E, n_features=n_features,
               warmup=warmup, updates=updates, seconds=sec, ms_per_step=1e3 * sec / updates, value=T * E * updates / sec,
               unit="rows/s")
    out.update(_threads())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("what", choices=["ia2c", "a2c_org", "acnets", "all"])
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--episodes", type=int, default=3)
    ap.add_argument("--rows-t", type=int, default=64)
    ap.add_argument("--rows-e", type=int, default=1024)
    ap.add_argument("--features", type=int, default=500)
    ap.add_argument("--warm-envs", type=int, default=0)
    a = ap.parse_args()
    if a.what == "all":   # one interpreter (one torch import) for the three CPU legs bench.py reports
        r = dict(ia2c=time_ia2c(a.envs, a.warmup, a.episodes, warm_envs=a.warm_envs), a2c_org=time_a2c_org(2, 10),
                 acnets=time_acnets(a.rows_t, a.rows_e, a.features, 6, 6, 1, 3))
    elif a.what == "ia2c":
        r = time_ia2c(a.envs, a.warmup, a.episodes, warm_envs=a.warm_envs)
    elif a.what == "a2c_org":
        r = time_a2c_org(a.warmup, a.episodes)
    else:
        r = time_acnets(a.rows_t, a.rows_e, a.features, 6, 6, a.warmup, a.episodes)
    print(json.dumps(r))


if __name__ == "__main__":
    main()
