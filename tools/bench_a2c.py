"""Native A2C trainer (A2COrgTrainer) for the a2c_org_test.py loop: time per update over a grid of (envs per run, runs),
against the drop-in class-API flow (compat Org / ac_nets driven the way a2c_org_test.py drives them) at one env.

For every (E, R): ms per update of all R runs from CUDA events around many warm updates, once back to back and once with the
L2 flushed (a 256 MiB buffer written) before every update, as tools/bench_runs.py does; env-steps/s = R * E * T per update
time.  The class-API iteration (100 env steps + critic and actor updates, one env) is timed with a host clock around whole
iterations that end in a device synchronise.  Prints one JSON line with the card's name, power limit and max SM clock
(read-only nvidia-smi query) taken in the same call.

    python tools/bench_a2c.py [--updates K] [--warmup W] [--class-iters N] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GRID = ((1, 1), (1, 64), (1, 1024), (64, 1), (64, 64), (4096, 1))
T = 100


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in out.split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as exc:   # the measurement stands without it, but says so
        return dict(name=f"unknown ({exc})")


def class_api_ms(iters, warmup):
    """ms per iteration of the a2c_org_test.py loop written against the drop-in modules (tests/test_gpu_compat.py's flow,
    sampling instead of replaying)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "ia2c_b200", "compat"))
    try:
        from ac_nets import ActorNetwork, CriticNetwork, F
        from Org import Org
    finally:
        sys.path.pop(0)
    n_rows, n_obs, n_act, gamma = 2, 6, 9, 0.99
    torch.manual_seed(0)
    env = Org()
    critic = CriticNetwork("main1", n_obs, n_act, 5e-5)
    actor = ActorNetwork("act1", n_obs, n_act, 1e-4, 0.01)
    states, _ = env.reset(seed=42)
    actions = actor.sample_action(torch.tensor(states).float(), grad=True)

    def iteration():
        nonlocal states, actions
        buf_s, buf_ns = torch.zeros(T, n_rows, n_obs), torch.zeros(T, n_rows, n_obs)
        buf_a, buf_na = torch.zeros(T, n_rows, 1), torch.zeros(T, n_rows, 1)
        buf_r, masks = torch.zeros(T, n_rows), torch.zeros(T, n_rows)
        for t in range(T):
            nxt, rew, terminated, _, _ = env.step(actions.detach().cpu().numpy())
            nxt_actions = actor.sample_action(torch.tensor(nxt).float(), grad=True)
            buf_r[t] = torch.tensor(rew)
            buf_s[t], buf_ns[t] = torch.tensor(states), torch.tensor(nxt)
            buf_a[t], buf_na[t] = actions.unsqueeze(-1), nxt_actions.unsqueeze(-1)
            masks[t] = torch.tensor(terminated)
            states, actions = nxt, nxt_actions
        q_next = critic.run_main(buf_ns, grad=True)
        oh_next = F.one_hot(buf_na.squeeze(-1).long(), num_classes=n_act).detach().float()
        target = buf_r.unsqueeze(-1) + gamma * masks.unsqueeze(-1) * (q_next * oh_next).sum(-1, keepdims=True)
        critic.batch_update(buf_s, buf_a, target)
        Q = critic.run_main(buf_s, grad=False)
        dist = actor.action_distribution(buf_s, grad=True)
        oh = F.one_hot(buf_a.squeeze(-1).long(), num_classes=n_act).float()
        actor.batch_update(buf_s, buf_a, (Q * oh).sum(-1, keepdims=True) - (Q * dist).sum(-1, keepdims=True))

    for _ in range(warmup):
        iteration()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        iteration()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--updates", type=int, default=50, help="timed updates per leg (>= 20)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--class-iters", type=int, default=10, help="timed class-API iterations")
    ap.add_argument("--quick", action="store_true", help="(E, R) = (1, 1) and (64, 1) only (a rehearsal)")
    a = ap.parse_args()
    if a.updates < 20:
        ap.error("--updates must be at least 20")

    import torch

    from ia2c_b200 import _lib
    from ia2c_b200.a2c import A2COrgTrainer

    _lib.require_cuda()
    torch.cuda.set_device(0)
    gpu = card()
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    K, W = a.updates, a.warmup

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def back_to_back(f):
        for _ in range(W):
            f()
        torch.cuda.synchronize()
        s, e = ev(), ev()
        s.record()
        for _ in range(K):
            f()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / K

    def flushed(f):
        marks = []
        for _ in range(K):
            flush_buf.zero_()
            m = (ev(), ev())
            m[0].record()
            f()
            m[1].record()
            marks.append(m)
        torch.cuda.synchronize()
        return sum(s.elapsed_time(e) for s, e in marks) / K

    grid = ((1, 1), (64, 1)) if a.quick else GRID
    rows = []
    for E, R in grid:
        tr = A2COrgTrainer(E, seeds=list(range(R)), steps_per_update=T)
        ms, ms_fl = back_to_back(tr.train_update), flushed(tr.train_update)
        steps = tr.env_steps_per_update()
        rows.append(dict(E=E, R=R, update_ms=round(ms, 4), update_ms_flushed=round(ms_fl, 4),
                         env_steps_per_s=round(steps / (ms * 1e-3), 1), env_steps_per_s_flushed=round(steps / (ms_fl * 1e-3), 1)))
        print(f"E={E:5d} R={R:5d}: {ms * 1e3:9.1f} us per update ({ms_fl * 1e3:9.1f} flushed), "
              f"{steps / (ms * 1e-3):.3e} env-steps/s", file=sys.stderr)
        del tr
    cls_ms = class_api_ms(a.class_iters, 2)
    native_1 = rows[0]["update_ms"]
    print(f"class API (E=1): {cls_ms:.2f} ms per iteration; native (1, 1) {native_1 * 1e3:.1f} us: "
          f"{cls_ms / native_1:.0f}x", file=sys.stderr)
    print(json.dumps(dict(tool="bench_a2c", gpu=gpu, T=T, updates=K, warmup=W,
                          l2="back to back, and with a 256 MiB buffer written before every update",
                          rows=rows, class_api_ms_per_iteration=round(cls_ms, 3),
                          class_api_env_steps_per_s=round(T / (cls_ms * 1e-3), 1),
                          speedup_1x1_vs_class_api=round(cls_ms / native_1, 1))))


if __name__ == "__main__":
    main()
