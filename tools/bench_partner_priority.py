"""What prioritized partner draws cost: recorded episodes of the uniform per-env mode against the prioritized one, the rollout
kernel's device time in both (the weighted draw is a binary search of ceil(log2 Q) dependent L2 loads in every env's
prologue), the record kernel's device time, and one prioritize_partners call.

Points — `IA2CTrainer` N = 2, E = 4096 (the headline shape); `IA2CRuns` N = 2, E = 10, R = 128; `IA2CRunsMany` N = 16, E = 10,
R = 64 — each with a pool of Q = 16, 256 and 4096 teams over the seats N/2 .. N-1 and two arms:
  uniform      set_partners(pool, per_env=True);
  prioritized  set_partners(pool, per_env=True, prioritized=True) after one prioritize_partners over recorded episodes, so
               the tables hold unequal weights: the same launches plus the record of the returns.
Per arm: µs per episode of train_episodes(K) back to back (host clock, one synchronisation at the end, the logs drained
inside the window), in two rounds with the arms alternating; then, in a separate profiled pass of 8 episodes per arm
(torch.profiler, CUDA activity), the mean device time of the rollout kernel and of partner_returns_kernel.  Finally
ia2c_prioritize_partners at R = 256, Q = 256 with random statistics: CUDA events around 200 calls.  Prints one JSON line with
the card's name, power limit and max SM clock (read-only nvidia-smi query, same call).

    python tools/bench_partner_priority.py [--episodes K] [--quick]
"""
import argparse
import ctypes as C
import gc
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_runs import card   # noqa: E402

POINTS = [("IA2CTrainer", 2, 4096, 1), ("IA2CRuns", 2, 10, 128), ("IA2CRunsMany", 16, 10, 64)]
QS = [16, 256, 4096]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--episodes", type=int, default=128, help="timed episodes per arm")
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--quick", action="store_true", help="every point, few episodes (a rehearsal)")
    a = ap.parse_args()

    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile

    from ia2c_b200 import _lib
    from ia2c_b200.partners import PartnerPool
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    from ia2c_b200.trainer import IA2CTrainer

    _lib.require_cuda()
    torch.cuda.set_device(0)
    gpu = card()
    K, W = (4, 2) if a.quick else (a.episodes, a.warmup)

    def make(kind, N, E, R):
        if kind == "IA2CTrainer":
            return IA2CTrainer(E, n_agents=N, n_models=5, seed=1)
        return (IA2CRuns if kind == "IA2CRuns" else IA2CRunsMany)(E, list(range(1000, 1000 + R)), n_agents=N, n_models=5)

    def drain(obj):
        obj.history(), obj.env_partner_history()

    def back_to_back(obj):
        obj.train_episodes(W)
        drain(obj)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        obj.train_episodes(K)
        drain(obj)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / K * 1e6

    def kernel_us(obj, episodes=8):
        """Mean device µs per launch of the rollout kernel and of partner_returns_kernel over `episodes` episodes."""
        obj.train_episodes(2)
        drain(obj)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            obj.train_episodes(episodes)
            torch.cuda.synchronize()
        drain(obj)
        out = {}
        for ev in prof.key_averages():
            for name in ("rollout_fused_kernel", "rollout_many_kernel", "partner_returns_kernel"):
                if name in ev.key:
                    key = "rollout" if name.startswith("rollout") else "record"
                    t = getattr(ev, "device_time_total", None)
                    if t is None:
                        t = ev.cuda_time_total
                    out[key] = round(out.get(key, 0.0) + t / episodes, 2)
        return out

    results = []
    for kind, N, E, R in POINTS:
        for Q in ([4, 16] if a.quick else QS):
            obj = make(kind, N, E, R)
            rng = np.random.RandomState(Q)
            split = N // 2
            S = N - split
            P = min(Q * S, 4096)
            rows = (rng.normal(size=(P, _lib.ACTOR_P)) * 0.5).astype(np.float32)
            teams = rng.randint(0, P, size=(Q, S)).astype(np.int32)
            pool = PartnerPool(rows, teams, np.arange(split, N, dtype=np.int32), N, device=obj.device)

            def arm(prioritized):
                obj.set_partners(pool, per_env=True, prioritized=prioritized)
                if prioritized:   # unequal weights: statistics of a few episodes, then one prioritize
                    obj.train_episodes(4)
                    obj.prioritize_partners(power=2, floor=0.1, reset=False)
                drain(obj)

            row = dict(cls=kind, N=N, E=E, R=R, Q=Q, S=S, episodes=K, rounds=[])
            for rnd in range(2):
                order = [False, True] if rnd == 0 else [True, False]
                t = {}
                for prioritized in order:
                    arm(prioritized)
                    t["prioritized" if prioritized else "uniform"] = round(back_to_back(obj), 1)
                t["prioritized_minus_uniform"] = round(t["prioritized"] - t["uniform"], 1)
                row["rounds"].append(t)
            for prioritized in (False, True):
                arm(prioritized)
                row["kernels_" + ("prioritized" if prioritized else "uniform")] = kernel_us(obj)
            print(json.dumps(dict(point=(kind, N, E, R, Q), **{k: v for k, v in row.items() if k not in ("cls", "N", "E", "R", "Q")})),
                  file=sys.stderr, flush=True)
            obj.set_partners(None)
            results.append(row)
            del obj, pool
            gc.collect()
            torch.cuda.empty_cache()

    # one prioritize_partners call at R = 256, Q = 256, statistics as after a few episodes
    lib = _lib.load()
    Rp, Qp = 256, 256
    count = torch.from_numpy(np.random.RandomState(0).randint(0, 40, size=(Rp, Qp)).astype(np.int64)).cuda()
    total = torch.from_numpy(np.random.RandomState(1).randint(-(40 << 25), 40 << 25, size=(Rp, Qp)).astype(np.int64)).cuda()
    table = torch.zeros((Rp, Qp + 1), dtype=torch.int64, device="cuda")
    w = _lib.PartnerPriorityDesc()
    w.count, w.sum, w.table, w.R, w.Q = count.data_ptr(), total.data_ptr(), table.data_ptr(), Rp, Qp
    stream = torch.cuda.current_stream().cuda_stream
    calls = 20 if a.quick else 200
    for _ in range(10):
        _lib.check(lib.ia2c_prioritize_partners(C.byref(w), 2, 0.1, 0, stream), "ia2c_prioritize_partners")
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(calls):
        _lib.check(lib.ia2c_prioritize_partners(C.byref(w), 2, 0.1, 0, stream), "ia2c_prioritize_partners")
    end.record()
    torch.cuda.synchronize()
    prioritize_us = round(start.elapsed_time(end) * 1e3 / calls, 2)
    print(json.dumps(dict(bench="partner_priority", gpu=gpu, points=results,
                          prioritize=dict(R=Rp, Q=Qp, calls=calls, us_per_call=prioritize_us))))


if __name__ == "__main__":
    main()
