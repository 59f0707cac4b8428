"""What freezing the partner seats saves: K recorded episodes of per-env partner training with every seat trained and with
freeze_seats(pool.seats), at the points of tools/bench_env_partners.py plus the largest agent count.

Points — `IA2CTrainer` N = 2, E = 4096 (the headline shape); `IA2CRuns` N = 2, E = 10, R = 128; `IA2CRunsMany` N = 16, E = 10,
R = 64; `IA2CTrainer` N = 64, E = 1024; `IA2CTrainer` N = 256, E = 1024 (all with actor_kernel="columns", which frozen seats
need) — each with a pool of Q = 64 teams over the seats N/2 .. N-1 in per-env mode and two arms, µs per episode of
train_episodes(K) (with its history record):
  trained   every seat trained (set_partners(pool, per_env=True));
  frozen    the same with freeze_seats(pool.seats): the update kernels run the trained half of the rows.
Each arm is timed back to back (K episodes after W warm-up episodes, host clock, one synchronisation at the end) and with the
L2 flushed (a 256 MiB buffer written and the device synchronised before every episode, host clock around each episode and its
synchronisation).  The arms run in two rounds, alternating, on the same object; both rounds are printed.  A separate pass
reads per-kernel device times of a few episodes of each arm from torch.profiler.  Prints one JSON line with the card's name,
power limit and max SM clock (read-only nvidia-smi query, same call).

    python tools/bench_frozen_seats.py [--episodes K] [--warmup W] [--quick]
"""
import argparse
import gc
import json
import os
import re
import sys
import time
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_runs import card   # noqa: E402

POINTS = [("IA2CTrainer", 2, 4096, 1), ("IA2CRuns", 2, 10, 128), ("IA2CRunsMany", 16, 10, 64), ("IA2CTrainer", 64, 1024, 1),
          ("IA2CTrainer", 256, 1024, 1)]
Q = 64


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--episodes", type=int, default=128, help="timed episodes per arm")
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--profile-episodes", type=int, default=8)
    ap.add_argument("--quick", action="store_true", help="every point, few episodes (a rehearsal)")
    a = ap.parse_args()

    import numpy as np
    import torch

    from ia2c_b200 import _lib
    from ia2c_b200.partners import PartnerPool
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    from ia2c_b200.trainer import IA2CTrainer

    _lib.require_cuda()
    torch.cuda.set_device(0)
    gpu = card()
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    K, W, KP = (4, 2, 2) if a.quick else (a.episodes, a.warmup, a.profile_episodes)

    def sync():
        torch.cuda.synchronize()

    def make(kind, N, E, R):
        if kind == "IA2CTrainer":
            return IA2CTrainer(E, n_agents=N, n_models=5, seed=1, actor_kernel="columns")
        return (IA2CRuns if kind == "IA2CRuns" else IA2CRunsMany)(E, list(range(1000, 1000 + R)), n_agents=N, n_models=5)

    def arms(obj, pool):
        """arm -> (set its mode, outside the timed region; run k episodes; drain the logs)."""
        def run(k):
            obj.train_episodes(k)

        def tail():
            obj.history(), obj.env_partner_history()
        return {"trained": (lambda: obj.freeze_seats(None), run, tail), "frozen": (lambda: obj.freeze_seats(pool.seats), run, tail)}

    def back_to_back(run, tail):
        run(W)
        tail()
        sync()
        t0 = time.perf_counter()
        run(K)
        tail()
        sync()
        return (time.perf_counter() - t0) / K * 1e6

    def flushed(run, tail):
        total = 0.0
        for _ in range(K):
            flush_buf.zero_()
            sync()
            t0 = time.perf_counter()
            run(1)
            sync()
            total += time.perf_counter() - t0
        t0 = time.perf_counter()
        tail()
        total += time.perf_counter() - t0
        return total / K * 1e6

    def kernel_times(run, tail):
        """Device µs per episode of each kernel name, from torch.profiler over KP episodes."""
        from torch.profiler import ProfilerActivity, profile
        run(2)
        tail()
        sync()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(KP)
            sync()
        tail()
        per = defaultdict(float)
        for ev in prof.key_averages():
            m = re.search(r"(\w+_kernel)", ev.key)
            t = getattr(ev, "device_time_total", None)
            if m and t:
                per[m.group(1)] += t
        return {k: round(v / KP, 2) for k, v in sorted(per.items(), key=lambda x: -x[1])}

    results = []
    for kind, N, E, R in POINTS:
        obj = make(kind, N, E, R)
        rng = np.random.RandomState(N)
        split = N // 2
        P = Q * (N - split)
        rows = (rng.normal(size=(P, _lib.ACTOR_P)) * 0.5).astype(np.float32)
        teams = np.arange(P, dtype=np.int32).reshape(Q, N - split)
        pool = PartnerPool(rows, teams, np.arange(split, N, dtype=np.int32), N, device=obj.device)
        obj.set_partners(pool, per_env=True)
        row = dict(cls=kind, N=N, E=E, R=R, Q=Q, S=N - split, episodes=K, rounds=[])
        for rnd in range(2):
            legs = list(arms(obj, pool).items())
            if rnd:
                legs.reverse()          # the arms alternate: what ran first in round 0 runs last in round 1
            t = {}
            for leg, (mode, run, tail) in legs:
                mode()
                t[leg] = (round(back_to_back(run, tail), 1), round(flushed(run, tail), 1))
            t["frozen_minus_trained"] = tuple(round(t["frozen"][i] - t["trained"][i], 1) for i in range(2))
            row["rounds"].append(t)
            print(json.dumps(dict(point=(kind, N, E, R), **t)), file=sys.stderr, flush=True)
        row["kernels_us"] = {}
        for leg, (mode, run, tail) in arms(obj, pool).items():
            mode()
            row["kernels_us"][leg] = kernel_times(run, tail)
        print(json.dumps(dict(point=(kind, N, E, R), kernels_us=row["kernels_us"])), file=sys.stderr, flush=True)
        obj.freeze_seats(None), obj.set_partners(None)
        results.append(row)
        del obj, pool
        gc.collect()
        torch.cuda.empty_cache()
    print(json.dumps(dict(bench="frozen_seats", gpu=gpu, points=results)))


if __name__ == "__main__":
    main()
