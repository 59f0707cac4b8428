"""What seating frozen partners costs: K episodes trained with and without a pool, the host loop a user writes without
set_partners, and the seat kernel alone.

For every point — `IA2CTrainer` N = 2, E = 4096; `IA2CRuns` N = 2, E = 10, R = 128; `IA2CRunsMany` N = 16, E = 10, R = 64 —
with a pool of Q = 64 teams over the seats N/2 .. N-1, four legs, each µs per episode:
  (a)  train_episodes(K), self-play;
  (b)  train_episodes(K) with set_partners(pool): one more launch per episode;
  (a') K x train_episode(), self-play, nothing recorded (the entry point of (c));
  (c)  K x [numpy draw of a team per run, torch index_copy_ of the drawn rows into the seat rows, train_episode()]: the loop a
       user writes without set_partners.
So (b) - (a) is what seating costs inside the recorded loop and (c) - (a') what the host loop costs on its own entry point.
Each leg is timed back to back (K episodes, host clock, one synchronisation at the end) and with the L2 flushed (a 256 MiB
buffer written and the device synchronised before every episode, host clock around each episode and its synchronisation).
The legs run twice, alternating, on the same objects; both rounds are printed.  The seat kernel alone (ia2c_seat_partners on
the point's descriptors) is timed with CUDA events, back to back and flushed.  Prints one JSON line with the card's name,
power limit and max SM clock (read-only nvidia-smi query, same call).

    python tools/bench_partners.py [--episodes K] [--quick]
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
Q = 64


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--episodes", type=int, default=128, help="timed episodes per leg")
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--kernel-calls", type=int, default=200)
    ap.add_argument("--quick", action="store_true", help="the first two points, few episodes (a rehearsal)")
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
    lib = _lib.load()
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    K, W = (8, 2) if a.quick else (a.episodes, a.warmup)
    points = POINTS[:2] if a.quick else POINTS

    def sync():
        torch.cuda.synchronize()

    def make(kind, N, E, R):
        if kind == "IA2CTrainer":
            return IA2CTrainer(E, n_agents=N, n_models=5, seed=1)
        return (IA2CRuns if kind == "IA2CRuns" else IA2CRunsMany)(E, list(range(1000, 1000 + R)), n_agents=N, n_models=5)

    def host_loop(obj, pool_rows, teams, seats, rng):
        """One episode of the loop a user writes without set_partners."""
        R, N = getattr(obj, "R", 1), obj.N
        draw = rng.integers(0, Q, size=R)
        dst = torch.from_numpy((np.arange(R)[:, None] * N + seats).ravel()).to(obj.device)
        src = torch.from_numpy(teams[draw].ravel()).to(obj.device)
        obj.actor_params.index_copy_(0, dst, pool_rows.index_select(0, src))
        obj.train_episode()

    def legs(obj, pool, host):
        rows_d, teams, seats = host
        rng = np.random.default_rng(0)

        def unseated(run):
            def go(k):
                obj.set_partners(None)
                run(k)
            return go

        def seated(k):
            obj.set_partners(pool)
            obj.train_episodes(k)

        return {"a": (unseated(obj.train_episodes), obj.history),
                "b": (seated, lambda: (obj.history(), obj.partner_history())),
                "a_plain": (unseated(lambda k: [obj.train_episode() for _ in range(k)]), None),
                "c": (unseated(lambda k: [host_loop(obj, rows_d, teams, seats, rng) for _ in range(k)]), None)}

    def back_to_back(run, tail):
        run(W)
        if tail:
            tail()
        sync()
        t0 = time.perf_counter()
        run(K)
        if tail:
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
        if tail:
            t0 = time.perf_counter()
            tail()
            total += time.perf_counter() - t0
        return total / K * 1e6

    def kernel_alone(obj, pool):
        R = getattr(obj, "R", 1)
        log = torch.empty(R, dtype=torch.int32, device=obj.device)
        p = _lib.PartnerDesc()
        p.rows, p.P, p.seats, p.S = pool.rows.data_ptr(), pool.P, pool.seats.data_ptr(), pool.S
        p.teams, p.Q, p.log_team = pool.teams.data_ptr(), pool.Q, log.data_ptr()
        runs = C.byref(obj.runs_desc) if isinstance(obj, IA2CRuns) else None
        args = (C.byref(obj.desc), runs, C.byref(p), torch.cuda.current_stream().cuda_stream)

        def one(k):
            p.episode = k
            _lib.check(lib.ia2c_seat_partners(*args), "ia2c_seat_partners")

        for k in range(10):
            one(k)
        sync()
        n = a.kernel_calls
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for k in range(n):
            one(k)
        e.record()
        sync()
        b2b = s.elapsed_time(e) / n * 1e3
        marks = []
        for k in range(n):
            flush_buf.zero_()
            m = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            m[0].record()
            one(k)
            m[1].record()
            marks.append(m)
        sync()
        return b2b, float(np.median([x.elapsed_time(y) for x, y in marks]) * 1e3)

    results = []
    for kind, N, E, R in points:
        obj = make(kind, N, E, R)
        rng = np.random.RandomState(N)
        split = N // 2
        P = Q * (N - split)
        rows = (rng.normal(size=(P, _lib.ACTOR_P)) * 0.5).astype(np.float32)
        teams = np.arange(P, dtype=np.int32).reshape(Q, N - split)
        seats = np.arange(split, N, dtype=np.int32)
        pool = PartnerPool(rows, teams, seats, N, device=obj.device)
        row = dict(cls=kind, N=N, E=E, R=R, Q=Q, S=N - split, episodes=K, rounds=[])
        for _ in range(2):
            t = {leg: (round(back_to_back(run, tail), 1), round(flushed(run, tail), 1))
                 for leg, (run, tail) in legs(obj, pool, (pool.rows, teams, seats)).items()}
            t["b_minus_a"] = (round(t["b"][0] - t["a"][0], 1), round(t["b"][1] - t["a"][1], 1))
            t["c_minus_a_plain"] = (round(t["c"][0] - t["a_plain"][0], 1), round(t["c"][1] - t["a_plain"][1], 1))
            row["rounds"].append(t)
            print(json.dumps(dict(point=(kind, N, E, R), **t)), file=sys.stderr, flush=True)
        obj.set_partners(None)
        b2b, fl = kernel_alone(obj, pool)
        row["kernel_us"], row["kernel_us_flushed"] = round(b2b, 2), round(fl, 2)
        results.append(row)
        del obj, pool
        gc.collect()
        torch.cuda.empty_cache()
    print(json.dumps(dict(bench="partners", gpu=gpu, points=results)))


if __name__ == "__main__":
    main()
