"""What recording a learning curve costs: K episodes trained three ways, and the record kernel alone.

For every point (N, E, R) — (2, 4096, 1) and (256, 1024, 1) standalone `IA2CTrainer`, (2, 10, 8) and (2, 10, 128) `IA2CRuns`,
(16, 10, 64) `IA2CRunsMany` — three legs, each timed with a host clock around work that ends in a device synchronisation:
  (a) K x train_episode()                      nothing is kept;
  (b) train_episodes(K) + history()            every episode recorded on the device, drained when the ring is full;
  (c) K x train_episode(sync_stats=True)       every episode read back on the host (read_stats).
Each leg is timed back to back (K episodes, one synchronisation at the end) and with the L2 flushed (a 256 MiB buffer written
and the device synchronised before every episode; the episode is timed to its own synchronisation, and (b)'s history() is
timed once and spread over the K episodes).  The record kernel alone (ia2c_record_episode on the point's buffers into a
two-slot ring) is timed with CUDA events, back to back and flushed.  Prints one JSON line with the card's name, power limit
and max SM clock (read-only nvidia-smi query, same call).

    python tools/bench_history.py [--episodes K] [--warmup W] [--quick]
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

POINTS = [("IA2CTrainer", 2, 4096, 1), ("IA2CRuns", 2, 10, 8), ("IA2CRuns", 2, 10, 128), ("IA2CRunsMany", 16, 10, 64),
          ("IA2CTrainer", 256, 1024, 1)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--episodes", type=int, default=128, help="timed episodes per leg (the ring holds 64: (b) drains in the loop)")
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--quick", action="store_true", help="the two smallest points only (a rehearsal)")
    a = ap.parse_args()

    import torch

    from ia2c_b200 import _lib
    from ia2c_b200.history import EpisodeHistory
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany
    from ia2c_b200.trainer import IA2CTrainer

    _lib.require_cuda()
    torch.cuda.set_device(0)
    gpu = card()
    lib = _lib.load()
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    K, W = a.episodes, a.warmup

    def sync():
        torch.cuda.synchronize()

    def legs(obj):
        return dict(a=(lambda k: [obj.train_episode() for _ in range(k)], None),
                    b=(lambda k: obj.train_episodes(k), obj.history),
                    c=(lambda k: [obj.train_episode(sync_stats=True) for _ in range(k)], None))

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

    def record_alone(obj, runs):
        ring = EpisodeHistory(lib, obj.device, runs, obj.N, obj.E, obj.T, 2)
        dref, stream = C.byref(obj.desc), torch.cuda.current_stream().cuda_stream

        def one(k):
            _lib.check(lib.ia2c_record_episode(dref, runs, ring._href, k & 1, stream), "ia2c_record_episode")

        for k in range(W):
            one(k)
        sync()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for k in range(K):
            one(k)
        e.record()
        sync()
        b2b = s.elapsed_time(e) / K * 1e3
        marks = []
        for k in range(K):
            flush_buf.zero_()
            m = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            m[0].record()
            one(k)
            m[1].record()
            marks.append(m)
        sync()
        return b2b, sum(x.elapsed_time(y) for x, y in marks) / K * 1e3

    points = POINTS[:2] if a.quick else POINTS
    rows = []
    for kind, N, E, R in points:
        if kind == "IA2CTrainer":
            obj = IA2CTrainer(E, n_agents=N, n_models=5, seed=1)
        else:
            obj = (IA2CRuns if kind == "IA2CRuns" else IA2CRunsMany)(E, list(range(1000, 1000 + R)), n_agents=N, n_models=5)
        t = {leg: (back_to_back(run, tail), flushed(run, tail)) for leg, (run, tail) in legs(obj).items()}
        rec_b2b, rec_fl = record_alone(obj, 1 if kind == "IA2CTrainer" else R)
        row = dict(kind=kind, N=N, E=E, R=R,
                   a_us=round(t["a"][0], 2), b_us=round(t["b"][0], 2), c_us=round(t["c"][0], 2),
                   a_us_flushed=round(t["a"][1], 2), b_us_flushed=round(t["b"][1], 2), c_us_flushed=round(t["c"][1], 2),
                   b_minus_a_us=round(t["b"][0] - t["a"][0], 2), b_over_a_pct=round(100 * (t["b"][0] / t["a"][0] - 1), 2),
                   c_over_b=round(t["c"][0] / t["b"][0], 2),
                   record_kernel_us=round(rec_b2b, 2), record_kernel_us_flushed=round(rec_fl, 2))
        rows.append(row)
        print(f"{kind:12s} N={N:3d} E={E:5d} R={R:3d}: (a) {row['a_us']:9.1f} us  (b) {row['b_us']:9.1f} us  (c) {row['c_us']:9.1f} us "
              f"per episode back to back; flushed {row['a_us_flushed']:9.1f} / {row['b_us_flushed']:9.1f} / {row['c_us_flushed']:9.1f}; "
              f"record kernel {rec_b2b:6.2f} us ({rec_fl:6.2f} flushed)", file=sys.stderr)
        del obj
        gc.collect()
        torch.cuda.empty_cache()
    print(json.dumps(dict(tool="bench_history", gpu=gpu, episodes=K, warmup=W, T=30, M=5,
                          timing="host clock to a device synchronisation; record kernel with CUDA events",
                          l2="back to back, and with a 256 MiB buffer written before every episode", rows=rows)))


if __name__ == "__main__":
    main()
