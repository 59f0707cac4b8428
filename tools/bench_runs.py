"""Batched independent runs (IA2CRuns) against the same runs as standalone IA2CTrainers trained one after the other.

For every (N, E, R) of the grid: ms per batched episode (all R runs advance one episode) and ms for the R standalone
episodes run back to back, both from CUDA events around many warm episodes, once back to back and once with the L2
flushed (a 256 MiB buffer written) before every episode — for the sequential leg before every standalone episode — as
bench.py does.  Prints one JSON line with the card's name and power limit (read-only nvidia-smi query).

    python tools/bench_runs.py [--episodes K] [--warmup W] [--quick]
"""
import argparse
import gc
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GRID_E = (10, 64, 1024)
GRID_R = (1, 8, 64, 128, 256)
N8_E = 10          # the one N = 8 row


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in out.split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as exc:   # the measurement stands without it, but says so
        return dict(name=f"unknown ({exc})")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--episodes", type=int, default=20, help="timed episodes per leg")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="E = 10 and R <= 8 only (a rehearsal)")
    a = ap.parse_args()

    import torch

    from ia2c_b200 import _lib
    from ia2c_b200.runs import IA2CRuns
    from ia2c_b200.trainer import IA2CTrainer, reference_init

    _lib.require_cuda()
    torch.cuda.set_device(0)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    K, W = a.episodes, a.warmup

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def back_to_back(fns):
        for _ in range(W):
            for f in fns:
                f()
        torch.cuda.synchronize()
        s, e = ev(), ev()
        s.record()
        for _ in range(K):
            for f in fns:
                f()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / K

    def flushed(fns):
        marks = []
        for _ in range(K):
            for f in fns:
                flush_buf.zero_()
                m = (ev(), ev())
                m[0].record()
                f()
                m[1].record()
                marks.append(m)
        torch.cuda.synchronize()
        return sum(s.elapsed_time(e) for s, e in marks) / K

    grid = [(2, E, R) for E in GRID_E for R in GRID_R] + [(8, N8_E, R) for R in GRID_R]
    if a.quick:
        grid = [(N, E, R) for N, E, R in grid if E == 10 and R <= 8]
    rows = []
    for N, E, R in grid:
        seeds = list(range(1000, 1000 + R))
        batch = IA2CRuns(E, seeds, n_agents=N)
        alone = [IA2CTrainer(E, n_agents=N, seed=s, init=reference_init(N, 5, seed=s)) for s in seeds]
        b_ms, b_fl = back_to_back([batch.train_episode]), flushed([batch.train_episode])
        fns = [tr.train_episode for tr in alone]
        s_ms, s_fl = back_to_back(fns), flushed(fns)
        steps = R * E * N * batch.T
        rows.append(dict(N=N, E=E, R=R, batched_ms=round(b_ms, 4), batched_ms_flushed=round(b_fl, 4),
                         sequential_ms=round(s_ms, 4), sequential_ms_flushed=round(s_fl, 4),
                         run_episodes_per_s=round(R / (b_ms * 1e-3), 1), agent_steps_per_s=round(steps / (b_ms * 1e-3), 1),
                         speedup=round(s_ms / b_ms, 2), speedup_flushed=round(s_fl / b_fl, 2)))
        print(f"N={N} E={E:5d} R={R:4d}: batched {b_ms * 1e3:9.1f} us ({b_fl * 1e3:9.1f} flushed), "
              f"sequential {s_ms * 1e3:10.1f} us ({s_fl * 1e3:10.1f} flushed), speed-up {s_ms / b_ms:6.2f}x", file=sys.stderr)
        del batch, alone, fns
        gc.collect()
        torch.cuda.empty_cache()
    print(json.dumps(dict(tool="bench_runs", gpu=card(), episodes=K, warmup=W, T=30, M=5,
                          l2="back to back, and with a 256 MiB buffer written before every (batched or standalone) episode",
                          rows=rows)))


if __name__ == "__main__":
    main()
