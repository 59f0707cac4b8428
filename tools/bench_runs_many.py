"""Batched independent Org-N runs (IA2CRunsMany, 9 <= N <= 256) against the same runs as standalone IA2CTrainers trained one
after the other.

For every (N, E, R) of the grid: ms per batched episode (all R runs advance one episode: six launches) and ms for the R
standalone `IA2CTrainer(actor_kernel="columns")` episodes run back to back — the trainer the batch is byte-identical to — and,
at N = 256, also for R standalone episodes with the trainer's default actor kernel there (the pipelined one, labelled "pipe").
All from CUDA events around warm episodes, once back to back and once with the L2 flushed (a 256 MiB buffer written) before
every episode — for the sequential legs before every standalone episode.  Points with R * N above 65535 nets or with belief
records (R * E * N * (N - 1) * 8 B) above 8 GB are skipped.  Prints one JSON line with the card's name, power limit and max SM
clock (read-only nvidia-smi query).  Every figure is Org-N (DESIGN.md §8): the reference has two agents.

    python tools/bench_runs_many.py [--episodes K] [--warmup W] [--quick]
"""
import argparse
import gc
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_runs import card   # noqa: E402

GRID_N = (16, 64, 256)
GRID_E = (10, 64, 1024)
GRID_R = (1, 8, 64)
MAX_RECORD_BYTES = 8e9
M = 5


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--episodes", type=int, default=10, help="timed episodes per leg")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--quick", action="store_true", help="N = 16, E = 10, R <= 8 only (a rehearsal)")
    a = ap.parse_args()

    import torch

    from ia2c_b200 import _lib
    from ia2c_b200.runs import IA2CRunsMany
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

    grid = [(N, E, R) for N in GRID_N for E in GRID_E for R in GRID_R]
    if a.quick:
        grid = [(N, E, R) for N, E, R in grid if N == 16 and E == 10 and R <= 8]
    rows, skipped = [], []
    for N, E, R in grid:
        if R * N > _lib.MAX_RUN_NETS or R * E * N * (N - 1) * 8 > MAX_RECORD_BYTES:
            skipped.append(dict(N=N, E=E, R=R))
            continue
        seeds = list(range(1000, 1000 + R))
        batch = IA2CRunsMany(E, seeds, n_agents=N, n_models=M)
        b_ms, b_fl = back_to_back([batch.train_episode]), flushed([batch.train_episode])
        del batch
        gc.collect()
        torch.cuda.empty_cache()
        legs = [("columns", "columns")] + ([("pipe", "auto")] if N == 256 else [])
        seq = {}
        for label, kernel in legs:
            alone = [IA2CTrainer(E, n_agents=N, n_models=M, seed=s, init=reference_init(N, M, seed=s), actor_kernel=kernel)
                     for s in seeds]
            fns = [tr.train_episode for tr in alone]
            seq[label] = (back_to_back(fns), flushed(fns))
            del alone, fns
            gc.collect()
            torch.cuda.empty_cache()
        s_ms, s_fl = seq["columns"]
        steps = R * E * N * 30
        row = dict(env="Org-N", N=N, E=E, R=R, batched_ms=round(b_ms, 4), batched_ms_flushed=round(b_fl, 4),
                   sequential_columns_ms=round(s_ms, 4), sequential_columns_ms_flushed=round(s_fl, 4),
                   speedup=round(s_ms / b_ms, 2), speedup_flushed=round(s_fl / b_fl, 2),
                   run_episodes_per_s=round(R / (b_ms * 1e-3), 1), agent_steps_per_s=round(steps / (b_ms * 1e-3), 1))
        if "pipe" in seq:
            row.update(sequential_pipe_ms=round(seq["pipe"][0], 4), sequential_pipe_ms_flushed=round(seq["pipe"][1], 4),
                       speedup_vs_pipe=round(seq["pipe"][0] / b_ms, 2))
        rows.append(row)
        print(f"Org-N N={N:3d} E={E:5d} R={R:3d}: batched {b_ms * 1e3:10.1f} us ({b_fl * 1e3:10.1f} flushed), "
              f"sequential columns {s_ms * 1e3:11.1f} us ({s_fl * 1e3:11.1f} flushed), speed-up {s_ms / b_ms:6.2f}x"
              + (f", sequential pipe {seq['pipe'][0] * 1e3:11.1f} us" if "pipe" in seq else ""), file=sys.stderr)
    print(json.dumps(dict(tool="bench_runs_many", env="Org-N", gpu=card(), episodes=K, warmup=W, T=30, M=M,
                          l2="back to back, and with a 256 MiB buffer written before every (batched or standalone) episode",
                          rows=rows, skipped=skipped)))


if __name__ == "__main__":
    main()
