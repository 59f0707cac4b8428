"""Cross-play (ia2c_evaluate_lineups): the R x R matrix of a sweep's runs at T = 30, against the route the library offered
before it (gather every lineup's actors into pseudo-runs, evaluate_actors in chunks of at most IA2C_MAX_RUN_NETS nets, reduce
the returns on the host).

Per point (N, R, E, K), P = R * R lineups (cell (a, b): agents 0 .. N/2-1 of run a, the rest of run b):
  * lineup_ms / lineup_flushed_ms: device time of one ia2c_evaluate_lineups call on preallocated outputs, from CUDA events
    around many warm calls back to back, and around each call with a 256 MiB buffer written before it (the L2 flushed);
  * cross_play_ms: host clock of IA2CRuns.cross_play (lineups built and uploaded, the call, statistics copied back) to a
    synchronise;
  * pseudo_run_ms: host clock of the pseudo-run route on the same runs, to its host mean and std;
  * returns_match: whether the pseudo-run route's returns equal the lineup call's byte for byte;
  * env_steps_per_s = P * K * E * T / lineup_ms.
Prints one JSON line with the card's name, power limit and max SM clock (read-only nvidia-smi query) taken in the same call.

    python tools/bench_cross_play.py [--calls K] [--warmup W]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

T = 30
# (N, R, E, K): two small-agent sweeps (128 and 256 runs), a 16-agent and a 64-agent sweep
POINTS = ((2, 128, 10, 16), (2, 256, 10, 16), (16, 64, 10, 4), (64, 16, 64, 4))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50, help="timed device calls per leg (>= 10)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-reps", type=int, default=3, help="timed host-clock repetitions of each route (best is kept)")
    a = ap.parse_args()
    if a.calls < 10:
        ap.error("--calls must be at least 10")

    import numpy as np
    import torch

    from bench_eval import card
    from ia2c_b200 import _lib
    from ia2c_b200.evaluate import evaluate_actors, lineup_desc
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany

    _lib.require_cuda()
    torch.cuda.set_device(0)
    lib = _lib.load()
    gpu = card()
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    stream = torch.cuda.current_stream().cuda_stream

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def host_ms(fn):
        best = float("inf")
        for _ in range(a.host_reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            best = min(best, (time.perf_counter() - t0) * 1e3)
        return best

    rows = []
    for N, R, E, K in POINTS:
        seeds = list(range(1, R + 1))
        init = [(np.random.RandomState(s).normal(0, 0.6, (N, _lib.ACTOR_P)), np.zeros((N, _lib.CRITIC_P)),
                 np.full((N, 5, 3), 1.0 / 3)) for s in seeds]
        runs = (IA2CRuns if N <= 8 else IA2CRunsMany)(E, seeds, n_agents=N, init=init)
        P, nets, mes = R * R, R * N, runs.desc.max_episode_steps
        xp = runs.cross_play(episodes=K)                       # warm, and the lineups
        lin_np = xp["lineups"]
        lin = torch.from_numpy(lin_np).cuda()
        policy = torch.empty((nets, 9, 3), dtype=torch.float32, device="cuda")
        returns = torch.empty((P, K, E), dtype=torch.float64, device="cuda")
        counts = torch.empty((P * N, 3), dtype=torch.int64, device="cuda")
        stats = torch.empty((2, P), dtype=torch.float64, device="cuda")
        d = lineup_desc(runs.actor_params, nets, N, lin, E, K, T, mes, False, 0, 0, policy, returns, counts, stats[0], stats[1])

        def call():
            _lib.check(lib.ia2c_evaluate_lineups(C.byref(d), stream), "ia2c_evaluate_lineups")

        for _ in range(a.warmup):
            call()
        s0, s1 = ev(), ev()
        s0.record()
        for _ in range(a.calls):
            call()
        s1.record()
        torch.cuda.synchronize()
        lineup_ms = s0.elapsed_time(s1) / a.calls
        flushed = []
        for _ in range(a.calls):
            flush_buf.fill_(1)
            e0, e1 = ev(), ev()
            e0.record()
            call()
            e1.record()
            torch.cuda.synchronize()
            flushed.append(e0.elapsed_time(e1))
        lineup_returns = returns.cpu().numpy()

        chunk = _lib.MAX_RUN_NETS // N                          # pseudo-runs per evaluate_actors call
        idx = torch.from_numpy(lin_np.reshape(-1).astype(np.int64)).cuda()

        def pseudo():
            rets = []
            for c0 in range(0, P, chunk):
                c1 = min(P, c0 + chunk)
                actors = runs.actor_params[idx[c0 * N:c1 * N]].contiguous()
                rets.append(evaluate_actors(actors, c1 - c0, N, E, K, T, mes, False, 0, 0, runs.device)["returns"])
            r = np.concatenate(rets)
            return r, r.reshape(P, -1).mean(1), r.reshape(P, -1).std(1)

        pseudo_returns = pseudo()[0]
        pseudo_ms = host_ms(pseudo)
        cross_ms = host_ms(lambda: runs.cross_play(episodes=K))
        match = bool(pseudo_returns.shape == lineup_returns.shape
                     and np.array_equal(pseudo_returns.view(np.uint8), lineup_returns.view(np.uint8)))
        steps = P * K * E * T
        rows.append(dict(N=N, R=R, E=E, K=K, T=T, lineups=P, pseudo_run_calls=-(-P // chunk),
                         lineup_ms=round(lineup_ms, 4), lineup_flushed_ms=round(float(np.median(flushed)), 4),
                         cross_play_ms=round(cross_ms, 3), pseudo_run_ms=round(pseudo_ms, 3), returns_match=match,
                         env_steps_per_call=steps, env_steps_per_s=float(f"{steps / (lineup_ms * 1e-3):.4g}"),
                         returns_bytes=P * K * E * 8))
        del runs, policy, returns, counts, stats
        torch.cuda.empty_cache()
    print(json.dumps(dict(bench="cross_play", gpu=gpu, calls=a.calls, rows=rows)))


if __name__ == "__main__":
    main()
