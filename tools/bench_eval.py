"""Frozen-policy evaluation (ia2c_evaluate): time per call over a set of (N, R, E, K) shapes at T = 30, and for the R = 1
shapes the only alternative the library had before it, IA2CTrainer.rollout() holding the same parameters.

Every figure is device time from CUDA events around many warm calls of the C entry point on preallocated outputs (no host
copies): once back to back, and once with a 256 MiB buffer written before every call (the L2 flushed), as
tools/bench_runs.py does.  env-steps/s = R * E * K * T per call time.  Prints one JSON line with the card's name, power
limit and max SM clock (read-only nvidia-smi query) taken in the same call.

    python tools/bench_eval.py [--calls K] [--warmup W]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

T = 30
# (N, R, E, K): the headline shape; a sweep of 128 small runs; a medium batch; two many-agent shapes (one warp per item)
ROWS = ((2, 1, 4096, 1), (2, 128, 10, 16), (8, 64, 64, 4), (64, 1, 1024, 1), (256, 1, 1024, 1))


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
    ap.add_argument("--calls", type=int, default=200, help="timed calls per leg (>= 50)")
    ap.add_argument("--warmup", type=int, default=10)
    a = ap.parse_args()
    if a.calls < 50:
        ap.error("--calls must be at least 50")

    import numpy as np
    import torch

    from ia2c_b200 import _lib
    from ia2c_b200.evaluate import eval_desc, evaluate_actors
    from ia2c_b200.trainer import IA2CTrainer, reference_init

    _lib.require_cuda()
    torch.cuda.set_device(0)
    lib = _lib.load()
    gpu = card()
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    K_CALLS, W = a.calls, a.warmup

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def back_to_back(f):
        for _ in range(W):
            f()
        torch.cuda.synchronize()
        s, e = ev(), ev()
        s.record()
        for _ in range(K_CALLS):
            f()
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) * 1e3 / K_CALLS

    def flushed(f):
        marks = []
        for _ in range(K_CALLS):
            flush_buf.zero_()
            m = (ev(), ev())
            m[0].record()
            f()
            m[1].record()
            marks.append(m)
        torch.cuda.synchronize()
        return sum(s.elapsed_time(e) for s, e in marks) * 1e3 / K_CALLS

    rows = []
    for N, R, E, K in ROWS:
        init = [reference_init(N, 5, seed=r) for r in range(R)]
        params = torch.from_numpy(np.concatenate([i[0] for i in init]).astype(np.float32)).cuda()
        policy = torch.empty(R * N, 9, 3, device="cuda")
        returns = torch.empty(R, K, E, dtype=torch.float64, device="cuda")
        counts = torch.empty(R * N, 3, dtype=torch.int64, device="cuda")
        d = eval_desc(params, R, N, E, K, T, 30, False, 0, 0, policy, returns, counts)
        stream = torch.cuda.current_stream().cuda_stream

        def call():
            _lib.check(lib.ia2c_evaluate(C.byref(d), stream), "ia2c_evaluate")

        us, us_fl = back_to_back(call), flushed(call)
        # the library's result equals the Python entry point's (same descriptor, same outputs)
        ref = evaluate_actors(params, R, N, E, K, T, 30, False, 0, 0, "cuda")
        assert np.array_equal(returns.cpu().numpy(), ref["returns"])
        steps = R * E * K * T
        row = dict(N=N, R=R, E=E, K=K, eval_us=round(us, 2), eval_us_flushed=round(us_fl, 2),
                   env_steps_per_s=round(steps / (us * 1e-6), 1), env_steps_per_s_flushed=round(steps / (us_fl * 1e-6), 1))
        msg = f"N={N:4d} R={R:4d} E={E:5d} K={K:3d}: eval {us:8.1f} us ({us_fl:8.1f} flushed)"
        if R == 1:
            tr = IA2CTrainer(E, n_agents=N, n_models=5, steps_per_episode=T, init=init[0])
            r_us, r_fl = back_to_back(tr.rollout), flushed(tr.rollout)
            row.update(rollout_us=round(r_us, 2), rollout_us_flushed=round(r_fl, 2), rollout_over_eval=round(r_us / us, 2))
            msg += f", rollout() {r_us:8.1f} us ({r_fl:8.1f} flushed): {r_us / us:.1f}x"
            del tr
        print(msg, file=sys.stderr)
        rows.append(row)
    print(json.dumps(dict(tool="bench_eval", gpu=gpu, T=T, max_episode_steps=30, calls=K_CALLS, warmup=W,
                          timing="CUDA events; eval_us / rollout_us back to back, *_flushed with a 256 MiB buffer written "
                                 "before every call",
                          rows=rows)))


if __name__ == "__main__":
    main()
