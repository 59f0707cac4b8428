"""What a population-based-training generation costs: G intervals of I recorded episodes trained three ways, and the two PBT
kernels alone.

For every point (N, E, R) — (2, 10, 128) `IA2CRuns`, (16, 10, 64) and (256, 64, 8) `IA2CRunsMany` — three legs, each a
host clock around G intervals that ends in a device synchronisation:
  (a) train_episodes(I)                                   per interval, no PBT;
  (b) train_episodes(I) + exploit_explore(window=I)       the generation on the device;
  (c) train_episodes(I) + the host PBT a user writes without exploit_explore: history() (synchronises), a numpy rank of
      the window's return sums, torch index_copy_ of the ten per-net buffers from donors to recipients, and the
      hyper-parameter tensors rewritten from numpy.
Reported per generation: each leg, (b) - (a) and (c) - (a), and the batched episode of (a) for scale.  The two kernels alone
(ia2c_pbt_step with the batch's own descriptors) are timed with CUDA events, back to back and with a 256 MiB buffer written
before each call.  Prints one JSON line with the card's name, power limit and max SM clock (read-only nvidia-smi query, same
call).

    python tools/bench_pbt.py [--generations G] [--interval I] [--quick]
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
from oracle.pbt import COPIED   # noqa: E402  the ten per-net buffers a recipient copies

POINTS = [("IA2CRuns", 2, 10, 128), ("IA2CRunsMany", 16, 10, 64), ("IA2CRunsMany", 256, 64, 8)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--generations", type=int, default=32, help="timed generations (intervals) per leg")
    ap.add_argument("--interval", type=int, default=8, help="recorded episodes per generation (= the fitness window)")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--kernel-calls", type=int, default=200)
    ap.add_argument("--quick", action="store_true", help="the first point, few generations (a rehearsal)")
    a = ap.parse_args()

    import numpy as np
    import torch

    from ia2c_b200 import _lib
    from ia2c_b200.runs import IA2CRuns, IA2CRunsMany

    _lib.require_cuda()
    torch.cuda.set_device(0)
    gpu = card()
    lib = _lib.load()
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    G, I, W = (4, a.interval, 1) if a.quick else (a.generations, a.interval, a.warmup)
    points = POINTS[:1] if a.quick else POINTS

    def make(cls, N, E, R):
        c = IA2CRuns if cls == "IA2CRuns" else IA2CRunsMany
        return c(E, list(range(1, R + 1)), n_agents=N, lr_actor=list(np.geomspace(1e-5, 1e-3, R)))

    def host_pbt(obj, rng, factors=(0.8, 1.2)):
        R, N, q = obj.R, obj.N, obj.R // 4
        obj._materialise_hyper()   # per-run hyper-parameter arrays, as exploit_explore makes them
        fit =obj.history()["return_sum"][-I:].sum(axis=0)
        order = np.lexsort((np.arange(R), -fit))
        rec, don = order[R - q:], order[rng.integers(0, q, size=q)]
        rows = lambda runs: torch.from_numpy((runs[:, None] * N + np.arange(N)).ravel()).to(obj.device)   # noqa: E731
        r_rows, d_rows = rows(rec), rows(don)
        for k in COPIED:
            t = getattr(obj, k)
            t.index_copy_(0, r_rows, t.index_select(0, d_rows))
        for k in ("lr_actor", "lr_critic", "beta", "gamma"):
            v = obj._hyper[k].cpu().numpy()
            v[rec] = v[don]
            if k != "gamma":
                v[rec] = (v[rec] * np.where(rng.random(q) < 0.5, factors[0], factors[1])).astype(v.dtype)
            obj._hyper[k].copy_(torch.from_numpy(v))

    def leg(obj, kind):
        rng = np.random.default_rng(0)

        def interval():
            obj.train_episodes(I)
            if kind == "b":
                obj.exploit_explore(I)
            elif kind == "c":
                host_pbt(obj, rng)

        for _ in range(W):
            interval()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(G):
            interval()
        obj.history()   # drain what (a) and (b) left in the ring: (c) drained every interval
        obj.pbt_history()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / G * 1e6

    def kernels_alone(obj):
        obj.train_episodes(I)
        obj.exploit_explore(I)   # materialises the hyper-parameter arrays, the log and the workspace
        ring, log = obj._history, obj._pbt_log
        p = _lib.PbtDesc()
        p.window, p.slot, p.q, p.perturb = I, (ring.head - 1) % ring.capacity, obj.R // 4, 7
        p.factor_lo, p.factor_hi, p.seed = 0.8, 1.2, 0
        for k in ("lr_actor", "lr_critic", "gamma", "beta"):
            setattr(p, k, obj._hyper[k].data_ptr())
        for k in ("fitness", "rank", "donor", "lr_actor", "lr_critic", "gamma", "beta"):
            setattr(p, "log_" + k, log.ptr[k])
        p.workspace, p.workspace_bytes = obj._pbt_ws.data_ptr(), obj._pbt_ws.numel()
        args = (C.byref(obj.desc), C.byref(obj.runs_desc), ring._href, C.byref(p), torch.cuda.current_stream().cuda_stream)

        def call(g):
            p.generation = g
            _lib.check(lib.ia2c_pbt_step(*args), "ia2c_pbt_step")

        for g in range(10):
            call(g)
        torch.cuda.synchronize()
        K = a.kernel_calls
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for g in range(K):
            call(g)
        e.record()
        torch.cuda.synchronize()
        b2b = s.elapsed_time(e) / K * 1e3
        marks = []
        for g in range(K):
            flush_buf.zero_()
            m = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            m[0].record()
            call(g)
            m[1].record()
            marks.append(m)
        torch.cuda.synchronize()
        flushed = float(np.median([x.elapsed_time(y) for x, y in marks]) * 1e3)
        return b2b, flushed

    results = []
    for cls, N, E, R in points:
        row = dict(cls=cls, N=N, E=E, R=R, q=R // 4, interval=I, generations=G)
        for kind in ("a", "b", "c"):
            obj = make(cls, N, E, R)
            row[kind + "_us"] = round(leg(obj, kind), 1)
            del obj
            gc.collect()
            torch.cuda.empty_cache()
        row["episode_us"] = round(row["a_us"] / I, 1)
        row["b_minus_a_us"] = round(row["b_us"] - row["a_us"], 1)
        row["c_minus_a_us"] = round(row["c_us"] - row["a_us"], 1)
        obj = make(cls, N, E, R)
        b2b, flushed = kernels_alone(obj)
        row["kernels_b2b_us"], row["kernels_flushed_us"] = round(b2b, 2), round(flushed, 2)
        del obj
        gc.collect()
        torch.cuda.empty_cache()
        results.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    print(json.dumps(dict(bench="pbt", gpu=gpu, points=results)))


if __name__ == "__main__":
    main()
