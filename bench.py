#!/usr/bin/env python
"""bench.py — IA2C rollout-and-update throughput on B200 (agent-steps/s including the A2C update).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA kernels through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the UNMODIFIED reference loop (oracle/_ref/ia2c.py)
                                                             # on the box's host cores
    python bench.py --gpus 1 --steps K --dump-outputs DIR    # + the last timed headline step's outputs as DIR/*.npy

A "step" is one IA2C episode: rollout of T=30 env steps for E envs x N agents (T+1 actor/belief evaluations)
followed by the critic phase and the actor phase (ia2c.py:62-129).  The headline (`value`, `e2e`) is BASELINE.json
configs[1] per GPU — Org domain, 2 agents, 4096 env instances per GPU (weak scaling: envs sharded across ranks, the
gradients of each optimiser phase exchanged by the fused NVLink all-reduce + Adam kernel).  The same JSON line
carries a `configs` array with the other BASELINE configs: cfg5 (256 agents x 8192 envs, STRONG scaling over the
ranks — the north-star configuration), and at N=1 also cfg4 (64 x 1024), cfg3 (ac_nets update at 65536 x 500) and
cfg1 (a2c_org_test.py's loop), each with its own ms_per_step, dominant-kernel roofline and CPU figure.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "agent-steps/sec incl. A2C update (Org domain)"
UNIT = "agent-steps/s"
DTYPE = "f32 nets / f64 env+belief"
T_STEPS, N_MODELS = 30, 5
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the ncu --set full captures summarised under profiles/
NCU_DRAM_BYTES = {"rollout_fused_kernel<2,5,1>@4096": 71168}
# fp32 FLOPs per agent-step (SURVEY.md §8 d4): rollout 210, critic phase 1512, actor phase 1044
FLOPS_ROLLOUT, FLOPS_CRITIC, FLOPS_ACTOR = 210, 1512, 1044


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000,
                    help="timed steps per block of the headline; configs[] clamp K to their own range (cfg5 2..5 per GPU, cfg4 2..30, "
                         "cfg3 3..30, cfg1 3..20) and report the steps they timed")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=4096)
    ap.add_argument("--agents", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=3, help="timed K-step blocks per region (median reported)")
    ap.add_argument("--comm", default="auto", help="multi-GPU gradient exchange: auto | p2p | p2p-multicast | nccl")
    ap.add_argument("--no-fused-rollout", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-kernel-rooflines", action="store_true")
    ap.add_argument("--skip-configs", action="store_true", help="headline only (no cfg1/3/4/5 entries)")
    ap.add_argument("--skip-parity-check", action="store_true")
    ap.add_argument("--cpu-envs", type=int, default=4096, help="n_envs of the reference's ia2c.py CPU run")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0, help="upper bound for the reference arm's CPU work")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed headline step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs:
        if args.impl != "ours":
            ap.error("--dump-outputs needs --impl ours")
        os.makedirs(args.dump_outputs, exist_ok=True)
    return args


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def med_spread(xs):
    xs = [float(x) for x in xs]
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "blocks": len(xs)}


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap,pcie.link.gen.current,pcie.link.width.current")

    def __init__(self, index):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(index)], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        self.marks = []

    def n_samples(self):
        try:
            return sum(1 for _ in open(self.tmp.name))
        except Exception:
            return 0

    def mark(self):
        self.marks.append(self.n_samples())

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        rows = []
        for line in open(self.tmp.name):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                try:
                    rows.append((float(parts[0]), float(parts[1]), parts[3:7], parts[7:9]))
                except ValueError:
                    pass
        os.unlink(self.tmp.name)
        lo = self.marks[0] if self.marks else 0
        hi = self.marks[1] if len(self.marks) > 1 else len(rows)
        load = rows[lo:max(hi, lo + 1)] or rows
        if not load:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(r[0] for r in load)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in load for i in range(4) if r[2][i].lower().startswith("active")})
        pcie = sorted({"gen" + "x".join(r[3]) for r in load if len(r[3]) == 2})
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[1] for r in load), "reasons": reasons, "samples": len(load),
                "pcie_link_seen": pcie}


# ------------------------------------------------------------------------------------------ CPU legs
def cpu_port_rate(n_agents, sample_envs, min_seconds, max_steps=None, warmup=1):
    """Times the oracle port (numpy restatement of ia2c.py's episode, oracle/loops.py) on the host cores."""
    import numpy as np
    from oracle import loops as L
    from ia2c_b200.trainer import reference_init

    actor, critic, fa = reference_init(n_agents, N_MODELS, seed=0)
    st = L.IA2CState(actor=actor, critic=critic, filter_action=fa)
    rng = np.random.RandomState(0)
    E, N, T = sample_envs, n_agents, T_STEPS

    def one():
        ua = rng.rand(T + 1, E, N).astype(np.float32)
        ub = rng.rand(T + 1, E, N, N - 1)
        L.ia2c_episode(st, E, u_act=ua, u_belief=ub)

    for _ in range(warmup):
        one()
    n, t0 = 0, time.perf_counter()
    while True:
        one()
        n += 1
        dt = time.perf_counter() - t0
        if (max_steps is not None and n >= max_steps) or (max_steps is None and dt >= min_seconds):
            break
    try:
        from threadpoolctl import threadpool_info
        blas = max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
    except Exception:
        blas = 1
    return dict(value=E * N * T * n / dt, seconds=dt, episodes=n, blas_threads=blas, ms_per_step=1e3 * dt / n)


def ref_runner(*argv, timeout=900):
    """Runs oracle/ref_runner.py (the UNMODIFIED reference files of oracle/_ref on the host CPU) in a fresh interpreter —
    the reference's module names (Org, ac_nets, belief_filter) must not meet the drop-in modules of this process.
    OMP/MKL thread limits that torchrun exports are dropped: the reference gets all the host threads it can use."""
    env = {k: v for k, v in os.environ.items() if k not in ("OMP_NUM_THREADS", "MKL_NUM_THREADS")}
    r = subprocess.run([sys.executable, "-m", "oracle.ref_runner", *[str(a) for a in argv]], capture_output=True, text=True,
                       cwd=ROOT, env=env, timeout=timeout)
    if r.returncode != 0:
        return None, (r.stderr or r.stdout).strip().splitlines()[-1:] or ["ref_runner failed"]
    return json.loads(r.stdout.strip().splitlines()[-1]), None


def cpu_baseline_legs(n_envs):
    """cpu_baseline for our arm's line (rank 0, N=1): the reference's own loops, bounded to ~20-30 s of CPU work."""
    out, err = ref_runner("all", "--envs", n_envs, "--warmup", 1, "--episodes", 6, "--warm-envs", 64)
    if out is None:
        r = cpu_port_rate(2, 2048, min_seconds=10.0)
        return {"value": r["value"], "unit": UNIT, "cores": r["blas_threads"], "kind": "port",
                "sample": f"{r['episodes']} episodes of 2048 envs x 2 agents x {T_STEPS} steps in {r['seconds']:.1f} s (oracle/loops.py "
                          f"numpy port; the staged reference was not available: {err})", "host_logical_cpus": os.cpu_count()}, None
    ia = out["ia2c"]
    base = {"value": ia["value"], "unit": UNIT, "cores": ia["torch_threads"], "kind": "reference",
            "sample": f"{ia['episodes']} episodes (after {ia['warmup']} warm-up) of the unmodified ia2c.py main loop (ia2c.py:62-134) at n_envs="
                      f"{ia['n_envs']}, 2 agents, T={T_STEPS}: {ia['seconds']:.1f} s; {ia['origin']}; gymnasium replaced by the in-process "
                      f"synchronous stand-in (oracle/gym_standin.py)",
            "ms_per_step": ia["ms_per_step"], "host_logical_cpus": ia["host_logical_cpus"], "torch_threads": ia["torch_threads"]}
    port = cpu_port_rate(2, 2048, min_seconds=4.0)
    base["port"] = {"value": port["value"], "unit": UNIT, "kind": "port", "cores": port["blas_threads"],
                    "sample": f"{port['episodes']} episodes of 2048 envs (oracle/loops.py vectorised numpy restatement; faster than the reference's own loop)"}
    return base, out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path — oracle/_ref/ia2c.py, unmodified, executed by
    oracle/ref_runner.py at the headline config (n_envs = envs per GPU), every step one episode of its main loop."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K, W = max(1, args.steps), max(0, args.warmup)
    n_envs = args.cpu_envs if args.cpu_envs != 4096 else args.envs_per_gpu
    config = {"workload": headline_workload(args.agents, args.envs_per_gpu, args.envs_per_gpu * max(1, args.gpus))}
    # a probe at 64 envs sizes the run: the loop's cost is linear in n_envs
    probe, err = ref_runner("ia2c", "--envs", 64, "--warmup", 1, "--episodes", 1)
    if probe is not None:
        per_ep = probe["ms_per_step"] * 1e-3 * n_envs / 64
        fit = int(args.cpu_budget_s / max(per_ep, 1e-6))
        w_eff = min(W, max(1, fit // 8))
        k_eff = max(1, min(K, fit - w_eff))
        out, err = ref_runner("ia2c", "--envs", n_envs, "--warmup", w_eff, "--episodes", k_eff, timeout=3600)
    if probe is None or out is None:
        r = cpu_port_rate(args.agents, min(n_envs, 2048), min_seconds=0, max_steps=K, warmup=max(1, min(W, 3)))
        kind, value, ms, k_eff, w_eff, cores = "port", r["value"], r["ms_per_step"], r["episodes"], W, r["blas_threads"]
        sample = (f"{r['episodes']} episodes of {min(n_envs, 2048)} envs x {args.agents} agents x {T_STEPS} steps, oracle/loops.py numpy port of "
                  f"ia2c.py:62-129 (staged reference unavailable: {err})")
        extra = {}
    else:
        kind, value, ms, cores = "reference", out["value"], out["ms_per_step"], out["torch_threads"]
        sample = (f"{k_eff} timed episodes (after {w_eff} warm-up) of the unmodified ia2c.py main loop at n_envs={n_envs}, 2 agents, "
                  f"T={T_STEPS} (rollout + critic + actor updates), {out['seconds']:.1f} s; {out['origin']}; gymnasium -> in-process "
                  f"synchronous stand-in (oracle/gym_standin.py), belief_filter_deprecated aliased as belief_filter")
        extra = {"torch_threads": out["torch_threads"], "per_episode_s": out["per_episode_s"]}
        if k_eff != K or w_eff != W:
            extra["bounded"] = f"asked for {W}+{K} episodes; {w_eff}+{k_eff} fit the {args.cpu_budget_s:.0f} s CPU budget"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": k_eff,
        "warmup": w_eff, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": config,
        "cpu_baseline": dict({"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                              "host_logical_cpus": os.cpu_count()}, **extra),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def headline_workload(n_agents, envs_per_gpu, envs_total):
    return (f"Org domain, {n_agents} agents, {envs_per_gpu} envs per GPU, T={T_STEPS}, M={N_MODELS} belief models, "
            f"rollout + critic + actor update (BASELINE configs[1] per GPU)")


# ------------------------------------------------------------------------------------------ helpers (GPU)
class Ctx:
    """Rank / device / collective helpers shared by the legs."""

    def __init__(self, torch):
        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        self._flush = None

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.dist is None:
            return float(x)
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def min_over_ranks(self, x):
        return -self.max_over_ranks(-x)

    def ev(self):
        return self.torch.cuda.Event(enable_timing=True)

    def flush(self):
        if self._flush is None:
            self._flush = self.torch.empty(256 << 20, dtype=self.torch.uint8, device=self.dev)  # > 126 MB L2
        self._flush.zero_()

    def drop_flush(self):
        self._flush = None


def time_steps_flushed(ctx, step_fns, K):
    """K steps, L2 flushed before each (outside the per-step events).  step_fns: callables executed in order per step; returns
    (ms summed over steps for the whole step, [ms of each segment])."""
    n_seg = len(step_fns)
    marks = [[ctx.ev() for _ in range(n_seg + 1)] for _ in range(K)]
    ctx.barrier()
    for m in marks:
        ctx.flush()
        m[0].record()
        for j, fn in enumerate(step_fns):
            fn()
            m[j + 1].record()
    ctx.barrier()
    total = sum(m[0].elapsed_time(m[-1]) for m in marks)
    segs = [sum(m[j].elapsed_time(m[j + 1]) for m in marks) for j in range(n_seg)]
    return total, segs


def time_block(ctx, fn, K):
    """K calls of fn back to back under one event pair -> per-rank ms."""
    ctx.barrier()
    s, e = ctx.ev(), ctx.ev()
    s.record()
    for _ in range(K):
        fn()
    e.record()
    ctx.barrier()
    return s.elapsed_time(e)


# ------------------------------------------------------------------------------------------ kernel rooflines
def fp32_issue_peak(torch, _lib):
    """Measured FP32 fma-pipe peak (csrc/debug.cu): FFMA2 (what the MLP kernels are written in) and scalar FFMA."""
    import ctypes as C
    lib = _lib.load()
    out = torch.zeros(1, dtype=torch.float32, device="cuda")
    res = {}
    for name, packed in (("ffma2", 1), ("ffma", 0)):
        flops = C.c_double(0.0)
        best = 0.0
        for _ in range(3):
            _lib.check(lib.ia2c_debug_fp32_peak(_lib.ptr(out), 4096, packed, 8, C.byref(flops), _lib.stream_ptr()))
        for _ in range(5):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            _lib.check(lib.ia2c_debug_fp32_peak(_lib.ptr(out), 4096, packed, 8, C.byref(flops), _lib.stream_ptr()))
            e.record()
            e.synchronize()
            best = max(best, flops.value / (s.elapsed_time(e) * 1e-3) / 1e12)
        res[name] = best
    return res


def kernel_rooflines(torch, _lib, peak_gbs):
    """Standalone streaming kernels at HBM-saturating sizes (algorithmic bytes per SURVEY.md §8 d4)."""
    lib = _lib.load()
    out = []
    dev = torch.device("cuda")

    def timeit(fn, iters=20):
        for _ in range(3):
            fn()
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        tot = 0.0
        for _ in range(iters):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            e.synchronize()
            tot += s.elapsed_time(e)
        return tot / iters * 1e-3

    def entry(kernel, units, bpu, nbytes, sec, **kw):
        d = {"kernel": kernel, "units": units, "bytes_per_unit": bpu, "achieved": nbytes / sec / 1e9, "peak": peak_gbs, "unit": "GB/s",
             "frac": nbytes / sec / 1e9 / peak_gbs, "bound": "hbm", "us": sec * 1e6}
        d.update(kw)
        return d

    # (1) Org env step, thread per env, N=2 per-agent uint8 actions
    E = 1 << 24
    from ia2c_b200.org_env import OrgVecEnv
    env = OrgVecEnv(E, n_agents=2)
    act = torch.randint(0, 3, (E, 2), dtype=torch.uint8, device=dev)
    st = _lib.stream_ptr()

    def env_step():
        _lib.check(lib.ia2c_org_step_agents(_lib.ptr(env.state), _lib.ptr(env.hist), _lib.ptr(env.cls), None, _lib.ptr(act),
                                            _lib.ptr(env.obs), None, _lib.ptr(env.reward_f32), None, None, E, 2, 0, st))
    sec = timeit(env_step)
    out.append(entry("org_step_thread_kernel", f"{E} env-steps (N=2)", 54, 54 * E, sec))
    del env, act
    # (1b) Org-N env step, a warp per 32 envs with the agents' action bytes in lanes (N=256 uint8 actions: 52 + N bytes per env-step)
    Ew, Nw = 1 << 21, 256
    env = OrgVecEnv(Ew, n_agents=Nw)
    act = torch.randint(0, 3, (Ew, Nw), dtype=torch.uint8, device=dev)

    def env_step_warp():
        _lib.check(lib.ia2c_org_step_agents(_lib.ptr(env.state), _lib.ptr(env.hist), _lib.ptr(env.cls), None, _lib.ptr(act),
                                            _lib.ptr(env.obs), None, _lib.ptr(env.reward_f32), None, None, Ew, Nw, 0, st))
    sec = timeit(env_step_warp)
    out.append(entry("org_step_warp32_kernel", f"{Ew} env-steps (N=256, Org-N)", 52 + Nw, (52 + Nw) * Ew, sec))
    del env, act
    # (2) belief update, dense reference layout (fp64 [R,5] in/out)
    R = 1 << 23
    fa = torch.rand(5, 3, dtype=torch.float64, device=dev)
    fa /= fa.sum(1, keepdim=True)
    lik = torch.full((R, 3), 0.1, dtype=torch.float64, device=dev)
    lik[torch.arange(R, device=dev), torch.randint(0, 3, (R,), device=dev)] = 0.8
    prev = torch.full((R, 5), 0.2, dtype=torch.float64, device=dev)
    u = torch.rand(R, dtype=torch.float64, device=dev)
    ap = torch.empty(R, dtype=torch.int64, device=dev)
    bp = torch.empty(R, 5, dtype=torch.float64, device=dev)

    def dense():
        _lib.check(lib.ia2c_belief_update_dense(_lib.ptr(fa), _lib.ptr(lik), _lib.ptr(prev), _lib.ptr(u), _lib.ptr(ap), _lib.ptr(bp),
                                                None, R, 5, 3, st))
    sec = timeit(dense)
    out.append(entry("belief_dense_kernel<5,3>", f"{R} belief updates", 88, 88 * R, sec,
                     note="the class API's interface forces 128 B/update of real traffic (likelihood row 24 B, u 8 B, int64 ap 8 B on top of "
                          "the algorithmic 88 B): ncu traffic / algorithmic = 1.31, i.e. 0.95 of HBM by actual bytes"))
    del lik, prev, u, ap, bp
    # (3) belief update, packed pairwise records at the config-5 per-GPU shape (1024 envs x 256 agents x 255 modelled others =
    #     1.07 GB of records read + written per launch) — K >= 32 dispatches to the table kernel
    En, N = 1024, 256
    K = N - 1
    rec = torch.zeros(En, N, K, 8, dtype=torch.uint8, device=dev)
    fan = torch.rand(N, 5, 3, dtype=torch.float64, device=dev)
    fan /= fan.sum(-1, keepdim=True)
    actn = torch.randint(0, 3, (En, N), dtype=torch.uint8, device=dev)
    partner = torch.empty(En, N, dtype=torch.uint8, device=dev)

    def pairs():
        _lib.check(lib.ia2c_belief_update_pairs(_lib.ptr(rec), _lib.ptr(fan), _lib.ptr(actn), None, None, None, _lib.ptr(partner),
                                                En, N, 5, 0, 1, 0, 1, 0, st))
    _lib.check(lib.ia2c_belief_update_pairs(_lib.ptr(rec), _lib.ptr(fan), _lib.ptr(actn), None, None, None, _lib.ptr(partner),
                                            En, N, 5, 1, 1, 0, 0, 0, st))
    sec = timeit(pairs)
    pairs_n = En * N * K
    out.append(entry("belief_pairs_table_kernel<5>", f"{pairs_n} (agent, modelled-other) updates, N=256", 16, 16 * pairs_n, sec,
                     pairs_per_s=pairs_n / sec,
                     note="uint8 records (16 B/update instead of the reference layout's 88 B) make this kernel instruction-issue bound, "
                          "not HBM bound (profiles/)"))
    del rec, fan, actn, partner
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------ legs of our arm
def make_trainer(ctx, E_total, N, fused=None, comm="auto", seed=1234, **kw):
    from ia2c_b200.trainer import IA2CTrainer, reference_init

    init = reference_init(N, N_MODELS, seed=0)  # identical on every rank
    return IA2CTrainer(E_total, n_agents=N, n_models=N_MODELS, steps_per_episode=T_STEPS, init=init, seed=seed, device=ctx.dev,
                       rank=ctx.rank, world_size=ctx.world, fused_rollout=fused, comm=comm, **kw)


DUMP_BYTES = 64_000_000
NPY_HEADER_BYTES = 256   # allowance per file for the .npy header (128 bytes for these shapes)


def dump_outputs(tr, out_dir, seed=0):
    """Writes what the trainer's last episode handed its caller — losses, episode returns, updated parameters and the episode's
    trajectory — as float32 / float64 DIR/<name>.npy, so that two builds can be compared output for output.  If the per-env
    files would exceed DUMP_BYTES on disk in all, they keep a fixed, seeded sample of envs; env_index.npy holds the global indices kept."""
    import numpy as np
    h = lambda t: t.detach().cpu().numpy()
    whole = {"critic_loss": h(tr.loss_out[0]), "actor_loss": h(tr.loss_out[1]),
             "actor_params": h(tr.actor_params), "critic_params": h(tr.critic_params)}
    per_env = {"ep_return": (h(tr.ep_return), 0), "obs": (h(tr.obs), 1), "reward": (h(tr.reward), 1),   # name -> (array, env axis)
               "act": (h(tr.act).astype(np.float32), 1), "partner_pred": (h(tr.partner_pred).astype(np.float32), 1)}
    env_bytes = sum(a.nbytes for a, _ in per_env.values()) // tr.E + 8
    room = (DUMP_BYTES - sum(a.nbytes for a in whole.values()) - NPY_HEADER_BYTES * (len(whole) + len(per_env) + 1)) // env_bytes
    keep = np.arange(tr.E) if tr.E <= room else np.sort(np.random.default_rng(seed).choice(tr.E, room, replace=False))
    for name, a in whole.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    for name, (a, axis) in per_env.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.take(a, keep, axis=axis))
    np.save(os.path.join(out_dir, "env_index.npy"), (tr.env_offset + keep).astype(np.float64))


def parity_check(ctx, comm):
    """Multi-rank self-check INSIDE the bench run: the sharded trainer (same comm path as the timed run) against a
    single-rank trainer of the same total workload on every GPU, as tests/multigpu_parity.py does.  Trajectories of the
    rank's env block must be byte-identical (random streams are keyed by the global env index); parameters agree up to the
    cross-rank summation order."""
    import numpy as np
    torch = ctx.torch
    ok, max_rel, cases = True, 0.0, []
    for N, E_total, fused in ((2, 64 * ctx.world, True), (66, 2 * ctx.world, False), (68, 2 * ctx.world, False)):
        sharded = make_trainer(ctx, E_total, N, fused=fused, comm=comm, seed=11, dumps=True)
        single_ctx_world, single_ctx_rank = ctx.world, ctx.rank
        from ia2c_b200.trainer import IA2CTrainer, reference_init
        single = IA2CTrainer(E_total, n_agents=N, init=reference_init(N, N_MODELS, seed=0), seed=11, device=ctx.dev,
                             fused_rollout=fused, dumps=True)
        for _ in range(2):
            sharded.train_episode()
            single.train_episode()
        torch.cuda.synchronize()
        sharded.check_comm()
        sl = slice(sharded.env_offset, sharded.env_offset + sharded.E)
        h = lambda t: t.detach().cpu().numpy()
        for name in ("obs", "reward", "act", "partner_pred", "partner_true", "belief_dump"):
            if not np.array_equal(h(getattr(sharded, name)), h(getattr(single, name))[:, sl]):
                ok = False
        for name in ("actor_params", "critic_params", "actor_grad_accum"):
            a, b = h(getattr(sharded, name)).astype(np.float64), h(getattr(single, name)).astype(np.float64)
            max_rel = max(max_rel, float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)))
        p = sharded.actor_params.clone()
        ctx.dist.broadcast(p, 0)
        if not torch.equal(p, sharded.actor_params):   # every rank must hold identical parameters
            ok = False
        cases.append(f"N={N} E={E_total}")
        del sharded, single
    if max_rel > 1e-6:
        ok = False
    ok = ctx.min_over_ranks(1.0 if ok else 0.0) > 0.5
    return {"ok": bool(ok), "max_rel": ctx.max_over_ranks(max_rel), "comm": comm, "cases": cases,
            "what": "2 episodes sharded vs single-rank on every GPU: trajectories byte-identical, parameters <= 1e-6 rel, ranks identical"}


def bench_headline(ctx, args, _lib, peak_gbs, peak_src, sampler):
    """cfg2 (weak scaling): region A (flushed per-step events), region B (back to back), e2e (host tapes through the C ABI)."""
    import numpy as np
    torch = ctx.torch
    N, E_gpu, T, M = args.agents, args.envs_per_gpu, T_STEPS, N_MODELS
    E_total = E_gpu * ctx.world
    fused = (not args.no_fused_rollout) and N <= 8
    tr = make_trainer(ctx, E_total, N, fused=fused, comm=args.comm)
    K, W, R = max(1, args.steps), max(3, args.warmup), max(1, args.repeats)
    for _ in range(W):
        tr.train_episode()
    ctx.barrier()
    if sampler:
        sampler.mark()
    # ---- region A: R blocks of K steps, L2 flushed between steps (outside the per-step events)
    def adv():
        tr.episode += 1
    blocks = []
    launches0 = _lib.launch_count()
    for r in range(R):   # one C call per episode per rank (world > 1: the two gradient exchanges are kernels in the same stream)
        total, _ = time_steps_flushed(ctx, [tr.train_episode], K)
        blocks.append(ctx.max_over_ranks(total))
    launches = (_lib.launch_count() - launches0) // R
    tr.check_comm()
    if args.dump_outputs and ctx.rank == 0:
        dump_outputs(tr, args.dump_outputs)
    total_ms = statistics.median(blocks)
    # the rollout kernel on its own (single rank): the same steps as three calls with an event between the phases -- the
    # records cost the programmatic-launch overlap between the kernels (~2 us each), so this pass feeds `roofline` only
    roll_ms = seg_ms = 0.0
    if ctx.world == 1:
        seg_ms, segs = time_steps_flushed(ctx, [tr.rollout, tr.update, adv], K)
        roll_ms = segs[0]
    # ---- region B: the same K steps back to back, one event pair (no flush)
    b2b = [ctx.max_over_ranks(time_block(ctx, tr.train_episode, K)) for _ in range(R)]
    tr.check_comm()
    # per-kernel split of a warm episode (single rank): CUDA events between the kernels inside one C call
    split = None
    if ctx.world == 1:
        acc = {}
        for _ in range(20):
            for k, v in tr.train_episode_timed().items():
                acc[k] = acc.get(k, 0.0) + v / 20
        split = acc
    # ---- e2e: the public host-buffer call — pinned uniforms H2D, episode, losses + returns D2H, one sync per call
    n_bufs = 4
    rng = np.random.RandomState(ctx.rank)
    tapes = [tr.pack_host_tape(rng.rand(T + 1, E_gpu, N).astype(np.float32), rng.rand(T + 1, E_gpu, N, N - 1)) for _ in range(n_bufs)]
    h2d, d2h = tapes[0].numel(), tr._result_region.numel()
    chunk = 50   # episodes per pipelined host call (each call ends with one stream sync)

    def e2e_run(n):
        done = 0
        while done < n:
            m = min(chunk, n - done)
            tr.train_episodes_host([tapes[(done + j) % n_bufs] for j in range(m)])
            done += m

    # warm-up with the SAME n (every buffer the timed call touches already exists) and for long enough that the PCIe link
    # has left its idle power state: the first tens of milliseconds of copies after a compute-only phase run at 10-20 GB/s
    # instead of ~50 GB/s (tools/e2e_probe.py, profiles/r02_e2e.md)
    for _ in range(max(1, -(-4000 // K))):
        e2e_run(K)
    e2e_blocks, e2e_wall = [], []
    for r in range(R):
        ctx.barrier()
        s, e = ctx.ev(), ctx.ev()
        t0 = time.perf_counter()
        s.record()
        e2e_run(K)
        e.record()
        e.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        ctx.barrier()
        e2e_wall.append(wall)
        e2e_blocks.append(ctx.max_over_ranks(max(s.elapsed_time(e), wall)))
    e2e_ms = statistics.median(e2e_blocks)
    # the e2e pipeline cannot run faster than its one pinned H2D copy per step: report that rate on this box next to it,
    # alone on this rank and with every rank copying at the same time (the ranks share the host's memory / PCIe root)
    probe_dst = torch.empty_like(tapes[0], device=ctx.dev)

    def h2d_probe(n=20):
        for _ in range(3):
            probe_dst.copy_(tapes[0], non_blocking=True)
        s, e = ctx.ev(), ctx.ev()
        s.record()
        for j in range(n):
            probe_dst.copy_(tapes[j % n_bufs], non_blocking=True)
        e.record()
        e.synchronize()
        return s.elapsed_time(e) / n * 1e3

    h2d_alone = None
    if ctx.world > 1:   # ranks take turns
        for r in range(ctx.world):
            ctx.barrier()
            if r == ctx.rank:
                h2d_alone = h2d_probe()
        ctx.barrier()
        h2d_all = ctx.max_over_ranks(h2d_probe())
    else:
        h2d_alone = h2d_probe()
        h2d_all = h2d_alone
    del probe_dst
    # keep the same load running until the clock sampler (rank 0) has data; the decision is COLLECTIVE
    for _ in range(50):
        need = 1 if (sampler is not None and sampler.n_samples() - sampler.marks[0] < 5) else 0
        if ctx.dist is not None:
            flag = torch.tensor([need], dtype=torch.int32, device=ctx.dev)
            ctx.dist.broadcast(flag, 0)
            need = int(flag.item())
        if not need:
            break
        for _ in range(200):
            tr.train_episode()
        torch.cuda.synchronize()
    if sampler:
        sampler.mark()
    tr.inject()  # back to the device Philox streams
    tr.check_comm()
    comm = tr.comm

    units = E_total * N * T  # agent-steps per step (whole job)
    line = {
        "metric": METRIC, "value": units * K / (total_ms * 1e-3), "unit": UNIT, "n_gpus": ctx.world, "steps": K, "warmup": W,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": DTYPE, "data": "synthetic",
        "config": {"workload": headline_workload(N, E_gpu, E_total), "envs_total": E_total,
                   "parallelism": (f"dp{ctx.world}: envs sharded, gradients of each optimiser phase exchanged by "
                                   + ("the fused NVLink all-reduce + Adam kernel (peer stores, comm=" + comm + ")" if comm.startswith("p2p")
                                      else "NCCL all-reduce (comm=nccl)")) if ctx.world > 1 else "single GPU",
                   "comm": comm,
                   "l2": "256 MiB buffer written between timed steps (L2 flush); per-step CUDA events summed",
                   "timing": f"{R} blocks of {K} steps per region; median block reported, spread in *_blocks_ms",
                   "sampler": "device Philox4x32-10 inverse-CDF (injected host uniforms in the e2e leg)",
                   "fused_rollout": fused, "roofline_peak_source": peak_src},
        "blocks_ms": med_spread(blocks),
        "back_to_back_ms_per_step": statistics.median(b2b) / K, "back_to_back_blocks_ms": med_spread(b2b),
        "e2e": {"value": units * K / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / K, "blocks_ms": med_spread(e2e_blocks), "wall_ms_per_step": statistics.median(e2e_wall) / K,
                "h2d_copy_us_alone": h2d_alone, "h2d_gbs_alone": h2d / (h2d_alone * 1e-6) / 1e9,
                "h2d_copy_us_all_ranks_at_once": h2d_all, "h2d_bound_ms_per_step": h2d_all * 1e-3,
                "api": ("IA2CTrainer.train_episodes_host -> ia2c_train_episodes_host (C ABI, pinned host tapes in, losses + returns "
                        "out per episode; one H2D and one D2H copy per episode, H2D of episode k+1 overlaps episode k; one sync per "
                        "50 episodes)") if ctx.world == 1 else
                       "IA2CTrainer.train_episodes_host -> ia2c_train_episodes_host_p2p (the same pipeline on every rank, fused NVLink "
                       "all-reduce + Adam after each gradient phase)"},
        "gpu_launches": int(launches),
    }
    # roofline of the dominant kernel: the rollout (fused: + critic gradient)
    traj_bytes = (T + 1) * E_gpu * (24 + 3 * N) + T * E_gpu * 4 + E_gpu * (26 + 8 * N * (N - 1))
    if fused:   # + the critic-gradient partials the fused critic stage writes (one 148-float row per block and agent)
        traj_bytes += (E_gpu * (2 if N <= 2 else 4 if N <= 4 else 8) // 32) * N * 148 * 4
    if ctx.world == 1:
        rollout_us = roll_ms / K * 1e3
        share = roll_ms / seg_ms
    else:
        rollout_us, share = None, None
    if rollout_us:
        achieved = traj_bytes / (rollout_us * 1e-6) / 1e9
        line["roofline"] = {
            "kernel": "rollout_fused_kernel (rollout + critic gradient)" if fused else "env_step_kernel + actor_step_kernel + belief_pairs_kernel (x31)",
            "bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
            "traffic": NCU_DRAM_BYTES.get(f"rollout_fused_kernel<2,5,1>@{E_gpu}") if (fused and N == 2) else None,
            "bytes_per_launch": traj_bytes, "us_per_launch": rollout_us, "share_of_step": share,
            "note": "latency/issue-bound by construction: 31 sequential steps per env and only E*N = 8192 lanes; the HBM figure is the "
                    "contract's, the meaningful denominator is the measured FP32 issue peak under 'issue' (SURVEY.md §8 d3)"}
    if split:
        line["episode_split_us"] = {k: v * 1e3 for k, v in split.items()}
    del tr, tapes
    ctx.drop_flush()
    torch.cuda.empty_cache()
    return line, comm, fused


def bench_org_n(ctx, args, _lib, name, label, E_total, N, steps, warmup, peak_gbs, cpu_ref_value, scaling):
    """cfg4 / cfg5: the many-agent Org-N trainer (builder-defined generalisation, DESIGN.md §8).  `scaling` "strong": E_total
    envs sharded over the ranks."""
    torch = ctx.torch
    lib = _lib.load()
    tr = make_trainer(ctx, E_total, N, comm=args.comm, seed=5)
    for _ in range(warmup):
        tr.train_episode()
    ctx.barrier()
    small = tr.belief_records.numel() < (256 << 20)   # working set within reach of the 126 MB L2 -> flush between steps
    l0 = _lib.launch_count()
    if small:
        total, _ = time_steps_flushed(ctx, [tr.train_episode], steps)
    else:
        total = time_block(ctx, tr.train_episode, steps)
    launches = _lib.launch_count() - l0
    ms = ctx.max_over_ranks(total) / steps
    tr.check_comm()
    # dominant kernel: the belief update of the episode's T+1 steps on the trainer's own buffers, same shape, timed standalone
    E, K = tr.E, N - 1
    st = _lib.stream_ptr()
    T1 = T_STEPS + 1
    episode_kernel = bool(lib.ia2c_belief_supports_episode(N, N_MODELS)) and not (tr.desc.flags & _lib.FLAG_BELIEF_PER_STEP)
    if episode_kernel:
        def belief():
            _lib.check(lib.ia2c_belief_update_pairs_episode(_lib.ptr(tr.belief_records), _lib.ptr(tr.filter_action), _lib.ptr(tr.act), None, None,
                                                            None, _lib.ptr(tr.partner_pred), E, N, N_MODELS, T1, 5, 0, tr.env_offset, st))
        launches_per_episode = 1
    else:
        def belief():
            _lib.check(lib.ia2c_belief_update_pairs(_lib.ptr(tr.belief_records), _lib.ptr(tr.filter_action), _lib.ptr(tr.act[1]), None, None, None,
                                                    _lib.ptr(tr.partner_pred[1]), E, N, N_MODELS, 0, 5, 0, 1, tr.env_offset, st))
        launches_per_episode = T1
    for _ in range(2):
        belief()
    n_b = 3 if episode_kernel else 6
    bs, be = ctx.ev(), ctx.ev()
    tot = 0.0
    for _ in range(n_b):
        if small:
            ctx.flush()
        bs.record(); belief(); be.record(); be.synchronize()
        tot += bs.elapsed_time(be)
    b_us = tot / n_b * 1e3
    pairs = E * N * K
    updates = pairs * (T1 if episode_kernel else 1)
    # actual unique bytes: the episode kernel writes each 8-byte record ONCE per episode and reads one action byte per update
    # (+ the partner mode per (env, agent, step)); the per-step kernel reads and writes the record at every update
    bytes_per_launch = (8 * pairs + updates + E * N * T1) if episode_kernel else 16 * pairs
    achieved = bytes_per_launch / (b_us * 1e-6) / 1e9
    units = E_total * N * T_STEPS
    value = units / (ms * 1e-3)
    roof = {"kernel": ("belief_pairs_episode_kernel<5>" if episode_kernel else ("belief_pairs_table_kernel<5>" if K >= 32 else "belief_pairs_kernel<5>")),
            "bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
            # ncu dram__bytes_read + write of one launch: 500.1 MB per 2.072e9 updates for the episode kernel at 1024 x 256
            # (profiles/r02_ncu_summary.md 1b), scaled to this shape; = the algorithmic 16 B per update for the per-step kernel
            "traffic": int(0.2416 * updates) if episode_kernel else bytes_per_launch,
            "bytes_per_launch": bytes_per_launch, "us_per_launch": b_us, "launches_per_episode": launches_per_episode,
            "share_of_step": launches_per_episode * b_us * 1e-3 / ms, "updates_per_s": updates / (b_us * 1e-6)}
    if episode_kernel:
        roof["streaming_equivalent"] = {"bytes_per_update": 16, "achieved": 16 * updates / (b_us * 1e-6) / 1e9,
                                        "frac": 16 * updates / (b_us * 1e-6) / 1e9 / peak_gbs}
        roof["note"] = ("the record stays in registers / shared memory for all T+1 updates of an episode and is written once, so the kernel "
                        "no longer streams: ~1.3 B of unique traffic per update instead of the 16 B (8-byte record read + written) of the per-step "
                        "kernel — it is bound by instruction issue on the ALU pipe (116 instructions per update, issue slots 71 %: "
                        "profiles/r02_ncu_summary.md). 'streaming_equivalent' is the HBM rate the per-step kernel (kernels[]: 0.42 of peak standalone) "
                        "would need for the same updates/s")
    else:
        roof["note"] = ("16 B per (agent, modelled-other) update: 8-byte record read + written (uint8-hundredths layout, lossless; the reference "
                        "layout would be 88 B); ncu dram traffic = the algorithmic 16 B/record (profiles/)")
    out = {"config": name, "workload": label, "envs_total": E_total, "envs_per_gpu": E, "agents": N, "n_gpus": ctx.world, "scaling": scaling,
           "steps": steps, "warmup": warmup, "ms_per_step": ms, "value": value, "unit": UNIT, "gpu_launches": int(launches), "comm": tr.comm,
           "l2": "L2 flushed between steps" if small else "back to back: the belief records (4.3 GB at 8192 x 256) outlive no episode in L2",
           "roofline": roof}
    if cpu_ref_value:
        out["cpu_baseline"] = {"value": cpu_ref_value, "unit": UNIT, "kind": "reference",
                               "sample": "agent-step-equivalent: the reference supports 2 agents only, its 2-agent ia2c.py rate per agent-step "
                                         "is quoted (SURVEY.md §8 d5)"}
    del tr
    ctx.drop_flush()
    torch.cuda.empty_cache()
    return out


def bench_cfg3(ctx, _lib, steps, peak_gbs, cpu):
    """cfg3: ac_nets critic + actor batch_update at a2c_test.py's shape (500 -> 6 -> 6 -> 6), batch 65536 = [64, 1024]."""
    import numpy as np
    torch = ctx.torch
    from ia2c_b200.nets import ActorNetwork, CriticNetwork
    T, E, F, O = 64, 1024, 500, 6
    rng = np.random.RandomState(0)
    idx = torch.from_numpy(rng.randint(0, F, size=(T, E)))
    act = torch.from_numpy(rng.randint(0, O, size=(T, E, 1)).astype(np.float32)).cuda()
    target, adv = torch.randn(T, E, 1).cuda(), torch.randn(T, E, 1).cuda()
    res = []
    for tag, obs in (("dense one-hot input float32[64,1024,500]", torch.nn.functional.one_hot(idx, F).float().cuda()),
                     ("index input int64[64,1024] (no one-hot tensor)", idx.cuda())):
        critic = CriticNetwork("c", F, O, 5e-4)
        actor = ActorNetwork("a", F, O, 1e-4, 0.01)

        def pair():
            critic.batch_update(obs, act, target)
            actor.batch_update(obs, act, adv)
        for _ in range(3):
            pair()
        torch.cuda.synchronize()
        dev_ms = 0.0
        t0 = time.perf_counter()
        for _ in range(steps):
            s, e = ctx.ev(), ctx.ev()
            s.record(); pair(); e.record(); e.synchronize()
            dev_ms += s.elapsed_time(e)
        wall = (time.perf_counter() - t0) / steps
        entry = {"input": tag, "ms_per_step": wall * 1e3, "device_ms_per_step": dev_ms / steps, "value": T * E / wall, "unit": "rows/s"}
        if obs.dtype.is_floating_point:
            # the dominant kernel timed on its own: ia2c_net_update (critic) through the C ABI, L2 flushed, CUDA events
            x_bytes = T * E * F * 4
            lib = _lib.load()
            P = 6 * F + 6 + 36 + 6 + 6 * O + O
            z = lambda n, dt=torch.float32: torch.zeros(n, dtype=dt, device="cuda")
            p_, g_, m_, v_, st_, ls_ = torch.randn(P, device="cuda") * 0.3, z(P), z(P), z(P), z(1, torch.int32), z(1)
            ws = torch.empty(int(lib.ia2c_net_update_workspace(T * E, F, O)), dtype=torch.float32, device="cuda")
            a_i, sig = act.reshape(-1).to(torch.int32).contiguous(), target.reshape(-1).contiguous()
            x2 = obs.reshape(-1, F)
            D = lambda t: t.data_ptr()

            def upd():
                _lib.check(lib.ia2c_net_update(0, D(p_), D(g_), D(m_), D(v_), D(st_), D(x2), None, D(a_i), D(sig), 0.0, 5e-4, D(ls_), None,
                                               D(ws), T * E, F, O, _lib.stream_ptr()))
            for _ in range(3):
                upd()
            tot = 0.0
            for _ in range(10):
                ctx.flush()
                s, e = ctx.ev(), ctx.ev()
                s.record(); upd(); e.record(); e.synchronize()
                tot += s.elapsed_time(e)
            us = tot / 10 * 1e3
            entry["roofline"] = {"kernel": "net_update_dense_kernel<0> + net_update_reduce_adam_kernel (one critic update, X read once)",
                                 "bound": "hbm", "achieved": x_bytes / (us * 1e-6) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                                 "frac": x_bytes / (us * 1e-6) / 1e9 / peak_gbs, "traffic": 135582464, "bytes_per_launch": x_bytes,
                                 "us_per_launch": us,
                                 "note": "single pass: 32-row tiles by cp.async.bulk + mbarrier, forward products and dW1 from the same staged "
                                         "tile; ncu dram__bytes_read = 131.6 MB = rows x F x 4 (profiles/r02_ncu_summary.md); the kernel alone "
                                         "takes 48 us (0.42), the figure here includes the reduce + Adam kernel and launch gaps"}
            ctx.drop_flush()
            del ws, x2
        res.append(entry)
        del critic, actor, obs
    out = {"config": "cfg3", "workload": "ac_nets CriticNetwork/ActorNetwork.batch_update pair (ac_nets.py:62-80,112-127) at a2c_test.py's "
                                         "shape 500->6->6->6, batch 65536 (BASELINE configs[2])", "steps": steps, "inputs": res,
           "ms_per_step": res[0]["ms_per_step"], "value": res[0]["value"], "unit": "rows/s"}
    if cpu:
        out["cpu_baseline"] = {"value": cpu["value"], "unit": "rows/s", "ms_per_step": cpu["ms_per_step"], "cores": cpu["torch_threads"],
                               "kind": "reference", "sample": f"{cpu['updates']} update pairs of the unmodified ac_nets.py classes on the host, dense one-hot input"}
    torch.cuda.empty_cache()
    return out


def bench_cfg1(ctx, updates, cpu):
    """cfg1: a2c_org_test.py's loop — one Org instance, 100 steps + critic and actor update per iteration.  With the staged
    reference script present it is the UNMODIFIED a2c_org_test.py run on the drop-in modules (ia2c_b200.launcher)."""
    import builtins
    import contextlib
    import io
    from ia2c_b200 import launcher
    from oracle import ref_runner
    ref, origin = ref_runner.find_reference()
    if ref is None:
        return {"config": "cfg1", "unavailable": f"the reference's a2c_org_test.py is not staged under oracle/_ref ({origin})"}
    path = os.path.join(ref, "a2c_org_test.py")
    warm = 5
    stamps = []
    real_print = builtins.print

    def stamped(*a, **k):
        ctx.torch.cuda.synchronize()
        stamps.append(time.perf_counter())
    builtins.print = stamped
    saved_path, saved_mods = list(sys.path), set(sys.modules)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            t_start = time.perf_counter()
            launcher.run_script(path, {"n_updates": warm + updates})
    finally:
        builtins.print = real_print
        sys.path[:] = saved_path
    per = [b - a for a, b in zip(stamps[warm - 1:-1], stamps[warm:])]
    ms = 1e3 * sum(per) / len(per)
    out = {"config": "cfg1", "workload": "a2c_org_test.py main loop, unmodified script on the drop-in modules: 1 Org instance, 100 env steps "
                                         "(Org.step + sample_action each) + critic and actor batch_update per iteration (BASELINE configs[0])",
           "steps": len(per), "warmup": warm, "ms_per_step": ms, "value": 100 / (ms * 1e-3), "unit": "env-steps/s",
           "note": "single env, single Python thread: every env step is a host round trip (launch + .item()), so this config measures "
                   "launch latency, not the GPU; it exists for drop-in parity (tests/test_gpu_reference_scripts.py)"}
    if cpu:
        out["cpu_baseline"] = {"value": cpu["value"], "unit": "env-steps/s", "ms_per_step": cpu["ms_per_step"], "cores": cpu["torch_threads"],
                               "kind": "reference", "sample": f"{cpu['updates']} iterations of the unmodified a2c_org_test.py on the host"}
    return out


# ------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch

    from ia2c_b200 import _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference for the CPU arm)")
    ctx = Ctx(torch)
    if args.gpus != ctx.world and ctx.rank == 0 and ctx.world > 1:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={ctx.world}; using WORLD_SIZE", file=sys.stderr)
    peaks, peak_src = measured_peaks()
    peak_gbs = float(peaks["hbm_gbs"])
    sampler = ClockSampler(ctx.local) if ctx.rank == 0 else None
    try:
        line, comm, fused = bench_headline(ctx, args, _lib, peak_gbs, peak_src, sampler)
    finally:   # the nvidia-smi sampler must not outlive a failed run
        clocks = sampler.stop() if sampler else None
    line["clocks"] = clocks
    single = ctx.world == 1
    # ---- multi-rank self-check on the same comm path the timed regions used
    if not single and not args.skip_parity_check:
        line["parity_check"] = parity_check(ctx, comm)
    # ---- CPU legs (rank 0, N=1): the reference's own loops on this box's host cores
    cpu_all = None
    if ctx.rank == 0 and single and not args.skip_cpu_baseline:
        line["cpu_baseline"], cpu_all = cpu_baseline_legs(args.cpu_envs)
    # ---- measured FP32 issue peak and the two MLP-bound kernels of the headline step as a fraction of it
    if ctx.rank == 0 and single and not args.skip_kernel_rooflines:
        pk = fp32_issue_peak(torch, _lib)
        units_gpu = args.envs_per_gpu * args.agents * T_STEPS
        split = line.get("episode_split_us") or {}
        issue = {"peak_tflops_ffma2": pk["ffma2"], "peak_tflops_ffma": pk["ffma"],
                 "how": "ia2c_debug_fp32_peak: independent register-resident fma chains, 148 x 8 blocks x 256 threads, best of 5, CUDA events"}
        if fused and split.get("rollout"):
            f = (FLOPS_ROLLOUT + FLOPS_CRITIC) * units_gpu / (split["rollout"] * 1e-6) / 1e12
            issue["rollout_fused_kernel"] = {"tflops": f, "frac_of_ffma2_peak": f / pk["ffma2"], "us": split["rollout"],
                                             "flops_per_agent_step": FLOPS_ROLLOUT + FLOPS_CRITIC}
        if split.get("actor_grad"):
            f = FLOPS_ACTOR * units_gpu / (split["actor_grad"] * 1e-6) / 1e12
            issue["actor_grad_kernel"] = {"tflops": f, "frac_of_ffma2_peak": f / pk["ffma2"], "us": split["actor_grad"],
                                          "flops_per_agent_step": FLOPS_ACTOR}
        if "roofline" in line:
            line["roofline"]["issue"] = issue
        line["kernels"] = kernel_rooflines(torch, _lib, peak_gbs)
    # ---- the other BASELINE configs
    if not args.skip_configs:
        cpu2 = (line.get("cpu_baseline") or {}).get("value") if (line.get("cpu_baseline") or {}).get("kind") == "reference" else None
        cfgs = []
        k5 = max(2, min(args.steps, 5 * ctx.world))
        cfgs.append(bench_org_n(ctx, args, _lib, "cfg5", "Org-N (builder-defined many-agent Org, DESIGN.md §8): 256 agents/env x 8192 envs in total, "
                                "sharded over the ranks, K=255 modelled others per agent, rollout + critic + actor update (BASELINE configs[4])",
                                8192, 256, k5, 2, peak_gbs, cpu2, "strong"))
        if single:
            cfgs.append(bench_org_n(ctx, args, _lib, "cfg4", "Org-N: 64 agents/env x 1024 envs, K=63 modelled others per agent (BASELINE configs[3])",
                                    1024, 64, max(2, min(args.steps, 30)), 3, peak_gbs, cpu2, "single GPU"))
            if ctx.rank == 0:
                cfgs.append(bench_cfg3(ctx, _lib, max(3, min(args.steps, 30)), peak_gbs, (cpu_all or {}).get("acnets")))
                cfgs.append(bench_cfg1(ctx, max(3, min(args.steps, 20)), (cpu_all or {}).get("a2c_org")))
        line["configs"] = cfgs
    if ctx.rank == 0:
        print(json.dumps(line))
    if ctx.dist is not None:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()
    if "parity_check" in line and not line["parity_check"]["ok"]:
        sys.exit(3)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
