"""Frozen-policy evaluation of IA2C actors on the GPU (``ia2c_evaluate``, include/ia2c_b200.h).

``evaluate_actors`` is the entry point: ``IA2CTrainer.evaluate`` and ``IA2CRuns.evaluate`` hand it their actor parameters.
``eval_desc`` is the one place that fills an ``ia2c_eval_desc`` (tools/bench_eval.py times the C call on it).  It reads them on the current stream of their device and writes nothing but the outputs it
allocates, so the training state is untouched.  With the same ``seed`` and ``episode0`` every run sees the same random
numbers, so the returns of the runs of a sweep are paired samples.

Cross-play (``ia2c_evaluate_lineups``): ``evaluate_lineups`` plays lineups whose seats are filled from a pool of actors, and
``cross_play`` builds the run-by-run matrix of a sweep from trainers and batches (``IA2CRuns.cross_play``).  ``lineup_desc``
is the one place that fills an ``ia2c_lineup_desc``.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib


def eval_desc(actor_params, R, N, E, K, T, max_episode_steps, greedy, seed, episode0, policy, returns, counts, tape=None):
    """The ``ia2c_eval_desc`` of one evaluation into caller-owned device outputs (policy f32[R*N, 9, 3], returns
    f64[R, K, E], counts 64-bit [R*N, 3]; tape f32[K, T, R*E, N] or None).  The library validates it."""
    d = _lib.EvalDesc()
    d.actor_params, d.R, d.N, d.E = actor_params.data_ptr(), R, N, E
    d.episodes, d.T, d.max_episode_steps, d.greedy = K, T, max_episode_steps, int(greedy)
    d.seed, d.episode0 = seed, episode0
    d.inj_u_action = tape.data_ptr() if tape is not None else None
    d.policy, d.policy_floats = policy.data_ptr(), policy.numel()
    d.returns, d.action_counts = returns.data_ptr(), counts.data_ptr()
    return d


def evaluate_actors(actor_params, R, N, envs, episodes, T, max_episode_steps, greedy, seed, episode0, device, u_action=None):
    """Evaluate R runs' actors (``actor_params`` f32[R*N, 105] on ``device``, run r at rows [r*N, (r+1)*N)) for ``episodes``
    episodes of T steps in each of ``envs`` envs per run.  ``u_action`` f32[episodes, T, R*envs, N] replaces the Philox
    uniforms (tests); greedy takes argmax actions and needs envs = episodes = 1.  Returns host arrays with a leading run axis:
    returns [R, episodes, envs] f64, mean_return / std_return [R], action_counts [R, N, 3] u64, action_freq [R, N, 3]
    (counts / (episodes * envs * T)), policy [R, N, 9, 3] f32 and, for greedy, greedy_actions [R, N, 9]."""
    R, N, E, K, T, mes = int(R), int(N), int(envs), int(episodes), int(T), int(max_episode_steps or 0)
    seed, episode0, greedy = int(seed), int(episode0), bool(greedy)
    if not 1 <= R <= _lib.EVAL_MAX_RUNS or not 2 <= N <= _lib.EVAL_MAX_AGENTS or R * N > _lib.MAX_RUN_NETS:
        raise ValueError(f"runs={R}, n_agents={N}: need 1 <= runs <= {_lib.EVAL_MAX_RUNS}, 2 <= n_agents <= "
                         f"{_lib.EVAL_MAX_AGENTS} and runs * n_agents <= {_lib.MAX_RUN_NETS}")
    if E < 1 or K < 1 or not 1 <= T <= _lib.EVAL_MAX_STEPS or mes < 0:
        raise ValueError(f"envs={E}, episodes={K} must be >= 1, T={T} in 1..{_lib.EVAL_MAX_STEPS}, max_episode_steps={mes} >= 0")
    if not 0 <= seed < 1 << 64 or episode0 < 0 or episode0 + K > 1 << 32:
        raise ValueError(f"seed={seed} must lie in [0, 2**64) and first episode {episode0} + episodes {K} within 2**32")
    if greedy and (E * K != 1 or u_action is not None):
        raise ValueError(f"greedy evaluation is deterministic: it plays one episode in one env per run (got envs={E}, "
                         f"episodes={K}) and takes no uniform tape")
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = torch.device(device)
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    if (actor_params.device != dev or actor_params.dtype != torch.float32 or not actor_params.is_contiguous()
            or tuple(actor_params.shape) != (R * N, _lib.ACTOR_P)):
        raise ValueError(f"actor_params must be a contiguous float32 [{R * N}, {_lib.ACTOR_P}] tensor on {dev}")
    with torch.cuda.device(dev):
        policy = torch.empty((R * N, 9, 3), dtype=torch.float32, device=dev)
        returns = torch.empty((R, K, E), dtype=torch.float64, device=dev)
        counts = torch.empty((R * N, 3), dtype=torch.int64, device=dev)
        tape = None
        if u_action is not None:
            tape = torch.as_tensor(u_action).to(dev, torch.float32).contiguous()
            if tuple(tape.shape) != (K, T, R * E, N):
                raise ValueError(f"u_action has shape {tuple(tape.shape)}, expected {(K, T, R * E, N)}")
        d = eval_desc(actor_params, R, N, E, K, T, mes, greedy, seed, episode0, policy, returns, counts, tape)
        _lib.check(lib.ia2c_evaluate(C.byref(d), torch.cuda.current_stream(dev).cuda_stream), "ia2c_evaluate")
        ret = returns.cpu().numpy()          # synchronises the stream (and keeps the tape alive until the kernels ran)
    cnt = counts.cpu().numpy().view(np.uint64).reshape(R, N, 3)
    pol = policy.cpu().numpy().reshape(R, N, 9, 3)
    out = dict(returns=ret, mean_return=ret.reshape(R, -1).mean(1), std_return=ret.reshape(R, -1).std(1),
               action_counts=cnt, action_freq=cnt / float(K * E * T), policy=pol)
    if greedy:
        out["greedy_actions"] = pol.argmax(-1)   # ties -> lowest action, as the kernel takes them
    return out


def lineup_desc(actor_params, nets, N, lineups, E, K, T, max_episode_steps, greedy, seed, episode0, policy, returns, counts,
                return_sum, return_m2, tape=None):
    """The ``ia2c_lineup_desc`` of one cross-play evaluation into caller-owned device outputs (pool actor_params f32[nets, 105],
    lineups i32[P, N], policy f32[nets, 9, 3], returns f64[P, K, E], counts 64-bit [P*N, 3], return_sum / return_m2 f64[P];
    tape f32[K, T, P*E, N] or None).  The library validates it."""
    d = _lib.LineupDesc()
    d.actor_params, d.nets, d.N = actor_params.data_ptr(), nets, N
    d.P, d.lineups, d.E = lineups.shape[0], lineups.data_ptr(), E
    d.episodes, d.T, d.max_episode_steps, d.greedy = K, T, max_episode_steps, int(greedy)
    d.seed, d.episode0 = seed, episode0
    d.inj_u_action = tape.data_ptr() if tape is not None else None
    d.policy, d.policy_floats = policy.data_ptr(), policy.numel()
    d.returns, d.action_counts = returns.data_ptr(), counts.data_ptr()
    d.return_sum, d.return_m2 = return_sum.data_ptr(), return_m2.data_ptr()
    return d


def _check_run_args(E, K, T, mes, seed, episode0, greedy, tape):
    if E < 1 or K < 1 or not 1 <= T <= _lib.EVAL_MAX_STEPS or mes < 0:
        raise ValueError(f"envs={E}, episodes={K} must be >= 1, T={T} in 1..{_lib.EVAL_MAX_STEPS}, max_episode_steps={mes} >= 0")
    if not 0 <= seed < 1 << 64 or episode0 < 0 or episode0 + K > 1 << 32:
        raise ValueError(f"seed={seed} must lie in [0, 2**64) and first episode {episode0} + episodes {K} within 2**32")
    if greedy and (E * K != 1 or tape is not None):
        raise ValueError(f"greedy evaluation is deterministic: it plays one episode in one env per lineup (got envs={E}, "
                         f"episodes={K}) and takes no uniform tape")


def evaluate_lineups(actor_params, n_agents, lineups, envs, episodes, T, max_episode_steps, greedy, seed, episode0, device,
                     u_action=None):
    """Evaluate P lineups seated from a pool of actors (``actor_params`` f32[nets, 105] on ``device``): seat i of lineup p is
    pool row ``lineups[p, i]`` (int [P, N]; rows may repeat and change seats).  Lineup p plays ``episodes`` episodes of T steps
    in each of ``envs`` envs and computes byte for byte what ``evaluate_actors`` computes for one run of the actors
    ``actor_params[lineups[p]]`` with the same arguments, so all lineups see the same random numbers.  ``u_action`` f32[episodes,
    T, P*envs, N] replaces the Philox uniforms (tests).  Returns host arrays: mean_return / std_return [P] (ddof 0, from the
    device's fixed-order sums), action_counts [P, N, 3] u64 and action_freq [P, N, 3]; the returns stay on the device."""
    N, E, K, T, mes = int(n_agents), int(envs), int(episodes), int(T), int(max_episode_steps or 0)
    seed, episode0, greedy = int(seed), int(episode0), bool(greedy)
    if not 2 <= N <= _lib.EVAL_MAX_AGENTS:
        raise ValueError(f"n_agents={N} outside 2..{_lib.EVAL_MAX_AGENTS}")
    _check_run_args(E, K, T, mes, seed, episode0, greedy, u_action)
    nets = int(actor_params.shape[0]) if actor_params is not None and actor_params.ndim == 2 else 0
    host = lineups.detach().cpu().numpy() if hasattr(lineups, "detach") else np.asarray(lineups)
    if host.ndim != 2 or host.shape[1] != N or not 1 <= host.shape[0] <= _lib.EVAL_MAX_LINEUPS or host.dtype.kind not in "iu":
        raise ValueError(f"lineups must be an integer array [P, {N}] with 1 <= P <= {_lib.EVAL_MAX_LINEUPS}, got "
                         f"{host.dtype} {host.shape}")
    bad = (host < 0) | (host >= nets)
    if bad.any():
        p, i = np.argwhere(bad)[0]
        raise ValueError(f"lineups[{p}, {i}] = {host[p, i]} outside the pool's rows [0, {nets})")
    P = host.shape[0]
    torch = _lib.require_cuda()
    lib = _lib.load()
    dev = torch.device(device)
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    if (actor_params.device != dev or actor_params.dtype != torch.float32 or not actor_params.is_contiguous()
            or tuple(actor_params.shape) != (nets, _lib.ACTOR_P)):
        raise ValueError(f"actor_params must be a contiguous float32 [nets, {_lib.ACTOR_P}] tensor on {dev}")
    with torch.cuda.device(dev):
        lin = torch.from_numpy(np.ascontiguousarray(host, dtype=np.int32)).to(dev)
        policy = torch.empty((nets, 9, 3), dtype=torch.float32, device=dev)
        returns = torch.empty((P, K, E), dtype=torch.float64, device=dev)
        counts = torch.empty((P * N, 3), dtype=torch.int64, device=dev)
        stats = torch.empty((2, P), dtype=torch.float64, device=dev)
        tape = None
        if u_action is not None:
            tape = torch.as_tensor(u_action).to(dev, torch.float32).contiguous()
            if tuple(tape.shape) != (K, T, P * E, N):
                raise ValueError(f"u_action has shape {tuple(tape.shape)}, expected {(K, T, P * E, N)}")
        d = lineup_desc(actor_params, nets, N, lin, E, K, T, mes, greedy, seed, episode0, policy, returns, counts, stats[0],
                        stats[1], tape)
        _lib.check(lib.ia2c_evaluate_lineups(C.byref(d), torch.cuda.current_stream(dev).cuda_stream), "ia2c_evaluate_lineups")
        st = stats.cpu().numpy()             # synchronises the stream (and keeps lineups and tape alive until the kernels ran)
    cnt = counts.cpu().numpy().view(np.uint64).reshape(P, N, 3)
    n = float(K * E)
    return dict(mean_return=st[0] / n, std_return=np.sqrt(st[1] / n), action_counts=cnt, action_freq=cnt / float(K * E * T))


def cross_play(sources, episodes=1, num_envs=None, greedy=False, seed=0, first_episode=0, split=None):
    """The cross-play matrix of trained runs.  ``sources`` is an ``IA2CTrainer`` (one run), an ``IA2CRuns`` /
    ``IA2CRunsMany`` (its R runs), or a list of them sharing n_agents, steps_per_episode, max_episode_steps and device; runs
    are numbered in source order.  Cell (a, b) seats agents 0 .. split-1 of run a and agents split .. N-1 of run b, each in its
    own seat (default split = N // 2), so the diagonal is self-play and equals each run's ``evaluate``.  Every cell plays
    ``episodes`` episodes in each of ``num_envs`` envs (default: the first source's envs per run; greedy: 1) with the same
    random numbers (``evaluate_lineups``): the cells are paired samples.  Nothing of any source is written.  Returns
    mean_return / std_return [R, R], action_freq [R, R, N, 3] and the lineups used (i32 [R*R, N], rows of the sources'
    actor_params concatenated in source order)."""
    from .runs import IA2CRuns
    from .trainer import IA2CTrainer

    srcs = list(sources) if isinstance(sources, (list, tuple)) else [sources]
    if not srcs:
        raise ValueError("cross_play: no sources")
    for s in srcs:
        if not isinstance(s, (IA2CTrainer, IA2CRuns)):
            raise ValueError(f"cross_play: a source must be an IA2CTrainer, IA2CRuns or IA2CRunsMany, got {type(s).__name__}")
    first = srcs[0]
    N, T, mes, dev = first.N, first.T, int(first.desc.max_episode_steps), first.device
    for s in srcs[1:]:
        theirs = (s.N, s.T, int(s.desc.max_episode_steps), s.device)
        if theirs != (N, T, mes, dev):
            raise ValueError(f"cross_play: sources must share (n_agents, steps_per_episode, max_episode_steps, device) = "
                             f"{(N, T, mes, dev)}, got {theirs}")
    runs = [s.R if isinstance(s, IA2CRuns) else 1 for s in srcs]
    R = sum(runs)
    split = N // 2 if split is None else int(split)
    if not 1 <= split <= N - 1:
        raise ValueError(f"split={split} outside 1..{N - 1}: each cell seats agents of two runs")
    if R * R > _lib.EVAL_MAX_LINEUPS:
        raise ValueError(f"{R} runs make {R * R} cells, above the limit of {_lib.EVAL_MAX_LINEUPS} lineups")
    E = (1 if greedy else (first.E if isinstance(first, IA2CRuns) else first.E_total)) if num_envs is None else int(num_envs)
    torch = _lib.require_cuda()
    base = np.arange(R, dtype=np.int64)[:, None] * N                      # pool row of agent 0 of each run
    seat = np.arange(N, dtype=np.int64)
    a, b = np.repeat(np.arange(R), R), np.tile(np.arange(R), R)           # cell p = a * R + b
    lineups = np.where(seat < split, base[a] + seat, base[b] + seat).astype(np.int32)
    with torch.cuda.device(dev):
        pool = torch.cat([s.actor_params for s in srcs]) if len(srcs) > 1 else first.actor_params
        out = evaluate_lineups(pool, N, lineups, E, episodes, T, mes, greedy, seed, first_episode, dev)
    return dict(mean_return=out["mean_return"].reshape(R, R), std_return=out["std_return"].reshape(R, R),
                action_freq=out["action_freq"].reshape(R, R, N, 3), lineups=lineups)
