"""Frozen-policy evaluation of IA2C actors on the GPU (``ia2c_evaluate``, include/ia2c_b200.h).

``evaluate_actors`` is the entry point: ``IA2CTrainer.evaluate`` and ``IA2CRuns.evaluate`` hand it their actor parameters.
``eval_desc`` is the one place that fills an ``ia2c_eval_desc`` (tools/bench_eval.py times the C call on it).  It reads them on the current stream of their device and writes nothing but the outputs it
allocates, so the training state is untouched.  With the same ``seed`` and ``episode0`` every run sees the same random
numbers, so the returns of the runs of a sweep are paired samples.
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
