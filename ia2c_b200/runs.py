"""IA2CRuns — many independent IA2C training runs (seeds, hyper-parameter sweeps) advanced together on one GPU.

One episode of every run is ONE C call (``ia2c_train_episode_runs``) whose four launches each cover all R runs: the
standalone episode is latency-bound and leaves most of the B200 idle, so R runs cost far less than R standalone
episodes.  Run r computes byte for byte what ``IA2CTrainer(envs_per_run, seed=seeds[r], init=reference_init(N, M,
seed=seeds[r]), <run r's hyper-parameters>)`` computes over the same episodes (include/ia2c_b200.h states the contract).
``IA2CRunsMany`` does the same for Org-N runs of 9 to 256 agents in SIX launches per episode (``ia2c_train_episode_runs_many``);
its run r is byte-identical to that trainer with ``actor_kernel="columns"``.

The device buffers hold the runs stacked (DESIGN.md §3): per-net buffers have R*N rows, run r at rows [r*N, (r+1)*N);
per-env buffers have an env axis of length R*E, run r at [r*E, (r+1)*E).  ``run_view(r)`` returns those slices and
``run_state_dict(r)`` a checkpoint that a standalone ``IA2CTrainer`` loads, so the best run of a sweep can go on alone.

``exploit_explore`` runs one generation of population-based training on the device between episodes (``ia2c_pbt_step``):
the worst runs by recent recorded returns take copies of the best runs' state and perturbed copies of their
hyper-parameters; ``pbt_history`` reads back what each generation did.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from .history import DeviceRing, RecordsHistory
from .trainer import N_ACTIONS, N_FEATURES, IA2CTrainer, reference_init

# buffers with one row per (run, agent), and buffers with an env axis (its position) of length R * E
_NET = ("actor_params", "critic_params", "actor_grad", "critic_grad", "actor_grad_accum", "actor_m", "actor_v", "critic_m",
        "critic_v", "actor_step", "critic_step", "filter_action")
_ENV = {"env_state": 0, "env_hist": 0, "env_cls": 0, "env_elapsed": 0, "ep_return": 0, "belief_records": 0,
        "obs": 1, "reward": 1, "act": 1, "partner_true": 1, "partner_pred": 1}
# the per-run hyper-parameters, in ia2c_runs_desc order, with their device dtype
_HYPER = (("lr_actor", torch.float64), ("lr_critic", torch.float64), ("gamma", torch.float32), ("beta", torch.float32))
_PERTURB = {"lr_actor": _lib.PBT_LR_ACTOR, "lr_critic": _lib.PBT_LR_CRITIC, "beta": _lib.PBT_BETA}


def _per_run(name, value, R, dtype):
    """A hyper-parameter given as a scalar (-> (None, value): the descriptor's scalar serves every run) or as a length-R
    sequence (-> (array, value[0]))."""
    if np.ndim(value) == 0:
        v = float(value)
        if not math.isfinite(v):
            raise ValueError(f"{name} must be finite, got {value!r}")
        return None, v
    arr = np.asarray(value, dtype=np.float64)
    if arr.ndim != 1 or arr.shape[0] != R:
        raise ValueError(f"{name} must be a scalar or a sequence of one value per run ({R}), got shape {arr.shape}")
    if not np.all(np.isfinite(arr)):
        raise ValueError(f"{name} must be finite")
    return arr.astype(dtype), float(arr[0])


class IA2CRuns(RecordsHistory):
    # the C entry point of one batched episode and the descriptor flags it takes
    _ENTRY = "ia2c_train_episode_runs"
    _FLAGS = _lib.FLAG_FUSED_ROLLOUT | _lib.FLAG_FUSED_CRITIC | _lib.FLAG_ACTOR_COLUMNS
    PBT_LOG_CAPACITY = 16   # generations the device log holds before it drains (allocated on first use)
    _pbt_log = None
    _pbt_generation = 0     # generations run so far: the Philox counter of the next one
    _pbt_mark = 0           # the history ring's record count at the previous generation

    @classmethod
    def _check_shape(cls, lib, N, M):
        """Raises ValueError, before any device work, for an (n_agents, n_models) the entry point has no kernels for."""
        if not lib.ia2c_rollout_fused_supported(N, M):
            raise ValueError(f"n_agents={N}, n_models={M}: batches of runs need the fused path (N <= 8 with M = 5, or N = 2 with M = 3)")

    def __init__(self, envs_per_run, seeds, n_agents=2, n_models=5, steps_per_episode=30, max_episode_steps=30,
                 lr_critic=0.0002, lr_actor=0.0001, beta=0.001, gamma=0.9, init=None, device=None):
        self.lib = _lib.load()
        seeds = [int(s) for s in seeds]
        R, E, N, M, T = len(seeds), int(envs_per_run), int(n_agents), int(n_models), int(steps_per_episode)
        if R < 1:
            raise ValueError("seeds: need at least one run")
        if any(s < 0 or s >= 1 << 64 for s in seeds):
            raise ValueError("seeds must lie in [0, 2**64)")
        if E < 1 or not 0 < T < 65535:
            raise ValueError(f"envs_per_run={E} must be >= 1 and steps_per_episode={T} in 1..65534")
        self._check_shape(self.lib, N, M)
        if R * N > _lib.MAX_RUN_NETS:
            raise ValueError(f"runs * n_agents = {R * N} above the limit of {_lib.MAX_RUN_NETS}")
        hyper = {name: _per_run(name, v, R, dt) for name, v, dt in
                 (("lr_actor", lr_actor, np.float64), ("lr_critic", lr_critic, np.float64),
                  ("gamma", gamma, np.float32), ("beta", beta, np.float32))}
        if init is not None and len(init) != R:
            raise ValueError(f"init: need one (actor, critic, filter_action) tuple per run ({R}), got {len(init)}")
        _lib.require_cuda()
        self.R, self.E, self.N, self.M, self.T, self.K = R, E, N, M, T, N - 1
        self.seeds = seeds
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.episode = 0
        dev, RN, RE, K = self.device, R * N, R * E, N - 1

        def z(shape, dtype):
            return torch.zeros(shape, dtype=dtype, device=dev)

        f32, f64, u8, i32 = torch.float32, torch.float64, torch.uint8, torch.int32
        self.actor_params, self.critic_params = z((RN, _lib.ACTOR_P), f32), z((RN, _lib.CRITIC_P), f32)
        self.actor_grad, self.critic_grad = z((RN, _lib.ACTOR_P + 1), f32), z((RN, _lib.CRITIC_P + 1), f32)
        self.actor_grad_accum = z((RN, _lib.ACTOR_P), f32)
        self.actor_m, self.actor_v = z((RN, _lib.ACTOR_P), f32), z((RN, _lib.ACTOR_P), f32)
        self.critic_m, self.critic_v = z((RN, _lib.CRITIC_P), f32), z((RN, _lib.CRITIC_P), f32)
        self.actor_step, self.critic_step = z((RN,), i32), z((RN,), i32)
        self.loss_out = z((2, RN), f32)
        self.filter_action = z((RN, M, N_ACTIONS), f64)
        self.env_state, self.env_hist = z((RE,), i32), z((RE,), f64)
        self.env_cls, self.env_elapsed = z((RE, 2), u8), z((RE,), i32)
        self.ep_return = z((RE,), f64)
        self.obs, self.reward = z((T + 1, RE, N_FEATURES), f32), z((T, RE), f32)
        self.act, self.partner_true, self.partner_pred = z((T + 1, RE, N), u8), z((T + 1, RE, N), u8), z((T + 1, RE, N), u8)
        self.belief_records = z((RE, N, K, _lib.BELIEF_RECORD), u8)
        self._seed = torch.from_numpy(np.asarray(seeds, dtype=np.uint64).view(np.int64)).to(dev)
        self._hyper = {k: (torch.from_numpy(a).to(dev) if a is not None else None) for k, (a, _) in hyper.items()}
        self._built_hyper = {k: a for k, (a, _) in hyper.items()}   # per-run arrays as given, None for a scalar (desc holds it)

        d = self.desc = _lib.EpisodeDesc()
        d.E, d.E_total, d.env_offset = E, E, 0
        d.N, d.T, d.M, d.max_episode_steps = N, T, M, int(max_episode_steps or 0)
        d.lr_actor, d.lr_critic = hyper["lr_actor"][1], hyper["lr_critic"][1]
        d.gamma, d.beta = hyper["gamma"][1], hyper["beta"][1]
        d.flags = self._FLAGS
        for name in _NET + tuple(_ENV) + ("loss_out",):
            setattr(d, name, getattr(self, name).data_ptr())
        n_part = int(self.lib.ia2c_runs_partials_floats(C.byref(d), R))
        self.partials = z((n_part,), f32)
        d.partials, d.partials_floats = self.partials.data_ptr(), n_part
        r = self.runs_desc = _lib.RunsDesc()
        r.runs, r.seed = R, self._seed.data_ptr()
        for k, t in self._hyper.items():
            setattr(r, k, t.data_ptr() if t is not None else None)

        self.critic_losses, self.actor_losses, self.reward_lst = [], [], []
        for k in range(R):
            self._load_init(k, *(init[k] if init is not None else reference_init(N, M, seed=seeds[k])))

    def _load_init(self, r, actor, critic, filter_action):
        rows = slice(r * self.N, (r + 1) * self.N)
        self.actor_params[rows].copy_(torch.as_tensor(np.asarray(actor), dtype=torch.float32))
        self.critic_params[rows].copy_(torch.as_tensor(np.asarray(critic), dtype=torch.float32))
        self.filter_action[rows].copy_(torch.as_tensor(np.asarray(filter_action), dtype=torch.float64))

    # ------------------------------------------------------------------ episodes
    def train_episode(self, sync_stats=False):
        """One episode of every run in one C call; asynchronous unless ``sync_stats``.  ``train_episodes(n)`` trains n
        episodes and records their statistics on the device for ``history()``; those episodes do not enter the
        ``read_stats`` windows."""
        self.desc.episode = self.episode
        with torch.cuda.device(self.device):
            _lib.check(getattr(self.lib, self._ENTRY)(C.byref(self.desc), C.byref(self.runs_desc),
                                                      torch.cuda.current_stream(self.device).cuda_stream),
                       self._ENTRY)
        self.episode += 1
        if sync_stats:
            return self.read_stats()

    def _history_dims(self):
        return self.R, self.N, self.E, self.T, False

    def _enqueue_episode(self, desc_ref, stream):
        _lib.check(getattr(self.lib, self._ENTRY)(desc_ref, C.byref(self.runs_desc), stream), self._ENTRY)

    def read_stats(self):
        """The last episode's losses ``[R, N]`` and returns ``[R, E]``, appended to each run's windows as
        ``IA2CTrainer._record_stats`` does (20-deep loss windows, last-50 returns); the window means are per run."""
        R, N, E = self.R, self.N, self.E
        loss = self.loss_out.cpu().numpy()
        ret = self.ep_return.cpu().numpy().reshape(R, E)
        critic, actor = loss[0].reshape(R, N), loss[1].reshape(R, N)
        self.critic_losses.append(critic), self.actor_losses.append(actor)
        del self.critic_losses[:-20], self.actor_losses[:-20]
        self.reward_lst.append(ret)
        del self.reward_lst[:-50]
        return dict(critic_loss=critic, actor_loss=actor, ep_return=ret,
                    critic_loss_window=np.mean(self.critic_losses, axis=0), actor_loss_window=np.mean(self.actor_losses, axis=0),
                    mean_return=np.array([np.mean([x[r] for x in self.reward_lst]) for r in range(R)]))

    # ------------------------------------------------------------------ one run's slice
    def run_view(self, r):
        """Views (no copies) of run r's slices of every device buffer, under the names ``IA2CTrainer`` uses."""
        if not 0 <= r < self.R:
            raise IndexError(f"run {r} of {self.R}")
        N, E = self.N, self.E
        v = {k: getattr(self, k)[r * N:(r + 1) * N] for k in _NET}
        for k, axis in _ENV.items():
            v[k] = getattr(self, k).narrow(axis, r * E, E)
        v["loss_out"] = self.loss_out[:, r * N:(r + 1) * N]
        return v

    def run_state_dict(self, r):
        """Run r as a checkpoint of a standalone ``IA2CTrainer(envs_per_run, ..., seed=seeds[r])``: its
        ``load_state_dict`` accepts it and the run continues alone bit-identically in
        ``IA2CTrainer(..., actor_kernel="columns")`` (the default up to 64 agents)."""
        torch.cuda.current_stream(self.device).synchronize()
        v = self.run_view(r)
        sd = {k: v[k].detach().cpu().clone() for k in IA2CTrainer._CKPT_TENSORS}
        sd.update(episode=self.episode, seed=self.seeds[r], dims=(self.E, self.E, self.N, self.M, self.T), rank=0, world=1,
                  critic_losses=[x[r].copy() for x in self.critic_losses], actor_losses=[x[r].copy() for x in self.actor_losses],
                  reward_lst=[x[r].copy() for x in self.reward_lst])
        return sd

    # ------------------------------------------------------------------ checkpoint / resume of the whole batch
    def state_dict(self):
        torch.cuda.current_stream(self.device).synchronize()
        sd = {k: getattr(self, k).detach().cpu().clone() for k in IA2CTrainer._CKPT_TENSORS}
        sd.update(episode=self.episode, seeds=list(self.seeds), dims=(self.R, self.E, self.N, self.M, self.T),
                  critic_losses=[x.copy() for x in self.critic_losses], actor_losses=[x.copy() for x in self.actor_losses],
                  reward_lst=[x.copy() for x in self.reward_lst])
        if self._pbt_generation > 0:   # PBT changed the hyper-parameters: they are part of the runs' state now
            sd.update(hyper={k: self._hyper[k].detach().cpu().clone() for k, _ in _HYPER}, pbt_generation=self._pbt_generation)
        return sd

    def load_state_dict(self, sd):
        """Restores parameters, optimiser, env and belief state, the episode counter, the runs' seeds and the windows.  A
        checkpoint taken after a PBT generation also restores the per-run hyper-parameters and the generation counter; one
        taken before any generation sets the hyper-parameters back to those this batch was built with (as
        ``IA2CTrainer.load_state_dict`` keeps them) and the generation counter to 0.  Either way the next ``exploit_explore``
        counts only episodes recorded after the load."""
        if tuple(sd["dims"]) != (self.R, self.E, self.N, self.M, self.T):
            raise ValueError(f"checkpoint is for (runs, E, N, M, T) = {tuple(sd['dims'])}, batch has {(self.R, self.E, self.N, self.M, self.T)}")
        for k in IA2CTrainer._CKPT_TENSORS:
            getattr(self, k).copy_(sd[k])
        self.episode = int(sd["episode"])
        self.seeds = [int(s) for s in sd["seeds"]]
        self._seed.copy_(torch.from_numpy(np.asarray(self.seeds, dtype=np.uint64).view(np.int64)))
        self.critic_losses, self.actor_losses = list(sd["critic_losses"]), list(sd["actor_losses"])
        self.reward_lst = list(sd["reward_lst"])
        if "pbt_generation" in sd:
            with torch.cuda.device(self.device):
                self._materialise_hyper()
            for k, _ in _HYPER:
                self._hyper[k].copy_(sd["hyper"][k])
            self._pbt_generation = int(sd["pbt_generation"])
        elif self._pbt_generation > 0:   # PBT changed this batch's hyper-parameters; the checkpoint predates any generation
            for k, _ in _HYPER:
                built = self._built_hyper[k]
                if built is None:
                    self._hyper[k].fill_(getattr(self.desc, k))   # the array holds the scalar, as _materialise_hyper fills it
                else:
                    self._hyper[k].copy_(torch.from_numpy(built))
            self._pbt_generation = 0
        self._pbt_mark = self._history.head if self._history is not None else 0   # the ring's records predate the load

    def save(self, path):
        torch.save(self.state_dict(), path)

    def load(self, path):
        self.load_state_dict(torch.load(path, map_location="cpu", weights_only=False))

    # ------------------------------------------------------------------ frozen-policy evaluation
    def evaluate(self, episodes=1, num_envs=None, greedy=False, seed=0, first_episode=0):
        """``IA2CTrainer.evaluate`` for every run at once (default ``num_envs``: envs_per_run; greedy: 1), with a leading
        run axis on every result (returns [R, K, E], mean_return [R], ...).  All runs see the same random numbers, so their
        returns are paired samples, and run r's results equal those of a standalone trainer holding ``run_state_dict(r)``."""
        from .evaluate import evaluate_actors

        E = (1 if greedy else self.E) if num_envs is None else num_envs
        return evaluate_actors(self.actor_params, self.R, self.N, E, episodes, self.T, self.desc.max_episode_steps, greedy,
                               seed, first_episode, self.device)

    def cross_play(self, episodes=1, num_envs=None, greedy=False, seed=0, first_episode=0, split=None):
        """``evaluate.cross_play(self, ...)``: the R x R matrix of this batch's runs played against each other (cell (a, b)
        seats agents 0 .. split-1 of run a and the rest of run b); the diagonal is each run's ``evaluate``."""
        from .evaluate import cross_play

        return cross_play(self, episodes=episodes, num_envs=num_envs, greedy=greedy, seed=seed, first_episode=first_episode,
                          split=split)

    def agent_steps_per_episode(self):
        return self.R * self.E * self.N * self.T

    # ------------------------------------------------------------------ population-based training
    def run_hyper(self, r):
        """Run r's current lr_actor, lr_critic, gamma and beta as Python floats (synchronises once PBT has changed them):
        ``IA2CTrainer(envs_per_run, n_agents=N, n_models=M, seed=seeds[r], **run_hyper(r))`` loaded with
        ``run_state_dict(r)`` continues run r bit-identically."""
        if not 0 <= r < self.R:
            raise IndexError(f"run {r} of {self.R}")
        return {k: float(self._hyper[k][r].item()) if self._hyper[k] is not None else float(getattr(self.desc, k))
                for k, _ in _HYPER}

    def _materialise_hyper(self):
        """Give every hyper-parameter a device array (filled from the scalar where the batch was built with one) and point
        the runs descriptor at it; the kernels compute the same bytes from the array as from the scalar."""
        for k, dtype in _HYPER:
            if self._hyper[k] is None:
                self._hyper[k] = torch.full((self.R,), getattr(self.desc, k), dtype=dtype, device=self.device)
                setattr(self.runs_desc, k, self._hyper[k].data_ptr())

    def _pbt_args(self, window, fraction, perturb, factors, seed):
        """exploit_explore's checks, all before any device work -> (window, q, perturb mask, factors, seed)."""
        window, fraction, seed = int(window), float(fraction), int(seed)
        cap = self._history.capacity if self._history is not None else self.HISTORY_CAPACITY
        if not 1 <= window <= cap - 1:
            raise ValueError(f"window={window} outside [1, HISTORY_CAPACITY - 1 = {cap - 1}]")
        if not 0.0 <= fraction <= 0.5:
            raise ValueError(f"fraction={fraction} outside [0, 0.5]: donors and recipients must be disjoint")
        mask = 0
        for name in ((perturb,) if isinstance(perturb, str) else perturb):
            if name == "gamma":
                raise ValueError("perturb: gamma is inherited from the donor, never perturbed")
            if name not in _PERTURB:
                raise ValueError(f"perturb: unknown hyper-parameter {name!r} (lr_actor, lr_critic, beta)")
            mask |= _PERTURB[name]
        factors = tuple(float(f) for f in factors)
        if len(factors) != 2 or not all(math.isfinite(f) and f > 0 for f in factors):
            raise ValueError(f"factors={factors}: need two finite factors > 0")
        if not 0 <= seed < 1 << 64:
            raise ValueError(f"seed={seed} outside [0, 2**64)")
        if self._history is None:
            raise ValueError("exploit_explore ranks runs by the returns train_episodes records: this batch has no history ring yet")
        recorded = self._history.head - self._pbt_mark
        if recorded < window:
            raise ValueError(f"window={window}: only {recorded} episodes recorded by train_episodes since the previous generation")
        return window, int(math.floor(fraction * self.R)), mask, factors, seed

    def exploit_explore(self, window, fraction=0.25, perturb=("lr_actor", "lr_critic", "beta"), factors=(0.8, 1.2), seed=0):
        """One generation of population-based training, on the device and asynchronous (include/ia2c_b200.h,
        ia2c_pbt_step, states the definitions).  Run r's fitness is the fp64 sum of its return_sum over the last ``window``
        episodes recorded by ``train_episodes``, oldest first; runs rank by fitness, higher first, NaN last, ties to the lower
        index.  Each of the bottom q = floor(fraction * R) runs takes a donor from the top q (Philox stream 5 keyed by
        ``seed``, counter word 3 the generation): its parameters, Adam moments and steps, actor gradient sum and belief
        models become a byte copy of the donor's, and it inherits the donor's hyper-parameters, each name in ``perturb``
        multiplied by factors[0] or factors[1].  A recipient keeps its seed, env state and statistics windows.  Afterwards
        run r equals ``IA2CTrainer(E, n_agents=N, n_models=M, seed=seeds[r], **run_hyper(r))`` (``actor_kernel="columns"``
        for N > 8) loaded with ``run_state_dict(r)``.  Two launches; the log (``pbt_history``) drains, synchronising, once
        every ``PBT_LOG_CAPACITY - 1`` generations that ``pbt_history`` has not read."""
        window, q, mask, (lo, hi), seed = self._pbt_args(window, fraction, perturb, factors, seed)
        ring, R = self._history, self.R
        with torch.cuda.device(self.device):
            self._materialise_hyper()
            if self._pbt_log is None:
                self._pbt_log = DeviceRing(self.device, self.PBT_LOG_CAPACITY, (
                    ("fitness", np.float64, (R,)), ("rank", np.int32, (R,)), ("donor", np.int32, (R,)),
                    ("lr_actor", np.float64, (R,)), ("lr_critic", np.float64, (R,)), ("gamma", np.float32, (R,)),
                    ("beta", np.float32, (R,))), ("generation", "episode"))
                self._pbt_ws = torch.empty(int(self.lib.ia2c_pbt_workspace_bytes(R)), dtype=torch.uint8, device=self.device)
            log = self._pbt_log
            slot = log.free_slot()
            p = _lib.PbtDesc()
            p.window, p.slot, p.q, p.perturb = window, (ring.head - 1) % ring.capacity, q, mask
            p.factor_lo, p.factor_hi, p.seed, p.generation = lo, hi, seed, self._pbt_generation
            for k, _ in _HYPER:
                setattr(p, k, self._hyper[k].data_ptr())
            for k in ("fitness", "rank", "donor", "lr_actor", "lr_critic", "gamma", "beta"):
                setattr(p, "log_" + k, log.ptr[k] + slot * log.row_bytes[k])
            p.workspace, p.workspace_bytes = self._pbt_ws.data_ptr(), self._pbt_ws.numel()
            _lib.check(self.lib.ia2c_pbt_step(C.byref(self.desc), C.byref(self.runs_desc), ring._href, C.byref(p),
                                              torch.cuda.current_stream(self.device).cuda_stream), "ia2c_pbt_step")
        log.commit(generation=self._pbt_generation, episode=self.episode)
        self._pbt_generation += 1
        self._pbt_mark = ring.head

    def pbt_history(self):
        """Synchronise and return every PBT generation since the previous call, generation axis first: ``generation`` and
        ``episode`` (the episode counter at the call) [g]; ``fitness`` f64, ``rank`` i32 and ``donor`` i32 (-1: the run kept
        its own state) [g, R]; ``lr_actor``, ``lr_critic`` (f64), ``beta`` and ``gamma`` (f32) [g, R] after the step.  The log
        is not part of a checkpoint: call this before ``save``."""
        chunks = self._pbt_log.take_chunks() if self._pbt_log is not None else []
        shapes = dict(generation=(np.int64, ()), episode=(np.int64, ()), fitness=(np.float64, (self.R,)),
                      rank=(np.int32, (self.R,)), donor=(np.int32, (self.R,)), lr_actor=(np.float64, (self.R,)),
                      lr_critic=(np.float64, (self.R,)), beta=(np.float32, (self.R,)), gamma=(np.float32, (self.R,)))
        return {k: (np.concatenate([c[k] for c in chunks]) if chunks else np.zeros((0,) + shape, dtype=dt))
                for k, (dt, shape) in shapes.items()}


class IA2CRunsMany(IA2CRuns):
    """R independent Org-N runs with 9 <= n_agents <= 256 (cfg4: 64 agents, cfg5: 256) in the six launches of one episode
    (``ia2c_train_episode_runs_many``): the whole-episode rollout and belief kernels, the critic gradient, the column actor
    gradient and both reduce + Adam steps, each covering all runs.  Run r computes byte for byte what
    ``IA2CTrainer(envs_per_run, n_agents=N, n_models=M, seed=seeds[r], init=reference_init(N, M, seed=seeds[r]),
    actor_kernel="columns", <run r's hyper-parameters>)`` computes.  Above 64 agents a standalone trainer defaults to the
    pipelined actor kernel, whose sums are ordered differently: the contract is with the column kernel.

    Layout, statistics, recorded histories (``train_episodes`` / ``history``), ``run_view`` / ``run_state_dict``, checkpoints
    and ``evaluate`` are those of ``IA2CRuns``."""
    _ENTRY = "ia2c_train_episode_runs_many"
    _FLAGS = _lib.FLAG_ACTOR_COLUMNS

    @classmethod
    def _check_shape(cls, lib, N, M):
        if N <= 8:
            raise ValueError(f"n_agents={N}: batches of N <= 8 agents run on the fused path, IA2CRuns")
        if N > 256:
            raise ValueError(f"n_agents={N} above 256: batches of runs cover 9..256 agents")
        if not lib.ia2c_belief_supports_episode(N, M):
            raise ValueError(f"n_models={M} outside 2..6")

    def __init__(self, envs_per_run, seeds, n_agents, n_models=5, steps_per_episode=30, max_episode_steps=30,
                 lr_critic=0.0002, lr_actor=0.0001, beta=0.001, gamma=0.9, init=None, device=None):
        super().__init__(envs_per_run, seeds, n_agents=n_agents, n_models=n_models, steps_per_episode=steps_per_episode,
                         max_episode_steps=max_episode_steps, lr_critic=lr_critic, lr_actor=lr_actor, beta=beta, gamma=gamma,
                         init=init, device=device)
