"""Training against frozen partners (``ia2c_seat_partners``, include/ia2c_b200.h).

A ``PartnerPool`` is a frozen device copy of actor rows, the partner seats and the teams that fill them.  While a pool is
set (``set_partners`` on ``IA2CTrainer`` at one GPU, ``IA2CRuns`` and ``IA2CRunsMany``), every call that starts an episode
first enqueues one launch that draws a team for each run (Philox stream 6 keyed by the run's training seed and the episode
number) and copies its rows into the run's partner seats; the episode then runs as it always does.  So the learning seats
train against partners drawn from a population instead of against one co-learning partner (fictitious co-play, population
play), and run r of a batch still equals a standalone trainer with the same seed and the same pool.

The partner seats' critics and actors are updated by the episode as before; those updates are discarded when the next
episode seats a partner again.  ``partner_history`` reads back which team every run played.

``set_partners(pool, per_env=True)`` draws a team for every ENV instead (Philox stream 7 keyed by the run's training seed, the
episode number and the env's index within its run), and the rollout kernels play each env's team in that env
(``ia2c_train_episode_env_partners``): a learner of E envs meets up to E partners per episode instead of one.  The partner
seats' own actor rows are not used to act while the mode is on; they still receive every episode's update, and after
``set_partners(None)`` self-play continues from them.  ``env_partner_history`` reads back the team of every env.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .history import DeviceRing


def _host_ints(x, name):
    a = x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    if a.dtype.kind not in "iu":
        raise ValueError(f"{name} must be an integer array, got {a.dtype}")
    return a


class PartnerPool:
    """``rows`` f32[P, 105] actor rows, ``teams`` int [Q, S] and ``seats`` int [S] for runs of ``n_agents`` agents: team t
    seats row ``teams[t, j]`` in seat ``seats[j]``.  Seats are distinct, lie in [0, n_agents) and leave at least one seat
    learning (1 <= S <= n_agents - 1).  Everything is checked on the host; then the rows are copied to ``device`` (default:
    the rows' CUDA device, else the current one), so the pool is frozen: training the rows' source later changes nothing."""

    def __init__(self, rows, teams, seats, n_agents, device=None):
        N = int(n_agents)
        if N < 2:
            raise ValueError(f"n_agents={N}: a pool needs a partner seat and a learning seat")
        dt = rows.dtype if isinstance(rows, torch.Tensor) else getattr(rows, "dtype", None)
        if dt not in (torch.float32, np.float32):
            raise ValueError(f"rows must be float32, got {dt}")
        if rows.ndim != 2 or rows.shape[1] != _lib.ACTOR_P or rows.shape[0] < 1:
            raise ValueError(f"rows must have shape [P >= 1, {_lib.ACTOR_P}], got {tuple(rows.shape)}")
        P = int(rows.shape[0])
        seats, teams = _host_ints(seats, "seats"), _host_ints(teams, "teams")
        if seats.ndim != 1 or not 1 <= seats.shape[0] <= N - 1:
            raise ValueError(f"seats must be a list of 1 .. n_agents - 1 = {N - 1} seats, got shape {seats.shape}")
        if seats.min() < 0 or seats.max() >= N:
            raise ValueError(f"seats {seats.tolist()} outside [0, {N})")
        if np.unique(seats).shape[0] != seats.shape[0]:
            raise ValueError(f"seats {seats.tolist()} repeat a seat")
        S = int(seats.shape[0])
        if teams.ndim != 2 or teams.shape[1] != S or not 1 <= teams.shape[0] <= _lib.PARTNER_MAX_TEAMS:
            raise ValueError(f"teams must have shape [Q, {S}] with 1 <= Q <= {_lib.PARTNER_MAX_TEAMS}, got {teams.shape}")
        bad = (teams < 0) | (teams >= P)
        if bad.any():
            t, j = np.argwhere(bad)[0]
            raise ValueError(f"teams[{t}, {j}] = {teams[t, j]} outside the pool's rows [0, {P})")
        _lib.require_cuda()
        if device is None:
            device = rows.device if isinstance(rows, torch.Tensor) and rows.is_cuda else torch.cuda.current_device()
        dev = torch.device(device)
        if dev.type != "cuda":
            raise ValueError(f"device={device}: a pool lives on a CUDA device")
        self.device = torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())
        self.N, self.P, self.S, self.Q = N, P, S, int(teams.shape[0])
        with torch.cuda.device(self.device):
            self.rows = torch.as_tensor(rows).to(self.device, torch.float32, copy=True).contiguous()
            self.teams = torch.from_numpy(np.ascontiguousarray(teams, dtype=np.int32)).to(self.device)
            self.seats = torch.from_numpy(np.ascontiguousarray(seats, dtype=np.int32)).to(self.device)

    @classmethod
    def from_sources(cls, sources, split=None):
        """A pool of the runs of ``sources`` (an ``IA2CTrainer``, ``IA2CRuns`` / ``IA2CRunsMany``, or a list of them sharing
        n_agents and device; runs numbered in source order, as ``cross_play`` numbers them): seats split .. N-1 (default
        split = N // 2) and team b = agents split .. N-1 of run b.  A learner trained with it plays the lineups of
        ``cross_play``'s cells (learner, b).  The rows are copied now, on the sources' stream."""
        from .runs import IA2CRuns
        from .trainer import IA2CTrainer

        srcs = list(sources) if isinstance(sources, (list, tuple)) else [sources]
        if not srcs:
            raise ValueError("from_sources: no sources")
        for s in srcs:
            if not isinstance(s, (IA2CTrainer, IA2CRuns)):
                raise ValueError(f"from_sources: a source must be an IA2CTrainer, IA2CRuns or IA2CRunsMany, got {type(s).__name__}")
        N, dev = srcs[0].N, srcs[0].device
        for s in srcs[1:]:
            if (s.N, s.device) != (N, dev):
                raise ValueError(f"from_sources: sources must share (n_agents, device) = {(N, dev)}, got {(s.N, s.device)}")
        split = N // 2 if split is None else int(split)
        if not 1 <= split <= N - 1:
            raise ValueError(f"split={split} outside 1..{N - 1}: a pool needs a partner seat and a learning seat")
        R, S = sum(s.R if isinstance(s, IA2CRuns) else 1 for s in srcs), N - split
        with torch.cuda.device(dev):
            rows = torch.cat([s.actor_params.view(-1, N, _lib.ACTOR_P)[:, split:].reshape(-1, _lib.ACTOR_P) for s in srcs])
        return cls(rows, np.arange(R * S, dtype=np.int32).reshape(R, S), np.arange(split, N, dtype=np.int32), N, device=dev)

    _policy = None

    def policy_table(self, lib):
        """The pool's policy table f32[P, 9, 3] (``ia2c_partner_policy``: row p's softmax at observation class 3 * prev + cur),
        built on the first call on the device's current stream and kept on the pool."""
        if self._policy is None:
            with torch.cuda.device(self.device):
                table = torch.empty((self.P, 9, 3), dtype=torch.float32, device=self.device)
                _lib.check(lib.ia2c_partner_policy(self.rows.data_ptr(), self.P, table.data_ptr(),
                                                   torch.cuda.current_stream(self.device).cuda_stream), "ia2c_partner_policy")
            self._policy = table
        return self._policy

    def state(self):
        """rows, teams and seats as CPU tensors (what a checkpoint carries)."""
        return {k: getattr(self, k).detach().cpu().clone() for k in ("rows", "teams", "seats")}


class SeatsPartners:
    """``set_partners`` / ``partner_history`` for a trainer class that defines ``_partner_runs()`` -> (runs, runs descriptor
    reference or None for one standalone run keyed by ``desc.seed``) and calls ``_seat_partners(stream)`` before every
    episode it starts."""

    PARTNER_LOG_CAPACITY = 64   # seated episodes the device log holds before it drains (allocated on first use)
    ENV_PARTNER_LOG_CAPACITY = 16   # per-env episodes the device log of env teams holds before it drains (allocated on first use)
    _partners = None
    _partner_log = None
    _env_partners = False       # per-env mode
    _env_partner_log = None

    def _check_partners(self):
        """Raise, before any device work, where partners cannot be seated."""

    def _check_env_partners(self):
        """Raise, before any device work, where partners cannot be played per env."""

    def set_partners(self, pool, per_env=False):
        """Seat partners from ``pool`` (a ``PartnerPool`` of this trainer's n_agents and device) before every episode that
        ``train_episode``, ``train_episodes`` (and ``IA2CTrainer.rollout``) start, or stop with ``None``.  Each run draws one
        team per episode (Philox stream 6: key = its training seed, counter word 3 = the episode number) and the team's rows
        overwrite its partner seats' actor rows; nothing else is written, and the episode trains every seat as before.  One
        more launch per episode and no synchronisation.  The partner seats' own updates are thrown away by the next seating:
        after the last seated episode (and after ``set_partners(None)``) a partner seat holds its last partner plus one
        update, from which self-play continues.

        ``per_env=True``: every env draws its own team before every episode (Philox stream 7: key = the run's training seed,
        counter = (env index within its run, episode)) and the rollout kernels play it in that env, so the learning seats
        meet up to E partners per episode.  No launch is added (for N > 8 the pool's policy table is built once, now, and
        kept on the pool).  The partner seats' own actor rows are never used to act in this mode, but they still receive the
        episode's updates, so after ``set_partners(None)`` self-play continues from rows trained on the partners'
        trajectories.  Refused (before any device work) where the rollout has no per-env kernels: the per-step rollout
        (``fused_rollout=False`` or an (N, M) without a fused instantiation up to 8 agents; ``rollout_kernel="step"`` or
        ``belief_kernel="step"`` above), N > 256 and more than one GPU; injected actions are refused when an episode starts."""
        if pool is None:
            self._partners, self._env_partners = None, False
            return
        self._check_partners()
        if not isinstance(pool, PartnerPool):
            raise ValueError(f"set_partners: expected a PartnerPool or None, got {type(pool).__name__}")
        if pool.N != self.N:
            raise ValueError(f"set_partners: the pool is for n_agents={pool.N}, this trainer has {self.N}")
        if pool.device != self.device:
            raise ValueError(f"set_partners: the pool lives on {pool.device}, this trainer on {self.device}")
        if per_env:
            self._check_env_partners()
            e = _lib.EnvPartnerDesc()
            e.rows, e.P, e.seats, e.S = pool.rows.data_ptr(), pool.P, pool.seats.data_ptr(), pool.S
            e.teams, e.Q = pool.teams.data_ptr(), pool.Q
            e.policy = pool.policy_table(self.lib).data_ptr() if self.N > 8 else None
            self._partners, self._env_partners, self._env_partner_desc = pool, True, e
            return
        p = _lib.PartnerDesc()
        p.rows, p.P, p.seats, p.S = pool.rows.data_ptr(), pool.P, pool.seats.data_ptr(), pool.S
        p.teams, p.Q = pool.teams.data_ptr(), pool.Q
        self._partners, self._env_partners, self._partner_desc = pool, False, p

    @property
    def partners(self):
        """The ``PartnerPool`` seated before each episode, or None."""
        return self._partners

    @property
    def partners_per_env(self):
        """True while the pool's partners are drawn per env (``set_partners(pool, per_env=True)``)."""
        return self._env_partners

    def _refuse_env_partners(self, what):
        if self._env_partners:
            raise _lib.IA2CError(f"{what} does not play partners per env: call set_partners(None) first")

    def _play_env_partners(self, call, name):
        """Enqueue one per-env episode: ``call(partner descriptor reference)`` returns the C status; its log slot is taken
        here."""
        if getattr(self, "inj_actions", None) is not None:
            raise _lib.IA2CError(f"{name}: injected actions replace the partners' samples (inject(actions=None) first)")
        R, _ = self._partner_runs()
        if self._env_partner_log is None:
            self._env_partner_log = DeviceRing(self.device, self.ENV_PARTNER_LOG_CAPACITY, (("env_team", np.int32, (R, self.E)),),
                                               ("episode",))
        log, p = self._env_partner_log, self._env_partner_desc
        slot = log.free_slot()
        p.log_env_team = log.ptr["env_team"] + slot * log.row_bytes["env_team"]
        _lib.check(call(C.byref(p)), name)
        log.commit(episode=self.episode)

    def env_partner_history(self):
        """Synchronise and return every per-env episode since the previous call: ``episode`` [n] and ``env_team`` [n, R, E]
        i32 (the team each env played, -1 where a device-side entry was out of range and the env played its own rows;
        ``IA2CTrainer``: [n, E]).  The log is not part of a checkpoint: call this before ``save``."""
        R, runs_ref = self._partner_runs()
        chunks = self._env_partner_log.take_chunks() if self._env_partner_log is not None else []
        ep = np.concatenate([c["episode"] for c in chunks]) if chunks else np.zeros(0, dtype=np.int64)
        team = np.concatenate([c["env_team"] for c in chunks]) if chunks else np.zeros((0, R, self.E), dtype=np.int32)
        return dict(episode=ep, env_team=team[:, 0] if runs_ref is None else team)

    def _refuse_partners(self, what):
        if self._partners is not None:
            raise _lib.IA2CError(f"{what} does not seat partners: call set_partners(None) first")

    def _seat_partners(self, stream):
        """Enqueue the seating of the episode ``self.episode`` on ``stream`` if a pool is set."""
        if self._partners is None:
            return
        R, runs_ref = self._partner_runs()
        if self._partner_log is None:
            self._partner_log = DeviceRing(self.device, self.PARTNER_LOG_CAPACITY, (("team", np.int32, (R,)),), ("episode",))
        log, p = self._partner_log, self._partner_desc
        slot = log.free_slot()
        p.episode, p.log_team = self.episode, log.ptr["team"] + slot * log.row_bytes["team"]
        _lib.check(self.lib.ia2c_seat_partners(C.byref(self.desc), runs_ref, C.byref(p), stream), "ia2c_seat_partners")
        log.commit(episode=self.episode)

    def partner_history(self):
        """Synchronise and return every seated episode since the previous call: ``episode`` [n] and ``team`` [n, R] i32 (the
        team each run played, -1 where a device-side entry was out of range; ``IA2CTrainer``: [n]).  The log is not part of a
        checkpoint: call this before ``save``."""
        R, runs_ref = self._partner_runs()
        chunks = self._partner_log.take_chunks() if self._partner_log is not None else []
        ep = np.concatenate([c["episode"] for c in chunks]) if chunks else np.zeros(0, dtype=np.int64)
        team = np.concatenate([c["team"] for c in chunks]) if chunks else np.zeros((0, R), dtype=np.int32)
        return dict(episode=ep, team=team[:, 0] if runs_ref is None else team)

    def _partner_state(self, sd):
        if self._partners is not None:
            sd["partners"] = self._partners.state()
            sd["partners_per_env"] = self._env_partners
        return sd

    def _load_partner_state(self, sd):
        """Restore the pool and mode a checkpoint carries (a checkpoint without the mode is per-episode), or clear the pool
        for one without."""
        part = sd.get("partners")
        self.set_partners(PartnerPool(part["rows"], part["teams"], part["seats"], self.N, device=self.device)
                          if part is not None else None, per_env=bool(sd.get("partners_per_env", False)))
