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

``set_partners(pool, per_env=True, prioritized=True)`` weights those draws (prioritized fictitious self-play): after every
episode one more launch adds each env's return to its run's statistics for the team it played (``ia2c_record_partner_returns``),
and ``prioritize_partners`` rebuilds every run's weight table from them in one launch (``ia2c_prioritize_partners``), giving
the teams a run does worst with the largest weights.  ``partner_returns`` and ``partner_weights`` read both back.

``freeze_seats(seats)`` freezes seats of every run (``ia2c_train_episode_frozen``): a frozen seat still acts, with its own
actor row, a seated pool row or its env's pool row, but nothing of it is updated and the update kernels skip it.
``freeze_seats(pool.seats)`` trains against truly frozen partners in every partner mode; without a pool it trains a best
response to fixed co-players.
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
    _priority = None            # prioritized per-env mode: {"count", "sum", "table"} device tensors and "desc"
    _frozen = frozenset()       # frozen seats
    _frozen_desc = None

    def _check_partners(self):
        """Raise, before any device work, where partners cannot be seated."""

    def _check_env_partners(self):
        """Raise, before any device work, where partners cannot be played per env."""

    def _check_frozen(self):
        """Raise, before any device work, where seats cannot be frozen."""

    def freeze_seats(self, seats):
        """Freeze ``seats`` (seat indices in [0, n_agents), the same for every run; at least one frozen and one trained) in
        every episode that ``train_episode`` and ``train_episodes`` start, or train every seat again with ``None``.  A frozen
        seat acts as before (its own actor row, the row a pool seats in it, or its env's pool row in the per-env mode), but
        its parameters, gradients, Adam moments and steps and actor gradient sum stay byte for byte as they are, its
        ``loss_out`` entries are NaN, and the gradient and reduce kernels do not run its rows.  Up to 8 agents the fused
        rollout still runs every seat's belief filter; from 9 agents the belief kernel skips frozen seats, whose belief
        records stay as they are and whose partner predictions read 0xFF ("no prediction", so ``history()`` counts no hit).
        A trained seat's every byte is what the episode computes with nothing frozen, and run r of a batch equals a
        standalone trainer with its seed, pool, partner mode and frozen set.  Launches per episode are unchanged.  Refused,
        before any device work, off the whole-episode kernel paths (see ``_check_frozen``); ``rollout`` / ``update``, the
        host-tape pipelines and ``train_episode_timed`` refuse to run while seats are frozen."""
        if seats is None:
            self._frozen, self._frozen_desc = frozenset(), None
            return
        fs = self._frozen_set(seats)
        f = _lib.FrozenSeats()
        for x in fs:
            f.mask[x >> 6] |= 1 << (x & 63)
        self._frozen, self._frozen_desc = fs, f

    def _frozen_set(self, seats):
        """``seats`` (a set, sequence, array or tensor of seat indices, e.g. ``pool.seats``) as a frozenset, after every check
        of ``freeze_seats``; raises before any device work."""
        if isinstance(seats, (int, np.integer)):
            raise ValueError("freeze_seats: pass a set of seats, e.g. freeze_seats({1})")
        if not isinstance(seats, (torch.Tensor, np.ndarray)):
            seats = np.asarray(list(seats), dtype=np.int64)
        fs = frozenset(int(x) for x in _host_ints(seats, "seats").reshape(-1))
        if any(not 0 <= x < self.N for x in fs):
            raise ValueError(f"freeze_seats: seats {sorted(fs)} outside [0, {self.N})")
        if not 1 <= len(fs) <= self.N - 1:
            raise ValueError(f"freeze_seats: {len(fs)} of {self.N} seats: at least one seat must be frozen and one trained")
        self._check_frozen()
        return fs

    def _check_frozen_state(self, sd):
        """Raise, before a checkpoint's tensors are copied, if its frozen seats cannot be frozen here."""
        if sd.get("frozen_seats"):
            self._frozen_set(sd["frozen_seats"])

    @property
    def frozen_seats(self):
        """The frozen seats (a frozenset, empty while every seat trains)."""
        return self._frozen

    def _refuse_frozen(self, what):
        if self._frozen:
            raise _lib.IA2CError(f"{what} does not freeze seats: call freeze_seats(None) first")

    def _enqueue_frozen(self, desc_ref, runs_ref, stream):
        """Enqueue one training episode with the frozen seats, in the partner mode that is set."""
        f, name = C.byref(self._frozen_desc), "ia2c_train_episode_frozen"
        if self._env_partners:
            self._play_env_partners(lambda p: self.lib.ia2c_train_episode_frozen(desc_ref, runs_ref, p, None, f, stream), name,
                                    lambda p, w: self.lib.ia2c_train_episode_frozen(desc_ref, runs_ref, p, w, f, stream),
                                    desc_ref, stream)
            return
        self._seat_partners(stream)
        _lib.check(self.lib.ia2c_train_episode_frozen(desc_ref, runs_ref, None, None, f, stream), name)

    def set_partners(self, pool, per_env=False, prioritized=False):
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
        ``belief_kernel="step"`` above), N > 256 and more than one GPU; injected actions are refused when an episode starts.

        ``prioritized=True`` (with ``per_env=True`` only): each run draws its envs' teams with the weights of its own table
        (include/ia2c_b200.h, ia2c_partner_priority_desc, states the definitions), equal until the first
        ``prioritize_partners``, so until then the episodes are byte for byte those of the uniform mode.  Every episode adds one
        launch that records each env's return for the team it played; nothing synchronises.  Every ``set_partners`` call
        starts from zeroed statistics and equal weights, and ``set_partners(None)`` drops them."""
        if prioritized and not per_env:
            raise ValueError("set_partners: prioritized=True draws per env: pass per_env=True")
        if pool is None:
            self._partners, self._env_partners, self._priority = None, False, None
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
            R, _ = self._partner_runs()
            if prioritized and R * pool.Q > _lib.PARTNER_PRIORITY_MAX_CELLS:
                raise ValueError(f"set_partners: runs * teams = {R * pool.Q} above PARTNER_PRIORITY_MAX_CELLS "
                                 f"({_lib.PARTNER_PRIORITY_MAX_CELLS})")
            e = _lib.EnvPartnerDesc()
            e.rows, e.P, e.seats, e.S = pool.rows.data_ptr(), pool.P, pool.seats.data_ptr(), pool.S
            e.teams, e.Q = pool.teams.data_ptr(), pool.Q
            e.policy = pool.policy_table(self.lib).data_ptr() if self.N > 8 else None
            self._partners, self._env_partners, self._env_partner_desc = pool, True, e
            self._priority = self._new_priority(R, pool.Q) if prioritized else None
            return
        p = _lib.PartnerDesc()
        p.rows, p.P, p.seats, p.S = pool.rows.data_ptr(), pool.P, pool.seats.data_ptr(), pool.S
        p.teams, p.Q = pool.teams.data_ptr(), pool.Q
        self._partners, self._env_partners, self._partner_desc, self._priority = pool, False, p, None

    def _new_priority(self, R, Q):
        """Zeroed statistics and equal weights (C_q = q * 2^24) for R runs of Q teams, on the device."""
        with torch.cuda.device(self.device):
            pr = dict(count=torch.zeros((R, Q), dtype=torch.int64, device=self.device),
                      sum=torch.zeros((R, Q), dtype=torch.int64, device=self.device),
                      table=(torch.arange(Q + 1, dtype=torch.int64, device=self.device) << 24).repeat(R, 1))
        w = _lib.PartnerPriorityDesc()
        w.count, w.sum, w.table, w.R, w.Q = pr["count"].data_ptr(), pr["sum"].data_ptr(), pr["table"].data_ptr(), R, Q
        pr["desc"] = w
        return pr

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

    @property
    def partners_prioritized(self):
        """True while the per-env draws are weighted (``set_partners(pool, per_env=True, prioritized=True)``)."""
        return self._priority is not None

    def _play_env_partners(self, call, name, call_prioritized=None, desc_ref=None, stream=None):
        """Enqueue one per-env episode: ``call(partner descriptor reference)`` returns the C status; its log slot is taken
        here.  In the prioritized mode ``call_prioritized(partner descriptor reference, priority descriptor reference)`` runs
        the episode instead, followed by the record of its returns (``desc_ref``: the episode descriptor, on ``stream``)."""
        if getattr(self, "inj_actions", None) is not None:
            raise _lib.IA2CError(f"{name}: injected actions replace the partners' samples (inject(actions=None) first)")
        R, _ = self._partner_runs()
        if self._env_partner_log is None:
            self._env_partner_log = DeviceRing(self.device, self.ENV_PARTNER_LOG_CAPACITY, (("env_team", np.int32, (R, self.E)),),
                                               ("episode",))
        log, p = self._env_partner_log, self._env_partner_desc
        slot = log.free_slot()
        p.log_env_team = log.ptr["env_team"] + slot * log.row_bytes["env_team"]
        if self._priority is None:
            _lib.check(call(C.byref(p)), name)
        else:
            w = C.byref(self._priority["desc"])
            _lib.check(call_prioritized(C.byref(p), w), name + "_prioritized")
            _lib.check(self.lib.ia2c_record_partner_returns(desc_ref, p.log_env_team, w, stream), "ia2c_record_partner_returns")
        log.commit(episode=self.episode)

    def _require_priority(self, what):
        if self._priority is None:
            raise _lib.IA2CError(f"{what}: partners are not drawn with priorities (set_partners(pool, per_env=True, prioritized=True))")

    def prioritize_partners(self, power=2, floor=0.1, reset=True):
        """Rebuild every run's weight table from its statistics, in one launch and without synchronising: the team with the
        lowest mean return gets weight 1, the one with the highest gets ``floor``, and in between w = floor + (1 - floor) *
        x ** power, x = (best mean - mean) / (best mean - worst mean); a team never played gets 1, so it is tried.  ``reset``
        zeroes the statistics in the same launch, so that the next call weighs only the episodes after this one."""
        self._require_priority("prioritize_partners")
        if isinstance(power, bool) or not isinstance(power, (int, np.integer)) or not 0 <= power <= 16:
            raise ValueError(f"prioritize_partners: power={power!r} must be an integer in [0, 16]")
        floor = float(floor)
        if not 0.0 <= floor <= 1.0:
            raise ValueError(f"prioritize_partners: floor={floor} outside [0, 1]")
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ia2c_prioritize_partners(C.byref(self._priority["desc"]), int(power), floor, int(bool(reset)),
                                                         torch.cuda.current_stream(self.device).cuda_stream),
                       "ia2c_prioritize_partners")

    def _run_axis(self, a):
        return a[0] if self._partner_runs()[1] is None else a

    def partner_returns(self):
        """Synchronise and return the statistics since the last reset: ``count`` [R, Q] i64 (episodes' envs that played team
        q) and ``mean`` [R, Q] f64 (their mean return, as the fixed-point sums give it; NaN where count is 0).
        ``IA2CTrainer``: [Q]."""
        self._require_priority("partner_returns")
        with torch.cuda.device(self.device):
            count, total = self._priority["count"].cpu().numpy(), self._priority["sum"].cpu().numpy()
        with np.errstate(invalid="ignore", divide="ignore"):
            mean = np.where(count > 0, total.astype(np.float64) * 2.0 ** -20 / count, np.nan)
        return dict(count=self._run_axis(count), mean=self._run_axis(mean))

    def partner_weights(self):
        """Synchronise and return every run's team weights W [R, Q] i64 (2^24 is weight 1; ``IA2CTrainer``: [Q])."""
        self._require_priority("partner_weights")
        with torch.cuda.device(self.device):
            table = self._priority["table"].cpu().numpy()
        return self._run_axis(np.diff(table, axis=1))

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

    def _partner_state(self, sd, run=None):
        """Add the pool, the mode and the prioritized statistics and table (all runs', or run ``run``'s alone) and the frozen
        seats to ``sd``."""
        if self._frozen:
            sd["frozen_seats"] = sorted(self._frozen)
        if self._partners is not None:
            sd["partners"] = self._partners.state()
            sd["partners_per_env"] = self._env_partners
            if self._priority is not None:
                rows = slice(None) if run is None else slice(run, run + 1)
                sd["partner_priority"] = {k: self._priority[k][rows].detach().cpu().clone() for k in ("count", "sum", "table")}
        return sd

    def _load_partner_state(self, sd):
        """Restore the pool, mode and prioritized statistics a checkpoint carries (a checkpoint without the mode is
        per-episode, one without statistics is uniform), or clear the pool for one without; then the frozen seats (none
        for a checkpoint without them)."""
        part = sd.get("partners")
        prio = sd.get("partner_priority") if part is not None else None
        if prio is not None:
            R, Q = self._partner_runs()[0], int(part["teams"].shape[0])
            for k, shape in (("count", (R, Q)), ("sum", (R, Q)), ("table", (R, Q + 1))):
                if tuple(prio[k].shape) != shape:
                    raise ValueError(f"checkpoint partner_priority[{k!r}] has shape {tuple(prio[k].shape)}, expected {shape}")
        self.set_partners(PartnerPool(part["rows"], part["teams"], part["seats"], self.N, device=self.device)
                          if part is not None else None, per_env=bool(sd.get("partners_per_env", False)),
                          **({"prioritized": True} if prio is not None else {}))
        if prio is not None:
            for k in ("count", "sum", "table"):
                self._priority[k].copy_(prio[k])
        self.freeze_seats(sd.get("frozen_seats"))
