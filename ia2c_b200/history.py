"""Learning curves recorded on the GPU (``ia2c_record_episode``, include/ia2c_b200.h).

``train_episodes(n)`` of ``IA2CTrainer`` (one GPU), ``IA2CRuns`` and ``IA2CRunsMany`` trains n episodes exactly as n calls of
``train_episode()`` do, and after each one enqueues one more launch that reduces the episode's trajectory into a slot of a
device ring: every run's return sum, its agents' critic and actor losses, action counts and partner-prediction hits (how
often the belief filter's predicted partner action, the critic's ``ja`` input, equals the partner's true action).  Nothing
is read back per episode: the host synchronises only when the ring is full, and then drains it with one device-to-host copy.
``history()`` drains what is left and returns everything recorded since the previous ``history()`` call.

The ring holds ``HISTORY_CAPACITY`` slots (a class attribute; set it on the instance before the first ``train_episodes`` to
change it).  Each call clears the slot after its own for the next one, so the ring holds at most ``HISTORY_CAPACITY - 1``
episodes that have not been drained.  Episodes of ``train_episodes`` do not enter the ``read_stats`` windows, and the
history is not part of a checkpoint: call ``history()`` before ``save``.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib


class DeviceRing:
    """``capacity`` slots of fixed-size device rows, one array per field, carved in order from one zeroed device buffer, so
    that a drain is one copy of the byte span that holds the slots to read (the whole buffer when the range wraps).
    ``fields``: (name, numpy dtype, row shape) per array, field k at ``ptr[name]`` as ``dtype[capacity, *shape]``;
    ``tags``: names of host-side integers kept per slot (the episode number of a record, ...).

    A writer takes ``free_slot()``, enqueues its launch on that slot and then ``commit(**tags)``.  At most ``capacity - 1``
    records wait undrained (a history record clears the slot after its own): ``free_slot`` drains, which synchronises the
    device's current stream, when that many are pending."""

    def __init__(self, device, capacity, fields, tags):
        cap = int(capacity)
        if cap < 2:
            raise ValueError(f"capacity={capacity} must be >= 2")
        self.device, self.capacity = device, cap
        self._fields = tuple((name, np.dtype(dt), tuple(shape)) for name, dt, shape in fields)
        self._row = tuple(int(np.prod(shape, dtype=np.int64)) * dt.itemsize for _, dt, shape in self._fields)   # bytes per slot
        self._off = tuple(int(x) for x in np.concatenate([[0], np.cumsum([cap * b for b in self._row])]))
        self._dev = torch.zeros(self._off[-1], dtype=torch.uint8, device=device)
        self._host = torch.empty(self._off[-1], dtype=torch.uint8).pin_memory()
        base = self._dev.data_ptr()
        self.ptr = {name: base + o for (name, _, _), o in zip(self._fields, self._off)}
        self.row_bytes = {name: b for (name, _, _), b in zip(self._fields, self._row)}
        self._tags = tuple(tags)
        self._tag_of_slot = np.zeros((len(self._tags), cap), dtype=np.int64)
        self.head = self.tail = 0                       # records enqueued / drained since the ring was made
        self._chunks = []

    def free_slot(self):
        """The slot of the next record (draining first if capacity - 1 records are pending)."""
        if self.head - self.tail >= self.capacity - 1:
            self.drain()
        return self.head % self.capacity

    def commit(self, **tags):
        """Count the record just enqueued on ``free_slot()`` and keep its tags."""
        slot = self.head % self.capacity
        for i, k in enumerate(self._tags):
            self._tag_of_slot[i, slot] = tags[k]
        self.head += 1

    def drain(self):
        """Synchronise the device's current stream and move the pending slots to host arrays."""
        n = self.head - self.tail
        if n == 0:
            return
        cap, first = self.capacity, self.tail % self.capacity
        lo, hi = 0, self._off[-1]
        if first + n <= cap:   # one contiguous run of slots: from its row of the first field to its row of the last one
            lo, hi = self._off[0] + first * self._row[0], self._off[-2] + (first + n) * self._row[-1]
        with torch.cuda.device(self.device):
            self._host[lo:hi].copy_(self._dev[lo:hi], non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
        slots = (first + np.arange(n)) % cap
        buf = self._host.numpy()
        chunk = {k: self._tag_of_slot[i, slots] for i, k in enumerate(self._tags)}
        for (name, dt, shape), o0, o1 in zip(self._fields, self._off[:-1], self._off[1:]):
            chunk[name] = buf[o0:o1].view(dt).reshape(cap, *shape)[slots]
        self._chunks.append(chunk)
        self.tail = self.head

    def take_chunks(self):
        """Drain, then return and forget every chunk drained so far (a list of dicts of tag and field arrays)."""
        self.drain()
        chunks, self._chunks = self._chunks, []
        return chunks


class EpisodeHistory(DeviceRing):
    """The device ring of one trainer or batch (runs R, N agents, E envs per run, T steps): the four arrays of
    ``ia2c_history_desc``, and the drained host rows."""

    def __init__(self, lib, device, runs, N, E, T, capacity):
        if int(capacity) < 2:
            raise ValueError(f"HISTORY_CAPACITY={capacity} must be >= 2")
        R, RN = int(runs), int(runs) * int(N)
        super().__init__(device, capacity, (("return_sum", np.float64, (R,)), ("loss", np.float32, (2, RN)),
                                            ("action_counts", np.uint32, (RN, 3)), ("partner_hits", np.uint32, (RN,))),
                         ("episode",))
        self.lib, self.R, self.N, self.E, self.T = lib, R, int(N), int(E), int(T)
        h = self.desc = _lib.HistoryDesc()
        h.capacity = self.capacity
        h.return_sum, h.loss, h.action_counts, h.partner_hits = (self.ptr[k] for k in
                                                                 ("return_sum", "loss", "action_counts", "partner_hits"))
        self._href = C.byref(h)

    def record(self, desc_ref, episode, stream):
        """Enqueue the record of the episode ``desc_ref`` just ran (``episode`` is its number) on ``stream``."""
        slot = self.free_slot()
        _lib.check(self.lib.ia2c_record_episode(desc_ref, self.R, self._href, slot, stream), "ia2c_record_episode")
        self.commit(episode=episode)

    def take(self):
        """Drain, then return and forget every row drained so far (see ``history_arrays``)."""
        return history_arrays(self.take_chunks(), self.R, self.N, self.E, self.T)


def history_arrays(chunks, R, N, E, T):
    """The user-facing arrays of drained rows, episode axis first: episode [n]; return_sum and mean_return (= return_sum / E)
    [n, R]; critic_loss and actor_loss [n, R, N]; action_counts [n, R, N, 3] and action_freq (= counts / (T * E));
    partner_accuracy (= hits / (T * E)) [n, R, N]."""
    def cat(k, dtype, shape):
        parts = [c[k] for c in chunks]
        return np.concatenate(parts) if parts else np.zeros((0,) + shape, dtype=dtype)

    ep = cat("episode", np.int64, ())
    n = ep.shape[0]
    ret = cat("return_sum", np.float64, (R,))
    loss = cat("loss", np.float32, (2, R * N)).reshape(n, 2, R, N)
    counts = cat("action_counts", np.uint32, (R * N, 3)).reshape(n, R, N, 3)
    hits = cat("partner_hits", np.uint32, (R * N,)).reshape(n, R, N)
    steps = float(T * E)
    return dict(episode=ep, return_sum=ret, mean_return=ret / E, critic_loss=loss[:, 0], actor_loss=loss[:, 1],
                action_counts=counts, action_freq=counts / steps, partner_accuracy=hits / steps)


class RecordsHistory:
    """``train_episodes`` / ``history`` for a class that defines ``_history_dims()`` -> (runs, N, E, T, drop_run_axis) and
    ``_enqueue_episode(desc_ref, stream)``, the C call of one training episode with ``self.desc``."""

    HISTORY_CAPACITY = 64   # slots of the device ring of recorded episodes (allocated on first use)
    _history = None

    def _check_history(self):
        """Raise, before any device work, where recording is not supported."""

    def train_episodes(self, n):
        """Train ``n`` episodes, each exactly as ``train_episode()`` trains it, and record each one's statistics on the
        device (one more launch per episode).  Asynchronous: the host synchronises only when the ring is full.  The
        episodes do not enter the ``read_stats`` windows; ``history()`` returns their statistics."""
        n = int(n)
        if n < 0:
            raise ValueError(f"train_episodes: n={n} must be >= 0")
        self._check_history()
        runs, N, E, T, _ = self._history_dims()
        if self._history is None:
            self._history = EpisodeHistory(self.lib, self.device, runs, N, E, T, self.HISTORY_CAPACITY)
        ring, dref = self._history, C.byref(self.desc)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            for _ in range(n):
                self.desc.episode = self.episode
                self._enqueue_episode(dref, stream)
                ring.record(dref, self.episode, stream)
                self.episode += 1

    def history(self):
        """Synchronise and return the statistics of every episode recorded by ``train_episodes`` since the previous
        ``history()`` call, as numpy arrays with the episode axis first: ``episode`` (the episode number), ``return_sum``
        (the fp64 sum of the run's E returns, in the fixed order of include/ia2c_b200.h) and ``mean_return`` [n, R];
        ``critic_loss`` and ``actor_loss`` [n, R, N]; ``action_counts`` [n, R, N, 3] and ``action_freq`` (counts over
        T * E); ``partner_accuracy`` [n, R, N], the share of the T * E (step, env) pairs where the belief-predicted partner
        action equals the true one.  ``IA2CTrainer`` returns the same arrays without the run axis."""
        runs, N, E, T, drop = self._history_dims()
        out = self._history.take() if self._history is not None else history_arrays([], runs, N, E, T)
        if drop:
            out = {k: (v if k == "episode" else v[:, 0]) for k, v in out.items()}
        return out
