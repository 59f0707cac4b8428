"""IA2CTrainer — the whole episode of ia2c.py (rollout + critic phase + actor phase) on the GPU.

Reference path covered (thinclab/IA2C): the body of the episode loop, ia2c.py:62-131, with its
hyper-parameters (ia2c.py:25-31,40,43-46), for E batched Org instances and N agents
(N=2 is the reference; N>2 is the builder-defined "Org-N" extension, DESIGN.md).

Everything numeric is a kernel of libia2c_b200.so driven through ``ia2c_episode_desc``; this class
only owns the device buffers (torch tensors), the optional replay tapes, the multi-GPU all-reduce
(torch.distributed / NCCL, one per optimiser phase) and the loss windows / return statistics that
ia2c.py prints (ia2c.py:131-134; ac_nets.py:77-80,124-127).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .history import RecordsHistory
from .nets import hidden_size
from .partners import SeatsPartners
from .sharding import shard_envs

N_FEATURES, N_ACTIONS, N_JOINT = 6, 3, 9


def reference_init(n_agents, n_models, seed=None):
    """Initial parameters drawn the way ia2c.py:47-50,61 draws them: critics 1..N then actors 1..N
    (nn.Linear default init from torch's CPU generator), then one random model matrix per agent from
    numpy's global generator.  Returns (actor [N,105], critic [N,147], filter_action [N,M,3])."""
    if seed is not None:
        torch.manual_seed(seed)
        np.random.seed(seed)

    def net(out):
        ls = (nn.Linear(N_FEATURES, hidden_size), nn.Linear(hidden_size, hidden_size), nn.Linear(hidden_size, out))
        return torch.cat([t.detach().reshape(-1) for l in ls for t in (l.weight, l.bias)]).numpy()

    critic = np.stack([net(N_JOINT) for _ in range(n_agents)])
    actor = np.stack([net(N_ACTIONS) for _ in range(n_agents)])
    fa = []
    for _ in range(n_agents):
        m = np.random.rand(n_models, N_ACTIONS)
        m /= np.sum(m, axis=1)[:, np.newaxis]
        fa.append(m)
    return actor, critic, np.stack(fa)


class IA2CTrainer(SeatsPartners, RecordsHistory):
    def __init__(self, num_envs, n_agents=2, n_models=5, steps_per_episode=30, max_episode_steps=30,
                 lr_critic=0.0002, lr_actor=0.0001, beta=0.001, gamma=0.9, seed=0, device=None,
                 rank=0, world_size=1, process_group=None, dumps=False, fused_rollout=None, fused_critic=None,
                 init=None, comm="auto", actor_kernel="auto", belief_kernel="auto", rollout_kernel="auto"):
        _lib.require_cuda()
        if actor_kernel not in ("auto", "pipe", "columns"):
            raise ValueError("actor_kernel must be 'auto', 'pipe' or 'columns'")
        if actor_kernel == "auto":   # measured (tools/time_kernels.py): columns 22.6 vs pipe 26.5 us at 4096 x 2;
            actor_kernel = "pipe" if int(n_agents) > 64 else "columns"   # equal at 1024 x 64; pipe 395 vs 479 us at 1024 x 256
        self.lib = _lib.load()
        self.rank, self.world = int(rank), int(world_size)
        self.pg = process_group
        self.E_total = int(num_envs)
        self.env_offset, self.E = shard_envs(self.E_total, self.rank, self.world)
        self.N, self.M, self.T = int(n_agents), int(n_models), int(steps_per_episode)
        self.K = self.N - 1
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.episode = 0
        self.seed = int(seed)
        dev, E, N, K, M, T = self.device, self.E, self.N, self.K, self.M, self.T

        def z(shape, dtype):
            return torch.zeros(shape, dtype=dtype, device=dev)

        f32, f64, u8, i32 = torch.float32, torch.float64, torch.uint8, torch.int32
        self.actor_params, self.critic_params = z((N, _lib.ACTOR_P), f32), z((N, _lib.CRITIC_P), f32)
        self.actor_grad, self.critic_grad = z((N, _lib.ACTOR_P + 1), f32), z((N, _lib.CRITIC_P + 1), f32)
        self.actor_grad_accum = z((N, _lib.ACTOR_P), f32)
        self.actor_m, self.actor_v = z((N, _lib.ACTOR_P), f32), z((N, _lib.ACTOR_P), f32)
        self.critic_m, self.critic_v = z((N, _lib.CRITIC_P), f32), z((N, _lib.CRITIC_P), f32)
        self.actor_step, self.critic_step = z((N,), i32), z((N,), i32)
        # losses and episode returns share one "result region" so that one D2H copy returns both
        self._off_ret = (2 * N * 4 + 7) & ~7
        self._result_region = z((self._off_ret + E * 8,), u8)
        self.loss_out = self._result_region[:2 * N * 4].view(f32).view(2, N)
        self.filter_action = z((N, M, N_ACTIONS), f64)
        self.env_state, self.env_hist = z((E,), i32), z((E,), f64)
        self.env_cls, self.env_elapsed = z((E, 2), u8), z((E,), i32)
        self.ep_return = self._result_region[self._off_ret:].view(f64)
        self.obs, self.reward = z((T + 1, E, N_FEATURES), f32), z((T, E), f32)
        self.act, self.partner_true, self.partner_pred = z((T + 1, E, N), u8), z((T + 1, E, N), u8), z((T + 1, E, N), u8)
        self.belief_records = z((E, N, K, _lib.BELIEF_RECORD), u8)
        self.inj_actions = self.inj_u_action = self.inj_u_belief = None
        self.dumps = bool(dumps)
        if dumps:
            self.state_trace, self.reward_f64 = z((T, E), i32), z((T, E), f64)
            self.pred_dump, self.belief_dump = z((T + 1, E, N, K), u8), z((T + 1, E, N, K, M), u8)
            self.adv_dump, self.target_dump = z((N, T, E), f32), z((N, T, E), f32)
        self.desc = _lib.EpisodeDesc()
        d = self.desc
        d.E, d.E_total, d.env_offset = E, self.E_total, self.env_offset
        d.N, d.T, d.M, d.max_episode_steps = N, T, M, int(max_episode_steps or 0)
        d.gamma, d.beta, d.lr_actor, d.lr_critic = gamma, beta, lr_actor, lr_critic
        d.seed, d.episode = self.seed, 0
        if fused_rollout is None:   # the persistent one-launch rollout wherever it has an instantiation
            fused_rollout = bool(self.lib.ia2c_rollout_fused_supported(N, M))
        if fused_critic is None:
            fused_critic = bool(fused_rollout)   # the critic-gradient stage rides along with the fused rollout
        if belief_kernel not in ("auto", "episode", "step"):
            raise ValueError("belief_kernel must be 'auto', 'episode' or 'step'")
        # many modelled others (N > 8 path): "auto" / "episode" carry every belief record through the whole episode in ONE
        # kernel where the library supports it (N >= 33, N % 4 == 0), "step" streams the records once per step (A/B, parity)
        d.flags = ((_lib.FLAG_FUSED_ROLLOUT if fused_rollout else 0) | (_lib.FLAG_SKIP_ADAM if self.world > 1 else 0) |
                   (_lib.FLAG_BELIEF_PER_STEP if belief_kernel == "step" else 0) |
                   (_lib.FLAG_ROLLOUT_PER_STEP if rollout_kernel == "step" else 0) |   # N > 8: per-step env / actor kernels (A/B, parity)
                   (_lib.FLAG_FUSED_CRITIC if (fused_rollout and fused_critic) else 0) |
                   (_lib.FLAG_ACTOR_COLUMNS if actor_kernel == "columns" else 0))
        for name in ("actor_params", "actor_grad", "actor_grad_accum", "actor_m", "actor_v", "critic_params",
                     "critic_grad", "critic_m", "critic_v", "actor_step", "critic_step", "loss_out", "filter_action",
                     "env_state", "env_hist", "env_cls", "env_elapsed", "ep_return", "obs", "reward", "act",
                     "partner_true", "partner_pred", "belief_records"):
            setattr(d, name, getattr(self, name).data_ptr())
        if dumps:
            for name in ("state_trace", "reward_f64", "pred_dump", "belief_dump", "adv_dump", "target_dump"):
                setattr(d, name, getattr(self, name).data_ptr())
        n_part = int(self.lib.ia2c_episode_partials_floats(C.byref(d)))
        self.partials = z((n_part,), f32)
        d.partials, d.partials_floats = self.partials.data_ptr(), n_part
        # host-side bookkeeping the reference prints (ia2c.py:131-134)
        self.critic_losses, self.actor_losses, self.reward_lst = [], [], []
        self._h_loss = torch.zeros(2, N, dtype=f32).pin_memory()
        self._h_return = torch.zeros(E, dtype=f64).pin_memory()
        if init is None:
            init = reference_init(N, M)
        self.load_init(*init)
        self.comm = "none"
        if self.world > 1:
            self._setup_comm(comm)

    # ------------------------------------------------------------------ multi-GPU exchange
    def _setup_comm(self, comm):
        """comm="p2p": fused all-reduce + Adam kernel over NVLink peer memory (torch symmetric memory provides the
        peer mappings, the exchange itself is ia2c_allreduce_adam; "p2p-multicast" / "p2p-unicast" force the NVSwitch
        multicast store or the per-peer stores); comm="nccl": reduce -> NCCL all-reduce -> Adam.  "auto" tries p2p and
        falls back to NCCL if symmetric memory cannot be set up — the decision is COLLECTIVE (all ranks or none)."""
        import os

        import torch.distributed as dist

        if comm not in ("auto", "p2p", "p2p-unicast", "p2p-multicast", "nccl"):
            raise ValueError(f"unknown comm mode {comm!r}")
        ok, mc_ptr, err = 0, 0, None
        if comm != "nccl" and self.world <= 8:
            try:
                import torch.distributed._symmetric_memory as symm

                group = self.pg if self.pg is not None else dist.group.WORLD
                n_words = int(self.lib.ia2c_peer_inbox_bytes(C.byref(self.desc), self.world)) // 8
                self._inbox = symm.empty(n_words, dtype=torch.int64, device=self.device)
                self._comm_error = symm.empty(2, dtype=torch.int32, device=self.device)
                self._inbox.zero_()
                self._comm_error.zero_()
                h_in = symm.rendezvous(self._inbox, group)
                h_err = symm.rendezvous(self._comm_error, group)
                self._symm_handles = (h_in, h_err)
                mc_ptr = int(getattr(h_in, "multicast_ptr", 0) or 0)
                ok = 1
            except Exception as exc:  # symmetric memory unavailable on this rank
                err = exc
        want_mc = comm == "p2p-multicast" or (comm in ("auto", "p2p") and os.environ.get("IA2C_P2P_MULTICAST", "0") == "1")
        flags = torch.tensor([ok, 1 if (mc_ptr and want_mc) else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(flags, op=dist.ReduceOp.MIN, group=self.pg)   # every rank takes the same path
        all_ok, all_mc = (int(x) for x in flags.tolist())
        if comm == "p2p-multicast" and all_ok and not all_mc:
            raise _lib.IA2CError("comm='p2p-multicast' requested but the symmetric buffer has no multicast mapping on every rank")
        if not all_ok:
            if comm != "auto" and comm != "nccl":
                raise _lib.IA2CError(f"comm={comm!r} requested but symmetric memory setup failed on some rank"
                                     + (f" (this rank: {err})" if err else ""))
            self.comm = "nccl"
            return
        h_in, h_err = self._symm_handles
        self.peers = _lib.PeerDesc()
        self.peers.rank, self.peers.world = self.rank, self.world
        for p in range(self.world):
            self.peers.inbox[p] = int(h_in.buffer_ptrs[p])
            self.peers.error[p] = int(h_err.buffer_ptrs[p])
        self.peers.mc_inbox = mc_ptr if all_mc else None
        self.peers.timeout_us = int(os.environ.get("IA2C_P2P_TIMEOUT_US", "0"))
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.pg)      # every rank's inbox is zero (epoch 0) before anyone pushes a word
        self.comm = "p2p-multicast" if all_mc else "p2p"
        self._epoch = 0
        self.desc.flags |= _lib.FLAG_GRAD_ONLY

    @property
    def p2p(self):
        return self.comm.startswith("p2p")

    # ------------------------------------------------------------------ parameters
    def load_init(self, actor, critic, filter_action):
        self.actor_params.copy_(torch.as_tensor(np.asarray(actor), dtype=torch.float32))
        self.critic_params.copy_(torch.as_tensor(np.asarray(critic), dtype=torch.float32))
        self.filter_action.copy_(torch.as_tensor(np.asarray(filter_action), dtype=torch.float64))

    # ------------------------------------------------------------------ injected randomness
    def inject(self, actions=None, u_action=None, u_belief=None):
        """Replay tapes for the NEXT episodes (kept until changed): ``actions`` uint8[T+1,E,N] (the
        reference's sampled actions), ``u_action`` float32[T+1,E,N] (uniforms for the inverse-CDF sampler),
        ``u_belief`` float64[T+1,E,N,K] (the belief filter's ``np.random.rand`` draws).  None -> Philox."""
        T, E, N, K, dev = self.T, self.E, self.N, self.K, self.device

        def put(x, dtype, shape):
            if x is None:
                return None
            t = torch.as_tensor(np.asarray(x) if not isinstance(x, torch.Tensor) else x).to(dev, dtype).contiguous()
            assert tuple(t.shape) == shape, (tuple(t.shape), shape)
            return t

        self.inj_actions = put(actions, torch.uint8, (T + 1, E, N))
        if u_action is not None and u_belief is not None:   # both tapes: keep them in staging region A (one region)
            self._ensure_stage()
            self.inj_u_action.copy_(put(u_action, torch.float32, (T + 1, E, N)))
            self.inj_u_belief.copy_(put(u_belief, torch.float64, (T + 1, E, N, K)))
        else:
            self.inj_u_action = put(u_action, torch.float32, (T + 1, E, N))
            self.inj_u_belief = put(u_belief, torch.float64, (T + 1, E, N, K))
        self.desc.inj_actions = self.inj_actions.data_ptr() if self.inj_actions is not None else None
        self.desc.inj_u_action = self.inj_u_action.data_ptr() if self.inj_u_action is not None else None
        self.desc.inj_u_belief = self.inj_u_belief.data_ptr() if self.inj_u_belief is not None else None

    # ------------------------------------------------------------------ one episode
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def rollout(self):
        self.desc.episode = self.episode
        with torch.cuda.device(self.device):
            s = self._stream()
            if self._env_partners:
                self._play_env_partners(lambda p: self.lib.ia2c_rollout_env_partners(C.byref(self.desc), p, s), "ia2c_rollout_env_partners")
                return
            self._seat_partners(s)
            _lib.check(self.lib.ia2c_rollout(C.byref(self.desc), s), "ia2c_rollout")

    def update(self):
        d, s = C.byref(self.desc), self._stream()
        with torch.cuda.device(self.device):
            if self.p2p:
                step = self.episode + 1          # one Adam step per net per episode
                _lib.check(self.lib.ia2c_critic_phase(d, s), "ia2c_critic_phase")      # gradient partials only
                self._epoch += 1
                _lib.check(self.lib.ia2c_allreduce_adam(d, 0, C.byref(self.peers), self._epoch, step, s), "ia2c_allreduce_adam(critic)")
                _lib.check(self.lib.ia2c_actor_phase(d, s), "ia2c_actor_phase")
                self._epoch += 1
                _lib.check(self.lib.ia2c_allreduce_adam(d, 1, C.byref(self.peers), self._epoch, step, s), "ia2c_allreduce_adam(actor)")
                return
            _lib.check(self.lib.ia2c_critic_phase(d, s), "ia2c_critic_phase")
            if self.world > 1:
                self._allreduce(self.critic_grad)
                _lib.check(self.lib.ia2c_apply_adam(d, 0, s), "ia2c_apply_adam(critic)")
            _lib.check(self.lib.ia2c_actor_phase(d, s), "ia2c_actor_phase")
            if self.world > 1:
                self._allreduce(self.actor_grad)
                _lib.check(self.lib.ia2c_apply_adam(d, 1, s), "ia2c_apply_adam(actor)")

    def _allreduce(self, buf):
        import torch.distributed as dist

        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=self.pg)

    def train_episode(self, sync_stats=False):
        """One episode: rollout, critic update, actor update.  Asynchronous unless ``sync_stats``.  ``train_episodes(n)``
        (one GPU) trains n episodes and records their statistics on the device for ``history()``; those episodes do not
        enter the ``read_stats`` windows."""
        if self.world == 1:   # one C call for the whole episode
            self.desc.episode = self.episode
            with torch.cuda.device(self.device):
                self._enqueue_episode(C.byref(self.desc), self._stream())
        elif self.p2p:        # one C call per rank: the gradient exchanges are kernels of the same stream
            self.desc.episode = self.episode
            with torch.cuda.device(self.device):
                _lib.check(self.lib.ia2c_train_episode_p2p(C.byref(self.desc), C.byref(self.peers), self._epoch, self._stream()),
                           "ia2c_train_episode_p2p")
            self._epoch += 2
        else:
            self.rollout()
            self.update()
        self.episode += 1
        if sync_stats:
            return self.read_stats()

    # ---- learning curves recorded on the device (ia2c_b200/history.py: train_episodes, history) --------------------
    def _check_history(self):
        if self.world > 1:
            raise _lib.IA2CError("train_episodes records histories on one GPU (a rank sees only its env shard)")

    def _history_dims(self):
        return 1, self.N, self.E, self.T, True

    def _enqueue_episode(self, desc_ref, stream):
        if self._env_partners:
            self._play_env_partners(lambda p: self.lib.ia2c_train_episode_env_partners(desc_ref, None, p, stream),
                                    "ia2c_train_episode_env_partners")
            return
        self._seat_partners(stream)
        _lib.check(self.lib.ia2c_train_episode(desc_ref, stream), "ia2c_train_episode")

    # ---- frozen partners (ia2c_b200/partners.py: set_partners, partner_history) -------------------------------------
    def _check_partners(self):
        if self.world > 1:
            raise _lib.IA2CError("set_partners seats partners on one GPU (a rank sees only its env shard)")

    def _check_env_partners(self):
        """The rollouts with per-env kernels: the fused one (N <= 8) and the whole-episode one (9 <= N <= 256)."""
        N, M, flags = self.N, self.M, self.desc.flags
        if N > 256:
            raise _lib.IA2CError(f"set_partners(per_env=True): n_agents={N} above 256 runs the per-step rollout, which has no per-env kernels")
        if N <= 8 and not flags & _lib.FLAG_FUSED_ROLLOUT:
            raise _lib.IA2CError(f"set_partners(per_env=True): n_agents={N}, n_models={M} runs the per-step rollout "
                                 "(fused_rollout=False or no fused instantiation), which has no per-env kernels")
        if N > 8 and (flags & (_lib.FLAG_ROLLOUT_PER_STEP | _lib.FLAG_BELIEF_PER_STEP) or not self.lib.ia2c_belief_supports_episode(N, M)):
            raise _lib.IA2CError("set_partners(per_env=True): the per-step rollout (rollout_kernel='step', belief_kernel='step' "
                                 "or no whole-episode belief kernel) has no per-env kernels")

    def _partner_runs(self):
        return 1, None

    def train_episode_host(self, host_u_action, host_u_belief):
        """End-to-end form with HOST inputs/outputs: pinned uniforms in, losses + episode returns out;
        the copies and a stream sync are inside the call (single rank)."""
        if self.world > 1:
            raise _lib.IA2CError("train_episode_host is the single-rank entry point")
        self._refuse_partners("train_episode_host")
        if self.inj_u_action is None or self.inj_u_belief is None:
            T, E, N, K = self.T, self.E, self.N, self.K
            self.inject(u_action=torch.zeros(T + 1, E, N), u_belief=torch.zeros(T + 1, E, N, K, dtype=torch.float64))
        self.desc.episode = self.episode
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ia2c_train_episode_host(
                C.byref(self.desc), host_u_action.data_ptr(), host_u_belief.data_ptr(), self._h_loss.data_ptr(),
                self._h_return.data_ptr(), self._stream()), "ia2c_train_episode_host")
        self.episode += 1
        return self._record_stats()

    # ---- host-tape pipeline (end-to-end form) -----------------------------------------------------------------
    def host_tape_bytes(self):
        n_act = (self.T + 1) * self.E * self.N
        return ((n_act * 4 + 7) & ~7) + n_act * self.K * 8

    def pack_host_tape(self, u_action, u_belief):
        """One pinned host buffer per episode: [u_action f32[T+1,E,N] | pad | u_belief f64[T+1,E,N,K]]."""
        n_act = (self.T + 1) * self.E * self.N
        off = (n_act * 4 + 7) & ~7
        tape = torch.empty(self.host_tape_bytes(), dtype=torch.uint8).pin_memory()
        tape[:n_act * 4].view(torch.float32).copy_(torch.as_tensor(np.asarray(u_action), dtype=torch.float32).reshape(-1))
        tape[off:].view(torch.float64).copy_(torch.as_tensor(np.asarray(u_belief), dtype=torch.float64).reshape(-1))
        return tape

    HOST_STAGES = 4   # depth of the device staging ring of the pipelined host path (ia2c_host_pipe_set_stages)

    def _ensure_stage(self):
        """Device staging regions for the tapes: region A (the desc's injected-uniform pointers are views of it) and one
        buffer holding the HOST_STAGES - 1 further regions of the ring (its first region doubles as region B of the NCCL path)."""
        if getattr(self, "_stage", None) is None:
            nbytes = self.host_tape_bytes()
            stride = int(self.lib.ia2c_host_stage_stride(C.byref(self.desc)))
            self._stage_ring = torch.empty(stride * (self.HOST_STAGES - 1), dtype=torch.uint8, device=self.device)
            self._stage = [torch.empty(nbytes, dtype=torch.uint8, device=self.device), self._stage_ring[:nbytes]]
        self._point_at_stage(0)

    def _point_at_stage(self, b):
        T, E, N, K = self.T, self.E, self.N, self.K
        n_act = (T + 1) * E * N
        off = (n_act * 4 + 7) & ~7
        self.inj_u_action = self._stage[b][:n_act * 4].view(torch.float32).view(T + 1, E, N)
        self.inj_u_belief = self._stage[b][off:].view(torch.float64).view(T + 1, E, N, K)
        self.desc.inj_u_action, self.desc.inj_u_belief = self.inj_u_action.data_ptr(), self.inj_u_belief.data_ptr()

    def train_episodes_host(self, host_tapes):
        """Pipelined end-to-end form: a list of per-episode pinned host tapes (``pack_host_tape``) in, per-episode
        losses and returns out (the loss / return windows are updated; ``window_stats()`` computes their means on demand).  One H2D copy per episode, overlapping the previous episode's compute, and one D2H
        copy of the result region (``ia2c_train_episodes_host``; multi-rank: the same pipeline with torch streams)."""
        self._refuse_partners("train_episodes_host")
        n = len(host_tapes)
        N, E = self.N, self.E
        self._ensure_stage()
        res_bytes = self._result_region.numel()
        if getattr(self, "_h_results", None) is None or self._h_results.shape[0] < n:
            self._h_results = torch.zeros(max(n, 64), res_bytes, dtype=torch.uint8).pin_memory()   # grows rarely: not per call
            self._h_results_np = self._h_results.numpy()   # views of the pinned buffers: the per-call host work is ~100 us, it counts
            self._h_loss_np, self._h_return_np = self._h_loss.numpy(), self._h_return.numpy()
            self._tape_ptrs = {}
        if self.world > 1 and not self.p2p:
            self._pipeline_multirank(host_tapes)
        else:
            key = tuple(map(id, host_tapes))          # the same tapes are passed again and again: build the pointer array once
            hit = self._tape_ptrs.get(key)
            if hit is None:
                if len(self._tape_ptrs) >= 16:
                    self._tape_ptrs.clear()
                hit = self._tape_ptrs[key] = ((C.c_void_p * n)(*[t.data_ptr() for t in host_tapes]), list(host_tapes))   # the list keeps the ids alive
            ptrs = hit[0]
            if getattr(self, "_result_region_b", None) is None:
                self._result_region_b = torch.zeros_like(self._result_region)
            if getattr(self, "_pipe", None) is None:
                handle = C.c_void_p()
                with torch.cuda.device(self.device):
                    _lib.check(self.lib.ia2c_host_pipe_create(C.byref(handle)), "ia2c_host_pipe_create")
                    _lib.check(self.lib.ia2c_host_pipe_set_stages(handle, self.HOST_STAGES), "ia2c_host_pipe_set_stages")
                self._pipe = handle
            self.desc.episode = self.episode
            with torch.cuda.device(self.device):
                if self.world == 1:
                    _lib.check(self.lib.ia2c_train_episodes_host(C.byref(self.desc), self._pipe, self._stage[1].data_ptr(),
                                                                 self._result_region_b.data_ptr(), n, ptrs,
                                                                 self._h_results.data_ptr(), self._stream()),
                               "ia2c_train_episodes_host")
                else:   # every rank runs the same C pipeline; the gradient exchanges are the fused NVLink kernels
                    _lib.check(self.lib.ia2c_train_episodes_host_p2p(C.byref(self.desc), self._pipe, C.byref(self.peers), self._epoch,
                                                                     self._stage[1].data_ptr(), self._result_region_b.data_ptr(),
                                                                     n, ptrs, self._h_results.data_ptr(), self._stream()),
                               "ia2c_train_episodes_host_p2p")
                    self._epoch += 2 * n
            self.episode += n
            if self.world > 1:
                self.check_comm()
        # one vectorised pass over the pinned result slots: per-episode Python work (and the 50*E window means, which
        # ia2c.py only prints every 10 episodes) would leave the GPU idle between calls -> window_stats() is on demand
        res = self._h_results_np[:n]
        losses = res[:, :2 * N * 4].copy().view(np.float32).reshape(n, 2, N)
        rets = res[:, self._off_ret:self._off_ret + E * 8].copy().view(np.float64).reshape(n, E)
        self._h_loss_np[...] = losses[-1]
        self._h_return_np[...] = rets[-1]
        critic, actor = list(losses[:, 0]), list(losses[:, 1])
        ret_rows = list(rets)
        self.critic_losses = (self.critic_losses + critic[-20:])[-20:]
        self.actor_losses = (self.actor_losses + actor[-20:])[-20:]
        self.reward_lst = (self.reward_lst + ret_rows[-50:])[-50:]
        return [{"critic_loss": c, "actor_loss": a, "ep_return": r} for c, a, r in zip(critic, actor, ret_rows)]

    def _pipeline_multirank(self, host_tapes):
        """Same pipeline with torch streams/events around the per-phase entry points (the gradient exchanges sit
        between them, so the single C call cannot be used)."""
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        cur = torch.cuda.current_stream(self.device)
        copied = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]
        for ev_ in consumed:
            ev_.record(cur)
        for k, tape in enumerate(host_tapes):
            b = k & 1
            with torch.cuda.stream(self._copy_stream):
                self._copy_stream.wait_event(consumed[b])
                self._stage[b].copy_(tape, non_blocking=True)
                copied[b].record(self._copy_stream)
            cur.wait_event(copied[b])
            self._point_at_stage(b)
            self.rollout()
            self.update()
            consumed[b].record(cur)
            self.episode += 1
            self._h_results[k].copy_(self._result_region, non_blocking=True)
        cur.synchronize()
        self._point_at_stage(0)
        self.check_comm()

    def train_episode_timed(self):
        """One episode with CUDA events between the kernels (profiling): returns the five warm durations in ms
        {rollout, critic_grad, critic_reduce_adam, actor_grad, actor_reduce_adam}.  Single rank."""
        if self.world > 1:
            raise _lib.IA2CError("train_episode_timed is the single-rank profiling entry point")
        self._refuse_env_partners("train_episode_timed")
        ms = (C.c_float * 5)()
        self.desc.episode = self.episode
        with torch.cuda.device(self.device):
            self._seat_partners(self._stream())   # before the first event: the timings cover the episode's kernels only
            _lib.check(self.lib.ia2c_train_episode_timed(C.byref(self.desc), ms, self._stream()), "ia2c_train_episode_timed")
        self.episode += 1
        return dict(zip(("rollout", "critic_grad", "critic_reduce_adam", "actor_grad", "actor_reduce_adam"), list(ms)))

    def check_comm(self):
        """Raise if a fused all-reduce failed anywhere in the job: a rank whose peers did not arrive within the time
        budget applies nothing, stops exchanging and raises the error word of EVERY rank (csrc/trainer.cu), so all
        ranks fail here together.  Called before statistics are read, before a checkpoint is taken and at the end of
        every pipelined host call; parameters of a run that raised here must not be used."""
        if self.p2p and int(self._comm_error[0].item()):
            raise _lib.IA2CError("ia2c_allreduce_adam: a rank's gradient words did not arrive within the time budget; "
                                 "the update was NOT applied and the exchange is disabled (parameters may differ across ranks)")

    def __del__(self):
        pipe, self._pipe = getattr(self, "_pipe", None), None
        if pipe is not None:
            try:
                self.lib.ia2c_host_pipe_destroy(pipe)
            except Exception:
                pass

    def read_stats(self):
        self.check_comm()
        self._h_loss.copy_(self.loss_out, non_blocking=True)
        self._h_return.copy_(self.ep_return, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return self._record_stats()

    def _record_stats(self, windows=True):
        """Append this episode's losses / returns to the reference's windows (20-deep loss windows, ac_nets.py:77-80;
        last-50 returns, ia2c.py:134).  The window means are what ia2c.py prints every 10 episodes; computing them is
        host work proportional to 50*E, so the pipelined path asks for them only when it needs them."""
        loss = self._h_loss.numpy().copy()
        ret = self._h_return.numpy().copy()
        self.critic_losses.append(loss[0]), self.actor_losses.append(loss[1])
        del self.critic_losses[:-20], self.actor_losses[:-20]
        self.reward_lst.append(ret)
        del self.reward_lst[:-50]
        out = dict(critic_loss=loss[0], actor_loss=loss[1], ep_return=ret)
        if windows:
            out.update(self.window_stats())
        return out

    def window_stats(self):
        return dict(critic_loss_window=np.mean(self.critic_losses, axis=0), actor_loss_window=np.mean(self.actor_losses, axis=0),
                    mean_return=np.mean(self.reward_lst))

    # ------------------------------------------------------------------ checkpoint / resume (SURVEY.md §8 f4)
    _CKPT_TENSORS = ("actor_params", "critic_params", "actor_grad_accum", "actor_m", "actor_v", "critic_m", "critic_v",
                     "actor_step", "critic_step", "filter_action", "env_state", "env_hist", "env_cls", "env_elapsed",
                     "belief_records")

    def state_dict(self):
        """Everything a resumed run needs to continue bit-identically: network parameters, Adam moments and step
        counters, the actor's never-zeroed gradient accumulators (SURVEY.md Q2), the belief models, env and belief
        state, the episode counter that keys the Philox streams, and the loss / return windows that ia2c.py prints
        (the reference has no checkpointing; SURVEY.md §5 lists this state)."""
        torch.cuda.current_stream(self.device).synchronize()
        self.check_comm()   # never checkpoint parameters of a run whose gradient exchange failed
        sd = {k: getattr(self, k).detach().cpu().clone() for k in self._CKPT_TENSORS}
        sd.update(episode=self.episode, seed=self.seed, dims=(self.E_total, self.E, self.N, self.M, self.T),
                  rank=self.rank, world=self.world, critic_losses=list(self.critic_losses),
                  actor_losses=list(self.actor_losses), reward_lst=list(self.reward_lst))
        return self._partner_state(sd)

    def load_state_dict(self, sd):
        if tuple(sd["dims"]) != (self.E_total, self.E, self.N, self.M, self.T) or sd["world"] != self.world:
            raise ValueError(f"checkpoint is for dims/world {sd['dims']}/{sd['world']}, "
                             f"trainer has {(self.E_total, self.E, self.N, self.M, self.T)}/{self.world}")
        for k in self._CKPT_TENSORS:
            getattr(self, k).copy_(sd[k])
        self.episode, self.seed = int(sd["episode"]), int(sd["seed"])
        self.desc.seed = self.seed
        self.critic_losses, self.actor_losses = list(sd["critic_losses"]), list(sd["actor_losses"])
        self.reward_lst = list(sd["reward_lst"])
        self._load_partner_state(sd)   # the checkpoint's pool, or none

    def save(self, path):
        torch.save(self.state_dict(), path)

    def load(self, path):
        self.load_state_dict(torch.load(path, map_location="cpu", weights_only=False))

    # ------------------------------------------------------------------ frozen-policy evaluation
    def evaluate(self, episodes=1, num_envs=None, greedy=False, seed=0, first_episode=0):
        """Evaluate the current actors without training: ``episodes`` episodes of T steps in each of ``num_envs`` envs
        (default E_total; greedy: 1) from the reset state, with this trainer's max_episode_steps.  Actions are sampled from
        the actors with Philox stream 4 keyed by ``seed`` (episodes ``first_episode`` onwards) or, with ``greedy``, are their
        argmax.  Reads ``actor_params`` on the trainer's stream and writes no trainer buffer; at world > 1 it runs on the
        calling rank alone, with its replicated parameters.  Returns returns [K, E], mean_return, std_return,
        action_counts / action_freq [N, 3] (freq = counts / (K * E * T)), policy [N, 9, 3] and, greedy, greedy_actions [N, 9]."""
        from .evaluate import evaluate_actors

        E = (1 if greedy else self.E_total) if num_envs is None else num_envs
        out = evaluate_actors(self.actor_params, 1, self.N, E, episodes, self.T, self.desc.max_episode_steps, greedy, seed,
                              first_episode, self.device)
        return {k: v[0] for k, v in out.items()}

    # ------------------------------------------------------------------ accounting
    def agent_steps_per_episode(self):
        return self.E_total * self.N * self.T
