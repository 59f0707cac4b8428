"""A2COrgTrainer — the single-agent A2C loop of a2c_org_test.py:43-92 on the GPU, for many envs and independent runs.

One update of every run is ONE C call (``ia2c_a2c_train_update``) that makes four launches: rollout + critic gradient,
critic reduce + Adam, actor gradient, actor reduce + Adam.  The reference runs one env and one run per process and is
latency-bound; here E envs per run and R runs (seeds, hyper-parameter sweeps) share the same four launches.

What one update computes (include/ia2c_b200.h states it in full; SURVEY.md §0.1 lists the quirks):
  * one joint agent with 9 actions; actor and critic are 6 -> 6 -> 6 -> 9 MLPs (the actor ends in a softmax);
  * the envs are reset once, at construction, and never again; there is no TimeLimit (Q6).  Env state, the fp64 reward
    history and the pending action carry across updates;
  * step t: ``Org.step(pending)``, then the next action is sampled from the post-step observation; the stored pair is
    (post-step obs, action taken) (Q4).  Update 0 first draws one action from the reset observation;
  * critic: target = reward, ``L = mean((r - Q(S)[a])^2)``, Adam.  The reference's ``masks`` are always 0 (Q5), so its
    discount multiplies zero and has no effect: this trainer has no ``gamma``;
  * actor: Q from the updated critic, ``V = sum(Q * pi)``, ``adv = Q[a] - V`` with gradient through pi (Q7), policy
    gradient + beta * entropy, Adam on the never-zeroed running sum of the gradients (Q2);
  * one row per env: the reference's two buffer rows are copies of its one env, and a mean over the copies is the mean
    over one row.  The means divide by T * E.

Sampling draws from Philox (key = run seed, counter = (env within its run, slot | 3 << 16, update); DESIGN.md §4), or
``inject(actions)`` replays actions, e.g. the reference's recorded ``torch.multinomial`` draws.

Run r of a batch computes byte for byte what ``A2COrgTrainer(num_envs, seeds=seeds[r], <run r's hyper-parameters>,
init=[init[r]])`` computes.  The device buffers hold the runs stacked: per-net buffers have R rows, per-env buffers an env
axis of length R * E with run r at [r*E, (r+1)*E); ``run_view(r)`` returns run r's slices.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .nets import hidden_size
from .runs import _per_run

N_FEATURES, N_JOINT = 6, 9
P = _lib.CRITIC_P   # 147 parameters in each of the two nets

_NET = ("actor_params", "critic_params", "actor_grad", "critic_grad", "actor_grad_accum", "actor_m", "actor_v", "critic_m",
        "critic_v", "actor_step", "critic_step")
_ENV = {"env_state": 0, "env_hist": 0, "env_cls": 0, "env_elapsed": 0, "pending_action": 0, "ep_return": 0,
        "obs": 1, "act": 1, "reward": 1}
_CKPT = _NET + tuple(_ENV)


def a2c_reference_init(seed=None):
    """Initial parameters drawn the way a2c_org_test.py:36-37 draws them: ``torch.manual_seed(seed)``, then the critic's
    three ``nn.Linear`` (default init from torch's CPU generator), then the actor's.  Returns (actor [147], critic [147])."""
    if seed is not None:
        torch.manual_seed(seed)

    def net():
        ls = (nn.Linear(N_FEATURES, hidden_size), nn.Linear(hidden_size, hidden_size), nn.Linear(hidden_size, N_JOINT))
        return torch.cat([t.detach().reshape(-1) for l in ls for t in (l.weight, l.bias)]).numpy()

    critic = net()
    actor = net()
    return actor, critic


class A2COrgTrainer:
    def __init__(self, num_envs=1, seeds=0, steps_per_update=100, lr_actor=1e-4, lr_critic=5e-5, beta=0.01, init=None,
                 device=None):
        self.lib = _lib.load()
        seeds = [int(seeds)] if np.ndim(seeds) == 0 else [int(s) for s in seeds]
        R, E, T = len(seeds), int(num_envs), int(steps_per_update)
        if R < 1:
            raise ValueError("seeds: need at least one run")
        if R > _lib.A2C_MAX_RUNS:
            raise ValueError(f"{R} runs above the limit of {_lib.A2C_MAX_RUNS}")
        if any(s < 0 or s >= 1 << 64 for s in seeds):
            raise ValueError("seeds must lie in [0, 2**64)")
        if E < 1 or R * E > _lib.A2C_MAX_ENVS:
            raise ValueError(f"num_envs={E} must be >= 1 and runs * num_envs at most {_lib.A2C_MAX_ENVS}")
        if not 1 <= T <= _lib.A2C_MAX_STEPS:
            raise ValueError(f"steps_per_update={T} outside 1..{_lib.A2C_MAX_STEPS}")
        hyper = {name: _per_run(name, v, R, dt) for name, v, dt in
                 (("lr_actor", lr_actor, np.float64), ("lr_critic", lr_critic, np.float64), ("beta", beta, np.float32))}
        if init is not None:
            if len(init) != R:
                raise ValueError(f"init: need one (actor, critic) pair per run ({R}), got {len(init)}")
            init = [tuple(np.asarray(x, dtype=np.float32).reshape(-1) for x in pair) for pair in init]
            if any(len(pair) != 2 or pair[0].size != P or pair[1].size != P for pair in init):
                raise ValueError(f"init: every run needs (actor, critic) with {P} parameters each")
        _lib.require_cuda()
        self.R, self.E, self.T = R, E, T
        self.seeds = seeds
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.update = 0
        dev, RE = self.device, R * E

        def z(shape, dtype):
            return torch.zeros(shape, dtype=dtype, device=dev)

        f32, f64, u8, i32 = torch.float32, torch.float64, torch.uint8, torch.int32
        self.actor_params, self.critic_params = z((R, P), f32), z((R, P), f32)
        self.actor_grad, self.critic_grad = z((R, P + 1), f32), z((R, P + 1), f32)
        self.actor_grad_accum = z((R, P), f32)
        self.actor_m, self.actor_v, self.critic_m, self.critic_v = z((R, P), f32), z((R, P), f32), z((R, P), f32), z((R, P), f32)
        self.actor_step, self.critic_step = z((R,), i32), z((R,), i32)
        self.loss_out = z((2, R), f32)
        self.env_state, self.env_hist = z((RE,), i32), z((RE,), f64)
        self.env_cls, self.env_elapsed = z((RE, 2), u8), z((RE,), i32)
        self.pending_action, self.ep_return = z((RE,), u8), z((RE,), f64)
        self.obs, self.act, self.reward = z((T, RE, N_FEATURES), f32), z((T, RE), u8), z((T, RE), f32)
        self.inj_actions = None
        self._seed = torch.from_numpy(np.asarray(seeds, dtype=np.uint64).view(np.int64)).to(dev)
        self._hyper = {k: (torch.from_numpy(a).to(dev) if a is not None else None) for k, (a, _) in hyper.items()}

        d = self.desc = _lib.A2CDesc()
        d.E, d.R, d.T, d.update = E, R, T, 0
        d.lr_actor, d.lr_critic, d.beta = hyper["lr_actor"][1], hyper["lr_critic"][1], hyper["beta"][1]
        d.seed = self._seed.data_ptr()
        d.lr_actor_run, d.lr_critic_run, d.beta_run = (self._hyper[k].data_ptr() if self._hyper[k] is not None else None
                                                       for k in ("lr_actor", "lr_critic", "beta"))
        for name in _CKPT + ("loss_out",):
            setattr(d, name, getattr(self, name).data_ptr())
        n_part = int(self.lib.ia2c_a2c_partials_floats(C.byref(d)))
        self.partials = z((n_part,), f32)
        d.partials, d.partials_floats = self.partials.data_ptr(), n_part

        self.critic_losses, self.actor_losses = [], []   # 20-deep windows (ac_nets.py:77-80,124-127), one column per run
        for r in range(R):
            actor, critic = init[r] if init is not None else a2c_reference_init(seeds[r])
            self.actor_params[r].copy_(torch.as_tensor(np.asarray(actor, dtype=np.float32).reshape(-1)))
            self.critic_params[r].copy_(torch.as_tensor(np.asarray(critic, dtype=np.float32).reshape(-1)))
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ia2c_org_reset(self.env_state.data_ptr(), self.env_hist.data_ptr(), self.env_cls.data_ptr(),
                                               self.env_elapsed.data_ptr(), None, RE, self._stream()), "ia2c_org_reset")

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    # ------------------------------------------------------------------ updates
    def inject(self, actions):
        """Replay actions instead of sampling: uint8-valued codes 0..8 of shape [T+1, R*E] (or [T+1, R, E]) in slot order —
        slot 0 is update 0's first draw (read at update 0 only), slot t+1 the draw after step t.  None returns to Philox."""
        if actions is None:
            self.inj_actions = None
            self.desc.inj_actions = None
            return
        a = np.asarray(actions)
        if a.shape not in ((self.T + 1, self.R * self.E), (self.T + 1, self.R, self.E)):
            raise ValueError(f"actions must have shape [T+1, R*E] = {(self.T + 1, self.R * self.E)}, got {a.shape}")
        if a.size and (a.min() < 0 or a.max() > N_JOINT - 1):
            raise ValueError("actions must be joint codes in 0..8")
        self.inj_actions = torch.as_tensor(a.reshape(self.T + 1, self.R * self.E).astype(np.uint8)).to(self.device)
        self.desc.inj_actions = self.inj_actions.data_ptr()

    def freeze_seats(self, seats):
        """Refused: the native A2C trainer trains one joint agent, which has no seats to freeze."""
        raise _lib.IA2CError("A2COrgTrainer trains one joint agent: it has no seats to freeze")

    def train_update(self, sync_stats=False):
        """One update of every run in one C call; asynchronous unless ``sync_stats``."""
        self.desc.update = self.update
        with torch.cuda.device(self.device):
            _lib.check(self.lib.ia2c_a2c_train_update(C.byref(self.desc), self._stream()), "ia2c_a2c_train_update")
        self.update += 1
        if sync_stats:
            return self.read_stats()

    def read_stats(self):
        """The last update's losses ``[R]`` and returns ``[R, E]`` (fp64 sum of the update's rewards), appended to each run's
        20-deep loss windows; the window means are what a2c_org_test.py:92 prints after the return."""
        loss = self.loss_out.cpu().numpy()
        self.critic_losses.append(loss[0].copy()), self.actor_losses.append(loss[1].copy())
        del self.critic_losses[:-20], self.actor_losses[:-20]
        return dict(critic_loss=loss[0], actor_loss=loss[1], ep_return=self.ep_return.cpu().numpy().reshape(self.R, self.E),
                    critic_loss_window=np.mean(self.critic_losses, axis=0, dtype=np.float32),
                    actor_loss_window=np.mean(self.actor_losses, axis=0, dtype=np.float32))

    # ------------------------------------------------------------------ one run's slice
    def run_view(self, r):
        """Views (no copies) of run r's slices of every device buffer."""
        if not 0 <= r < self.R:
            raise IndexError(f"run {r} of {self.R}")
        v = {k: getattr(self, k)[r:r + 1] for k in _NET}
        for k, axis in _ENV.items():
            v[k] = getattr(self, k).narrow(axis, r * self.E, self.E)
        v["loss_out"] = self.loss_out[:, r:r + 1]
        return v

    # ------------------------------------------------------------------ checkpoint / resume
    def state_dict(self):
        """Parameters, Adam moments and steps, the actor's gradient running sum, env state, reward history, pending action,
        the last update's trajectory, the update counter, the seeds and the loss windows."""
        torch.cuda.current_stream(self.device).synchronize()
        sd = {k: getattr(self, k).detach().cpu().clone() for k in _CKPT}
        sd.update(update=self.update, seeds=list(self.seeds), dims=(self.R, self.E, self.T),
                  critic_losses=[x.copy() for x in self.critic_losses], actor_losses=[x.copy() for x in self.actor_losses])
        return sd

    def load_state_dict(self, sd):
        """Restores everything ``state_dict`` holds; the hyper-parameters stay those this trainer was built with."""
        if tuple(sd["dims"]) != (self.R, self.E, self.T):
            raise ValueError(f"checkpoint is for (runs, E, T) = {tuple(sd['dims'])}, trainer has {(self.R, self.E, self.T)}")
        for k in _CKPT:
            getattr(self, k).copy_(sd[k])
        self.update = int(sd["update"])
        self.seeds = [int(s) for s in sd["seeds"]]
        self._seed.copy_(torch.from_numpy(np.asarray(self.seeds, dtype=np.uint64).view(np.int64)))
        self.critic_losses, self.actor_losses = list(sd["critic_losses"]), list(sd["actor_losses"])

    def save(self, path):
        torch.save(self.state_dict(), path)

    def load(self, path):
        self.load_state_dict(torch.load(path, map_location="cpu", weights_only=False))

    def env_steps_per_update(self):
        return self.R * self.E * self.T
