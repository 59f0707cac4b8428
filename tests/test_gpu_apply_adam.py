"""GPU: reduce_adam_kernel's Adam step (ia2c_apply_adam: Adam from the gradient buffers) against a float64 Adam, over step
counters from the first step to ones where b2^t underflows — the bias corrections are computed in the kernel from the
device-side step counter."""
import ctypes as C

import numpy as np
import pytest

from tests.helpers import host

pytestmark = pytest.mark.gpu


def _adam(p, m, v, g, t, lr):
    b1, b2 = 0.9, 0.999
    p, m, v, g = (np.asarray(x, np.float64) for x in (p, m, v, g))
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    p = p - lr / (1 - b1 ** t) * (m / (np.sqrt(v) / np.sqrt(1 - b2 ** t) + 1e-8))
    return p, m, v


def _close(dev, ref, tol=1e-6):
    dev, ref = np.asarray(dev, np.float64), np.asarray(ref, np.float64)
    assert np.abs(dev - ref).max() <= tol * np.abs(ref).max()


@pytest.mark.parametrize("step0", [0, 1, 9, 1000, 123456, 2 ** 30])
def test_apply_adam_matches_float64_adam(step0):
    import torch
    from ia2c_b200.trainer import IA2CTrainer
    tr = IA2CTrainer(64, n_agents=3, seed=0)
    rng = np.random.RandomState(step0 % 1000)
    N = tr.N
    t = lambda x: torch.from_numpy(np.asarray(x, np.float32)).to(tr.device)
    for net, P in (("critic", 147), ("actor", 105)):
        getattr(tr, f"{net}_grad").copy_(t(rng.randn(N, P + 1) * 1e-2))
        getattr(tr, f"{net}_m").copy_(t(rng.randn(N, P) * 1e-3))
        getattr(tr, f"{net}_v").copy_(t(rng.rand(N, P) * 1e-5))
        getattr(tr, f"{net}_step").fill_(step0)
    tr.actor_grad_accum.copy_(t(rng.randn(N, 105) * 1e-2))
    torch.cuda.synchronize()
    pre = {k: host(getattr(tr, k)).copy() for k in ("critic_params", "critic_m", "critic_v", "critic_grad", "actor_params", "actor_m",
                                                    "actor_v", "actor_grad", "actor_grad_accum")}
    for which in (0, 1):
        assert tr.lib.ia2c_apply_adam(C.byref(tr.desc), which, tr._stream()) == 0
    torch.cuda.synchronize()
    assert (host(tr.critic_step) == step0 + 1).all() and (host(tr.actor_step) == step0 + 1).all()
    assert np.array_equal(host(tr.loss_out)[0], pre["critic_grad"][:, -1]) and np.array_equal(host(tr.loss_out)[1], pre["actor_grad"][:, -1])
    p, m, v = _adam(pre["critic_params"], pre["critic_m"], pre["critic_v"], pre["critic_grad"][:, :-1], step0 + 1, tr.desc.lr_critic)
    _close(host(tr.critic_params), p), _close(host(tr.critic_m), m), _close(host(tr.critic_v), v)
    g = pre["actor_grad_accum"].astype(np.float64) + pre["actor_grad"][:, :-1]       # never zeroed (Q2)
    _close(host(tr.actor_grad_accum), g)
    p, m, v = _adam(pre["actor_params"], pre["actor_m"], pre["actor_v"], host(tr.actor_grad_accum), step0 + 1, tr.desc.lr_actor)
    _close(host(tr.actor_params), p), _close(host(tr.actor_m), m), _close(host(tr.actor_v), v)
