"""ia2c_b200 — B200-native (sm_100a) implementation of IA2C's rollout-and-update hot path.

Host code is Python/PyTorch (device memory, streams, torch.distributed); every numeric step is a
hand-written CUDA kernel in libia2c_b200.so behind the C ABI of include/ia2c_b200.h.  There is no CPU
fallback: importing the compute classes without the built library or without a CUDA device raises.

Drop-in modules for the reference's scripts live in ``ia2c_b200/compat`` (importable as ``Org``,
``ac_nets``, ``belief_filter`` once that directory is on ``sys.path``).
"""
__version__ = "0.1.0"

from . import _lib  # noqa: F401


def __getattr__(name):  # lazy: torch-dependent classes are imported on first use
    if name in ("OrgVecEnv", "Org"):
        from . import org_env
        return getattr(org_env, name)
    if name in ("NeuralNet", "CriticNetwork", "ActorNetwork", "Adam"):
        from . import nets
        return getattr(nets, name)
    if name == "BeliefFilter":
        from .belief import BeliefFilter
        return BeliefFilter
    if name in ("IA2CTrainer", "reference_init"):
        from . import trainer
        return getattr(trainer, name)
    if name in ("IA2CRuns", "IA2CRunsMany"):
        from . import runs
        return getattr(runs, name)
    if name in ("A2COrgTrainer", "a2c_reference_init"):
        from . import a2c
        return getattr(a2c, name)
    raise AttributeError(name)
