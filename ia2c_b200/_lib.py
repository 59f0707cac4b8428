"""ctypes binding of libia2c_b200.so (C ABI: include/ia2c_b200.h).

There is NO CPU fallback: if the shared library is missing or a CUDA device is absent, every product
entry point raises.  The library is built in-tree by ``python -m ia2c_b200.build`` (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IA2C_B200_LIB") or os.path.join(_PKG, "libia2c_b200.so")   # override: A/B runs of alternative builds

vp = C.c_void_p
i32, i64, u32, u64, f32, f64 = C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_float, C.c_double

FLAG_FUSED_ROLLOUT = 1
FLAG_SKIP_ADAM = 2
FLAG_FUSED_CRITIC = 4
FLAG_GRAD_ONLY = 8
FLAG_ACTOR_COLUMNS = 16
FLAG_BELIEF_PER_STEP = 32
FLAG_ROLLOUT_PER_STEP = 64
BELIEF_RECORD = 8
ABI_VERSION = 6
MAX_RUN_NETS = 65535   # IA2C_MAX_RUN_NETS: runs * n_agents of one batch
ACTOR_P = 105
CRITIC_P = 147
A2C_MAX_RUNS = 65535          # IA2C_A2C_MAX_RUNS
A2C_MAX_ENVS = 1 << 30        # IA2C_A2C_MAX_ENVS: envs per run and runs * envs
A2C_MAX_STEPS = 65534         # IA2C_A2C_MAX_STEPS
EVAL_MAX_RUNS = 65535         # IA2C_EVAL_MAX_RUNS
EVAL_MAX_AGENTS = 1023        # IA2C_EVAL_MAX_AGENTS
EVAL_MAX_STEPS = 65535        # IA2C_EVAL_MAX_STEPS
EVAL_MAX_LINEUPS = 1 << 20    # IA2C_EVAL_MAX_LINEUPS


class EpisodeDesc(C.Structure):
    """Mirror of ``ia2c_episode_desc`` (include/ia2c_b200.h) — field order and types must match."""
    _fields_ = [
        ("E", i64), ("E_total", i64), ("env_offset", i64),
        ("N", i32), ("T", i32), ("M", i32), ("max_episode_steps", i32),
        ("gamma", f32), ("beta", f32),
        ("lr_actor", f64), ("lr_critic", f64),
        ("seed", u64), ("episode", u32), ("flags", i32),
        ("actor_params", vp), ("actor_grad", vp), ("actor_grad_accum", vp), ("actor_m", vp), ("actor_v", vp),
        ("critic_params", vp), ("critic_grad", vp), ("critic_m", vp), ("critic_v", vp),
        ("actor_step", vp), ("critic_step", vp),
        ("loss_out", vp),
        ("filter_action", vp),
        ("env_state", vp), ("env_hist", vp), ("env_cls", vp), ("env_elapsed", vp),
        ("ep_return", vp),
        ("obs", vp), ("reward", vp), ("act", vp), ("partner_true", vp), ("partner_pred", vp),
        ("belief_records", vp),
        ("inj_actions", vp), ("inj_u_action", vp), ("inj_u_belief", vp),
        ("state_trace", vp), ("reward_f64", vp), ("pred_dump", vp), ("belief_dump", vp),
        ("adv_dump", vp), ("target_dump", vp),
        ("partials", vp), ("partials_floats", C.c_size_t),
    ]


class PeerDesc(C.Structure):
    """Mirror of ``ia2c_peer_desc``."""
    _fields_ = [("rank", i32), ("world", i32), ("inbox", vp * 8), ("mc_inbox", vp), ("error", vp * 8),
                ("timeout_us", u32), ("reserved", u32)]


class RunsDesc(C.Structure):
    """Mirror of ``ia2c_runs_desc``: a batch of independent runs (ia2c_train_episode_runs, ia2c_train_episode_runs_many)."""
    _fields_ = [("runs", i32), ("reserved", i32), ("seed", vp), ("lr_actor", vp), ("lr_critic", vp), ("gamma", vp), ("beta", vp)]


class A2CDesc(C.Structure):
    """Mirror of ``ia2c_a2c_desc``: one update of the native A2C trainer (ia2c_a2c_train_update)."""
    _fields_ = [
        ("E", i64), ("R", i32), ("T", i32), ("update", u32), ("beta", f32), ("lr_actor", f64), ("lr_critic", f64),
        ("seed", vp), ("lr_actor_run", vp), ("lr_critic_run", vp), ("beta_run", vp),
        ("actor_params", vp), ("actor_grad", vp), ("actor_grad_accum", vp), ("actor_m", vp), ("actor_v", vp),
        ("critic_params", vp), ("critic_grad", vp), ("critic_m", vp), ("critic_v", vp),
        ("actor_step", vp), ("critic_step", vp),
        ("env_state", vp), ("env_hist", vp), ("env_cls", vp), ("env_elapsed", vp), ("pending_action", vp), ("ep_return", vp),
        ("obs", vp), ("act", vp), ("reward", vp), ("loss_out", vp), ("inj_actions", vp),
        ("partials", vp), ("partials_floats", C.c_size_t),
    ]


class EvalDesc(C.Structure):
    """Mirror of ``ia2c_eval_desc``: a frozen-policy evaluation of R runs' actors (ia2c_evaluate)."""
    _fields_ = [
        ("actor_params", vp), ("R", i32), ("N", i32), ("E", i64),
        ("episodes", i32), ("T", i32), ("max_episode_steps", i32), ("greedy", i32),
        ("seed", u64), ("episode0", u32), ("inj_u_action", vp),
        ("policy", vp), ("policy_floats", C.c_size_t), ("returns", vp), ("action_counts", vp),
    ]


class LineupDesc(C.Structure):
    """Mirror of ``ia2c_lineup_desc``: a cross-play evaluation of P lineups seated from a pool of actors (ia2c_evaluate_lineups)."""
    _fields_ = [
        ("actor_params", vp), ("nets", i32), ("N", i32), ("P", i32), ("reserved", i32), ("lineups", vp), ("E", i64),
        ("episodes", i32), ("T", i32), ("max_episode_steps", i32), ("greedy", i32),
        ("seed", u64), ("episode0", u32), ("inj_u_action", vp),
        ("policy", vp), ("policy_floats", C.c_size_t), ("returns", vp), ("action_counts", vp),
        ("return_sum", vp), ("return_m2", vp),
    ]


class HistoryDesc(C.Structure):
    """Mirror of ``ia2c_history_desc``: the device ring of per-episode statistics (ia2c_record_episode)."""
    _fields_ = [("capacity", i32), ("return_sum", vp), ("loss", vp), ("action_counts", vp), ("partner_hits", vp)]


class PbtDesc(C.Structure):
    """Mirror of ``ia2c_pbt_desc``: one population-based-training generation of a batch (ia2c_pbt_step)."""
    _fields_ = [("window", i32), ("slot", i32), ("q", i32), ("perturb", u32), ("factor_lo", f64), ("factor_hi", f64),
                ("seed", u64), ("generation", u32), ("reserved", i32),
                ("lr_actor", vp), ("lr_critic", vp), ("gamma", vp), ("beta", vp),
                ("log_fitness", vp), ("log_rank", vp), ("log_donor", vp), ("log_lr_actor", vp), ("log_lr_critic", vp),
                ("log_gamma", vp), ("log_beta", vp), ("workspace", vp), ("workspace_bytes", C.c_size_t)]


PBT_LR_ACTOR, PBT_LR_CRITIC, PBT_BETA = 1, 2, 4   # IA2C_PBT_* bits of PbtDesc.perturb

_DP = C.POINTER(EpisodeDesc)

# name -> (restype, argtypes); every symbol declared in include/ia2c_b200.h
SIGNATURES = {
    "ia2c_last_error": (C.c_char_p, []),
    "ia2c_abi_version": (C.c_int, []),
    "ia2c_launch_count": (u64, []),
    "ia2c_org_reset": (C.c_int, [vp, vp, vp, vp, vp, i64, vp]),
    "ia2c_org_step_joint": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, vp]),
    "ia2c_org_step_agents": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, vp]),
    "ia2c_belief_update_dense": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, vp]),
    "ia2c_belief_update_pairs": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, u64, u32, u32, i64, vp]),
    "ia2c_belief_supports_episode": (C.c_int, [i32, i32]),
    "ia2c_belief_update_pairs_episode": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, u64, u32, i64, vp]),
    "ia2c_debug_divide": (C.c_int, [vp, vp, vp, vp, i64, vp]),
    "ia2c_debug_fp32_peak": (C.c_int, [vp, i32, i32, i32, C.POINTER(f64), vp]),
    "ia2c_mlp_forward": (C.c_int, [vp, vp, vp, vp, i64, i32, i32, i32, i32, vp]),
    "ia2c_mlp_backward_workspace": (C.c_size_t, [i64, i32, i32]),
    "ia2c_mlp_backward": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, i32, vp]),
    "ia2c_actor_sample": (C.c_int, [vp, vp, vp, vp, vp, i64, i32, i32, u64, u64, vp]),
    "ia2c_mlp_forward_index": (C.c_int, [vp, vp, vp, vp, i64, i32, i32, i32, vp]),
    "ia2c_mlp_backward_index": (C.c_int, [vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, i32, vp]),
    "ia2c_actor_sample_index": (C.c_int, [vp, vp, vp, vp, vp, i64, i32, i32, u64, u64, vp]),
    "ia2c_critic_loss": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, i64, i32, vp]),
    "ia2c_actor_loss": (C.c_int, [vp, vp, vp, f32, vp, vp, vp, vp, vp, i64, i32, vp]),
    "ia2c_loss_workspace": (C.c_size_t, [i64]),
    "ia2c_adam_step": (C.c_int, [vp, vp, vp, vp, vp, vp, f64, f64, f64, f64, i32, i32, vp]),
    "ia2c_net_update_workspace": (C.c_size_t, [i64, i32, i32]),
    "ia2c_net_update": (C.c_int, [i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_float, f64, vp, vp, vp, i64, i32, i32, vp]),
    "ia2c_episode_partials_floats": (C.c_size_t, [_DP]),
    "ia2c_rollout_fused_supported": (C.c_int, [i32, i32]),
    "ia2c_rollout": (C.c_int, [_DP, vp]),
    "ia2c_critic_phase": (C.c_int, [_DP, vp]),
    "ia2c_actor_phase": (C.c_int, [_DP, vp]),
    "ia2c_apply_adam": (C.c_int, [_DP, i32, vp]),
    "ia2c_peer_inbox_bytes": (C.c_size_t, [_DP, i32]),
    "ia2c_allreduce_adam": (C.c_int, [_DP, i32, C.POINTER(PeerDesc), u32, i32, vp]),
    "ia2c_train_episode": (C.c_int, [_DP, vp]),
    "ia2c_train_episode_p2p": (C.c_int, [_DP, C.POINTER(PeerDesc), u32, vp]),
    "ia2c_train_episode_host": (C.c_int, [_DP, vp, vp, vp, vp, vp]),
    "ia2c_train_episode_timed": (C.c_int, [_DP, vp, vp]),
    "ia2c_host_tape_bytes": (C.c_size_t, [_DP]),
    "ia2c_host_result_bytes": (C.c_size_t, [_DP]),
    "ia2c_host_pipe_create": (C.c_int, [C.POINTER(vp)]),
    "ia2c_host_pipe_destroy": (C.c_int, [vp]),
    "ia2c_host_pipe_set_stages": (C.c_int, [vp, i32]),
    "ia2c_host_stage_stride": (C.c_size_t, [_DP]),
    "ia2c_train_episodes_host": (C.c_int, [_DP, vp, vp, vp, i32, C.POINTER(vp), vp, vp]),
    "ia2c_train_episodes_host_p2p": (C.c_int, [_DP, vp, C.POINTER(PeerDesc), u32, vp, vp, i32, C.POINTER(vp), vp, vp]),
    "ia2c_runs_partials_floats": (C.c_size_t, [_DP, i32]),
    "ia2c_train_episode_runs": (C.c_int, [_DP, C.POINTER(RunsDesc), vp]),
    "ia2c_train_episode_runs_many": (C.c_int, [_DP, C.POINTER(RunsDesc), vp]),
    "ia2c_a2c_partials_floats": (C.c_size_t, [C.POINTER(A2CDesc)]),
    "ia2c_a2c_train_update": (C.c_int, [C.POINTER(A2CDesc), vp]),
    "ia2c_eval_policy_floats": (C.c_size_t, [C.POINTER(EvalDesc)]),
    "ia2c_evaluate": (C.c_int, [C.POINTER(EvalDesc), vp]),
    "ia2c_evaluate_lineups": (C.c_int, [C.POINTER(LineupDesc), vp]),
    "ia2c_record_episode": (C.c_int, [_DP, i32, C.POINTER(HistoryDesc), i32, vp]),
    "ia2c_pbt_workspace_bytes": (C.c_size_t, [i32]),
    "ia2c_pbt_step": (C.c_int, [_DP, C.POINTER(RunsDesc), C.POINTER(HistoryDesc), C.POINTER(PbtDesc), vp]),
}

_lib = None


class IA2CError(RuntimeError):
    pass


def load():
    """Load the shared library (building it first if nvcc is available and it is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build

        try:
            _build.build()
        except Exception as exc:  # no toolchain: fail loudly, there is no other implementation
            raise ImportError(
                f"ia2c_b200: {LIB_PATH} is missing and could not be built ({exc}). "
                "Run `python -m ia2c_b200.build` where CUDA 12.9 nvcc is installed.") from exc
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.ia2c_abi_version() != ABI_VERSION:
        raise ImportError("ia2c_b200: ABI version mismatch between _lib.py and libia2c_b200.so")
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().ia2c_last_error().decode(errors="replace")
        raise IA2CError(f"{what} failed with status {rc}: {msg}")


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise IA2CError("ia2c_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch


def ptr(t):
    """data_ptr of a CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "ia2c_b200 kernels take contiguous CUDA tensors"
    return t.data_ptr()


def stream_ptr():
    import torch

    return torch.cuda.current_stream().cuda_stream


def launch_count():
    return int(load().ia2c_launch_count())
