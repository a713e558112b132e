"""ctypes binding of libb2rl.so (include/b2rl.h).  There is NO fallback: if the CUDA library is
missing or CUDA is unavailable the product path raises immediately."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libb2rl.so")

B2RL_MAX_ENC = 12
B2RL_MAX_HEAD = 6

ACT = {None: 0, "Identity": 0, "ReLU": 1, "ELU": 2, "GELU": 3, "Tanh": 4}
LAYER_CONV, LAYER_LINEAR = 0, 1
LN_NONE, LN_AFFINE, LN_PLAIN = 0, 1, 2
NET_Q, NET_RAINBOW = 0, 1


class Layer(Structure):
    _fields_ = [
        ("kind", c_int32), ("in_c", c_int32), ("in_h", c_int32), ("in_w", c_int32),
        ("out_c", c_int32), ("out_h", c_int32), ("out_w", c_int32), ("ksize", c_int32),
        ("stride", c_int32), ("act", c_int32), ("ln", c_int32), ("noisy", c_int32),
        ("w_off", c_int64), ("b_off", c_int64), ("ws_off", c_int64), ("bs_off", c_int64),
        ("we_off", c_int64), ("be_off", c_int64), ("lnw_off", c_int64), ("lnb_off", c_int64),
    ]


class NetDesc(Structure):
    _fields_ = [
        ("kind", c_int32), ("n_enc", c_int32), ("n_val", c_int32), ("n_adv", c_int32),
        ("enc", Layer * B2RL_MAX_ENC), ("val", Layer * B2RL_MAX_HEAD), ("adv", Layer * B2RL_MAX_HEAD),
        ("n_actions", c_int32), ("n_atoms", c_int32), ("obs_u8", c_int32), ("normalize", c_int32),
        ("obs_low", c_float), ("obs_high", c_float), ("obs_elems", c_int64),
        ("n_params", c_int64), ("n_eps", c_int64),
    ]


class LearnCfg(Structure):
    _fields_ = [
        ("batch", c_int64), ("gamma", c_double), ("v_min", c_double), ("v_max", c_double),
        ("delta_z", c_double), ("weights_mode", c_int32), ("driver_shapes", c_int32),
        ("double_dqn", c_int32), ("clip", c_int32), ("max_grad_norm", c_double),
        ("lr", c_double), ("beta1", c_double), ("beta2", c_double), ("adam_eps", c_double),
        ("bias_correction1", c_double), ("bias_correction2", c_double), ("tau", c_double),
        ("prior_eps", c_double), ("accumulate", c_int32), ("use_noise", c_int32),
        ("side_streams", c_int32), ("reserved_", c_int32),
    ]


class LearnBufs(Structure):
    _fields_ = [
        ("actor_params", c_void_p), ("target_params", c_void_p), ("actor_eps", c_void_p),
        ("target_eps", c_void_p), ("grads", c_void_p), ("exp_avg", c_void_p), ("exp_avg_sq", c_void_p),
        ("obs", c_void_p), ("next_obs", c_void_p), ("row_idx", c_void_p), ("action", c_void_p),
        ("reward", c_void_p), ("done", c_void_p), ("weights", c_void_p), ("support", c_void_p),
        ("loss_elem", c_void_p), ("priorities", c_void_p), ("loss_scalar", c_void_p),
        ("proj_dist", c_void_p), ("workspace", c_void_p), ("workspace_bytes", c_size_t),
        ("step_state", c_void_p),
    ]


class DdpgCfg(Structure):
    _fields_ = [
        ("batch", c_int64), ("twin", c_int32), ("policy_update", c_int32),
        ("gamma", c_double), ("tau", c_double), ("noise_clip", c_double), ("policy_noise", c_double),
        ("lr_actor", c_double), ("lr_critic", c_double), ("beta1", c_double), ("beta2", c_double), ("adam_eps", c_double),
        ("bc1_actor", c_double), ("bc2_actor", c_double), ("bc1_critic", c_double), ("bc2_critic", c_double),
        ("noise_seed", c_uint64), ("noise_offset", c_uint64),
    ]


class DdpgBufs(Structure):
    _fields_ = [
        ("actor", c_void_p), ("actor_target", c_void_p), ("actor_grads", c_void_p), ("actor_m", c_void_p), ("actor_v", c_void_p),
        ("critic", c_void_p * 2), ("critic_target", c_void_p * 2), ("critic_grads", c_void_p * 2), ("critic_m", c_void_p * 2),
        ("critic_v", c_void_p * 2),
        ("obs", c_void_p), ("next_obs", c_void_p), ("action", c_void_p), ("reward", c_void_p), ("done", c_void_p),
        ("noise", c_void_p), ("action_low", c_void_p), ("action_high", c_void_p),
        ("critic_loss", c_void_p), ("actor_loss", c_void_p), ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


B2RL_MAX_AGENTS = 8


class MaddpgCfg(Structure):
    _fields_ = [
        ("batch", c_int64), ("n_agents", c_int32), ("serial", c_int32),
        ("gamma", c_double), ("tau", c_double),
        ("lr_actor", c_double), ("lr_critic", c_double), ("beta1", c_double), ("beta2", c_double), ("adam_eps", c_double),
        ("bc1_actor", c_double), ("bc2_actor", c_double), ("bc1_critic", c_double), ("bc2_critic", c_double),
        ("twin", c_int32), ("critic_only", c_int32),
    ]


class MaddpgBufs(Structure):
    _fields_ = [
        ("actor", c_void_p * B2RL_MAX_AGENTS), ("actor_target", c_void_p * B2RL_MAX_AGENTS),
        ("actor_grads", c_void_p * B2RL_MAX_AGENTS), ("actor_m", c_void_p * B2RL_MAX_AGENTS), ("actor_v", c_void_p * B2RL_MAX_AGENTS),
        ("critic", c_void_p * B2RL_MAX_AGENTS), ("critic_target", c_void_p * B2RL_MAX_AGENTS),
        ("critic_grads", c_void_p * B2RL_MAX_AGENTS), ("critic_m", c_void_p * B2RL_MAX_AGENTS), ("critic_v", c_void_p * B2RL_MAX_AGENTS),
        ("obs", c_void_p), ("next_obs", c_void_p), ("action", c_void_p), ("reward", c_void_p), ("done", c_void_p),
        ("losses", c_void_p), ("workspace", c_void_p), ("workspace_bytes", c_size_t), ("step_state", c_void_p),
        ("critic2", c_void_p * B2RL_MAX_AGENTS), ("critic2_target", c_void_p * B2RL_MAX_AGENTS),
        ("critic2_grads", c_void_p * B2RL_MAX_AGENTS), ("critic2_m", c_void_p * B2RL_MAX_AGENTS),
        ("critic2_v", c_void_p * B2RL_MAX_AGENTS), ("actor_step_state", c_void_p),
    ]


class StepState(Structure):
    _fields_ = [
        ("beta", c_double), ("size", c_int64), ("sample_offset", c_uint64), ("noise_offset", c_uint64 * 2),
        ("lr", c_double), ("bias_correction1", c_double), ("bias_correction2", c_double),
    ]


_SIGS = {
    "b2rl_version": ([], c_int),
    "b2rl_debug_read": ([c_void_p, c_int], c_int),
    "b2rl_gae_scan": ([c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_double, c_double, c_int,
                       c_void_p, c_void_p, c_void_p], c_int),
    "b2rl_advantage_normalize": ([c_void_p, c_int64, c_void_p, c_void_p], c_int),
    "b2rl_gae_scan_normalize": ([c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_double, c_double,
                                 c_int, c_void_p, c_void_p, c_void_p, c_void_p], c_int),
    "b2rl_device_sm_count": ([c_int, POINTER(c_int)], c_int),
    "b2rl_tree_init": ([c_void_p, c_void_p, c_int64, c_void_p], c_int),
    "b2rl_tree_set": ([c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p], c_int),
    "b2rl_tree_set_range": ([c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_double, c_void_p], c_int),
    "b2rl_tree_set_range_devmax": ([c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_double, c_void_p, c_double,
                                    c_void_p], c_int),
    "b2rl_tree_set_from_priorities": ([c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_double,
                                       c_double, c_void_p, c_void_p], c_int),
    "b2rl_tree_retrieve": ([c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p], c_int),
    "b2rl_per_sample": ([c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_double, c_int64, c_void_p, c_void_p,
                         c_void_p], c_int),
    "b2rl_per_sample_philox": ([c_void_p, c_void_p, c_int64, c_uint64, c_uint64, c_int64, c_double, c_int64,
                                c_void_p, c_void_p, c_void_p], c_int),
    "b2rl_per_sample_fused": ([c_void_p, c_void_p, c_int64, c_void_p, c_uint64, c_uint64, c_int64, c_double, c_int64,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p], c_int),
    "b2rl_per_sample_fused_state": ([c_void_p, c_void_p, c_int64, c_uint64, c_void_p, c_int64, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p], c_int),
    "b2rl_noise_reset_state": ([POINTER(NetDesc), c_void_p, c_uint64, c_void_p, c_int, c_void_p], c_int),
    "b2rl_noise_reset_state_pair": ([POINTER(NetDesc), c_void_p, c_void_p, c_uint64, c_void_p, c_void_p], c_int),
    "b2rl_step_state_write": ([POINTER(StepState), c_void_p, c_void_p], c_int),
    "b2rl_copy_d2h": ([c_void_p, c_void_p, c_size_t, c_void_p], c_int),
    "b2rl_graph_begin": ([c_void_p], c_int),
    "b2rl_graph_end": ([c_void_p, POINTER(c_void_p)], c_int),
    "b2rl_graph_launch": ([c_void_p, POINTER(StepState), c_void_p], c_int),
    "b2rl_graph_launch_states": ([c_void_p, c_void_p, c_void_p, c_int, c_void_p], c_int),
    "b2rl_graph_kernel_count": ([c_void_p, POINTER(c_int)], c_int),
    "b2rl_graph_destroy": ([c_void_p], c_int),
    "b2rl_ddpg_workspace_bytes": ([POINTER(NetDesc), POINTER(NetDesc), c_int64, POINTER(c_size_t)], c_int),
    "b2rl_ddpg_learn": ([POINTER(NetDesc), POINTER(NetDesc), POINTER(DdpgCfg), POINTER(DdpgBufs), c_void_p], c_int),
    "b2rl_maddpg_workspace_bytes": ([c_void_p, c_void_p, c_int, c_int64, POINTER(c_size_t)], c_int),
    "b2rl_maddpg_workspace_bytes_cfg": ([c_void_p, c_void_p, POINTER(MaddpgCfg), POINTER(c_size_t)], c_int),
    "b2rl_maddpg_learn": ([c_void_p, c_void_p, POINTER(MaddpgCfg), POINTER(MaddpgBufs), c_void_p], c_int),
    "b2rl_gaussian_mutate": ([c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_uint64, c_uint64,
                              c_double, c_int64, c_void_p], c_int),
    "b2rl_actor_workspace_bytes": ([POINTER(NetDesc), c_int64, POINTER(c_size_t)], c_int),
    "b2rl_actor_forward": ([POINTER(NetDesc), c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_size_t, c_void_p], c_int),
    "b2rl_sample_uniform_distinct": ([c_uint64, c_uint64, c_int64, c_int64, c_void_p, c_void_p], c_int),
    "b2rl_host_priority_pow": ([c_void_p, c_int64, c_double, c_double, c_void_p, POINTER(c_double)], c_int),
    "b2rl_host_randperm_prefix": ([c_void_p, c_int64, c_int64, c_int64, c_void_p], c_int),
    "b2rl_philox_uniforms": ([c_uint64, c_uint64, c_int64, c_void_p, c_void_p], c_int),
    "b2rl_philox_normals": ([c_uint64, c_uint64, c_int64, c_void_p, c_void_p], c_int),
    "b2rl_ring_write": ([c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p], c_int),
    "b2rl_gather_rows": ([c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p], c_int),
    "b2rl_ring_write_multi": ([c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p], c_int),
    "b2rl_gather_rows_multi": ([c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p], c_int),
    "b2rl_nstep_ingest": ([c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_double, c_int64,
                           c_int64, c_void_p], c_int),
    "b2rl_nstep_fold": ([POINTER(c_void_p), POINTER(c_void_p), c_int, c_int64, c_double, c_void_p, c_void_p,
                         c_void_p], c_int),
    "b2rl_select_copy": ([c_void_p, POINTER(c_void_p), c_int, c_void_p, c_int64, c_void_p], c_int),
    "b2rl_net_workspace_bytes": ([POINTER(NetDesc), c_int64, c_int, POINTER(c_size_t)], c_int),
    "b2rl_noise_reset_from_normals": ([POINTER(NetDesc), c_void_p, c_void_p, c_void_p], c_int),
    "b2rl_noise_reset_philox": ([POINTER(NetDesc), c_void_p, c_uint64, c_uint64, c_void_p], c_int),
    "b2rl_noise_count": ([POINTER(NetDesc), POINTER(c_int64)], c_int),
    "b2rl_net_forward_q": ([POINTER(NetDesc), c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64,
                            c_void_p, c_void_p, c_void_p, c_size_t, c_void_p], c_int),
    "b2rl_net_forward_dist": ([POINTER(NetDesc), c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int64, c_int, c_void_p,
                               c_void_p, c_size_t, c_void_p], c_int),
    "b2rl_encoder_layer_forward": ([POINTER(NetDesc), c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                    c_size_t, c_int, c_void_p], c_int),
    "b2rl_encoder_layer_wgrad": ([POINTER(NetDesc), c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                  c_size_t, c_void_p], c_int),
    "b2rl_encoder_layer_dgrad": ([POINTER(NetDesc), c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_size_t,
                                  c_void_p], c_int),
    "b2rl_launch_count": ([], ctypes.c_ulonglong),
    "b2rl_conv_path_count": ([ctypes.c_int], ctypes.c_ulonglong),
    "b2rl_conv_staged_paths": ([ctypes.c_int], ctypes.c_int),
    "b2rl_rainbow_prep": ([POINTER(NetDesc), POINTER(LearnCfg), POINTER(LearnBufs), c_void_p], c_int),
    "b2rl_rainbow_loss": ([POINTER(NetDesc), POINTER(LearnCfg), POINTER(LearnBufs), c_void_p], c_int),
    "b2rl_rainbow_backward": ([POINTER(NetDesc), POINTER(LearnCfg), POINTER(LearnBufs), c_void_p], c_int),
    "b2rl_optim_step": ([POINTER(NetDesc), POINTER(LearnCfg), POINTER(LearnBufs), c_void_p], c_int),
    "b2rl_dqn_learn": ([POINTER(NetDesc), POINTER(LearnCfg), POINTER(LearnBufs), c_void_p], c_int),
    "b2rl_rainbow_learn": ([POINTER(NetDesc), POINTER(LearnCfg), POINTER(LearnBufs), c_void_p], c_int),
}

EXPORTS = tuple(_SIGS) + ("b2rl_last_error",)

_lib = None


class B2RLError(RuntimeError):
    pass


def load(require_cuda: bool = False):
    """Load libb2rl.so.  Raises if it has not been built (``python -m agilerl_b200.csrc.build``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B2RLError(
                f"{LIB_PATH} not found: the CUDA extension is not built. "
                "Run `python -m agilerl_b200.csrc.build` (there is no CPU fallback)."
            )
        lib = ctypes.CDLL(LIB_PATH)
        lib.b2rl_last_error.argtypes = []
        lib.b2rl_last_error.restype = c_char_p
        for name, (args, res) in _SIGS.items():
            fn = getattr(lib, name)   # AttributeError here == stale .so: rebuild
            fn.argtypes = args
            fn.restype = res
        _lib = lib
    if require_cuda and not torch.cuda.is_available():
        raise B2RLError("CUDA is not available: agilerl_b200 has no CPU fallback.")
    return _lib


def check(rc: int) -> None:
    if rc == 0:
        return
    msg = load().b2rl_last_error().decode()
    if rc == -1:
        raise ValueError(msg)
    if rc == -3:
        raise NotImplementedError(msg)
    raise B2RLError(msg)


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr(device=None) -> int:
    """cudaStream_t of torch's current stream on ``device`` (hot: called before every C-ABI launch)."""
    if _raw_stream is not None:
        if device is None:
            idx = torch.cuda.current_device()
        else:
            idx = device.index if isinstance(device, torch.device) else torch.device(device).index
            if idx is None:
                idx = torch.cuda.current_device()
        return _raw_stream(idx)
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda_tensor(t: torch.Tensor, what: str = "tensor") -> None:
    if not t.is_cuda:
        raise B2RLError(f"{what} must live on a CUDA device (got {t.device}); there is no CPU path.")


def as_device(device) -> torch.device:
    d = torch.device(device)
    if d.type != "cuda":
        raise B2RLError(
            f"agilerl_b200 runs on CUDA devices only (got device={device!r}); there is no CPU fallback."
        )
    load(require_cuda=True)
    cur = torch.cuda.current_device()
    if d.index is None:
        d = torch.device("cuda", cur)
    elif d.index != cur:
        # the library keeps per-process side streams / kernel attributes for ONE device and launches on the current
        # one: a buffer or agent elsewhere would fail later with an invalid resource handle
        raise B2RLError(f"device {d} is not the current CUDA device (cuda:{cur}): agilerl_b200 drives one GPU per process; "
                        "call torch.cuda.set_device first")
    return d
