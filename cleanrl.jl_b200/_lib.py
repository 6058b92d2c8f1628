"""ctypes binding of libcleanrl_cuda.so (include/cleanrl_cuda.h).

The library is loaded lazily and there is NO fallback: if the .so is missing, or no sm_100
GPU is usable, the first compute call raises. The host side never routes work to a CPU path.
"""
import ctypes as C
import os

import numpy as np

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcleanrl_cuda.so")
_lib = None


class CleanRLCudaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libcleanrl_cuda error %d: %s" % (code, msg))
        self.code = code


V, I32, I64, F32, F64, U64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double, C.c_uint64

# every symbol include/cleanrl_cuda.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "crl_version": (C.c_int, []),
    "crl_last_error": (C.c_char_p, []),
    "crl_device_count": (C.c_int, [V]),
    "crl_create": (C.c_int, [C.POINTER(_abi.crl_config), C.POINTER(V)]),
    "crl_destroy": (C.c_int, [V]),
    "crl_sync": (C.c_int, [V]),
    "crl_dims": (C.c_int, [V, V, V, V, V, V]),
    "crl_param_layout": (C.c_int, [V, V, V, I32]),
    "crl_set_params": (C.c_int, [V, V, I32]),
    "crl_get_params": (C.c_int, [V, V, I32]),
    "crl_get_grads": (C.c_int, [V, V, I32]),
    "crl_get_adam_state": (C.c_int, [V, V, V, V]),
    "crl_set_adam_state": (C.c_int, [V, V, V, V]),
    "crl_env_reset": (C.c_int, [V]),
    "crl_env_set_state": (C.c_int, [V, V, V]),
    "crl_rollout": (C.c_int, [V, V, V]),
    "crl_gae": (C.c_int, [V]),
    "crl_update_minibatch": (C.c_int, [V, V, I32, F64, V]),
    "crl_update_epochs": (C.c_int, [V, V, F64, V]),
    "crl_device_permutation": (C.c_int, [V, I64, I32, V]),
    "crl_train_update": (C.c_int, [V, F64]),
    "crl_fetch_update": (C.c_int, [V, V, V]),
    "crl_fetch_update_at": (C.c_int, [V, I32, V, V]),
    "crl_read_field": (C.c_int, [V, I32, V, C.c_size_t]),
    "crl_write_field": (C.c_int, [V, I32, V, C.c_size_t]),
    "crl_pop_episodes": (C.c_int, [V, V, I32, V, V]),
    "crl_comm_unique_id": (C.c_int, [V]),
    "crl_comm_init": (C.c_int, [V, V]),
    "crl_kernel_launches": (C.c_int, [V, V]),
    "crl_spec_replays": (C.c_int, [V, V]),
    "crl_profile": (C.c_int, [V, I32]),
    "crl_profile_read": (C.c_int, [V, V, I32]),
    "crl_stream": (C.c_int, [V, V]),
    "crl_gae_raw": (C.c_int, [V] * 7 + [I32, I64, F32, F32, I32, V]),
    "crl_env_step_raw": (C.c_int, [I32, V, V, V, V, V, I64, I32, V]),
    "crl_policy_forward_raw": (C.c_int, [I32, V, V, V, V, V, I64, V]),
    "crl_ppo_loss_raw": (C.c_int, [I32, V, V, I32] + [V] * 6 + [F32] * 3 + [V, V, V]),
    "crl_clip_adam_raw": (C.c_int, [I32, V, V, V, V, V, F64, F32, V]),
    "crl_dqn_create": (C.c_int, [C.POINTER(_abi.crl_dqn_config), C.POINTER(V)]),
    "crl_dqn_destroy": (C.c_int, [V]),
    "crl_dqn_set_params": (C.c_int, [V, V, I32]),
    "crl_dqn_get_params": (C.c_int, [V, V, V, I32]),
    "crl_dqn_reset": (C.c_int, [V]),
    "crl_dqn_run": (C.c_int, [V, I64, V]),
    "crl_dqn_comm_init": (C.c_int, [V, V, I32, I32, I32]),
    "crl_dqn_read_buffer": (C.c_int, [V] * 8),
    "crl_dqn_forward_raw": (C.c_int, [V, V, V, I64, V]),
    "crl_dqn_loss_raw": (C.c_int, [V, V, I32] + [V] * 5 + [F64, V, V, V]),
    "crl_tb_open": (C.c_int, [C.c_char_p, C.POINTER(V)]),
    "crl_tb_scalars": (C.c_int, [V, F64, I64, I32, C.c_char_p, V]),
    "crl_tb_flush": (C.c_int, [V]),
    "crl_tb_close": (C.c_int, [V]),
}

# every symbol include/cleanrl_ddpg.h declares (the DDPG handle and its raw kernels)
DDPG_SIGNATURES = {
    "crl_ddpg_create": (C.c_int, [C.POINTER(_abi.crl_ddpg_config), C.POINTER(V)]),
    "crl_ddpg_destroy": (C.c_int, [V]),
    "crl_ddpg_set_params": (C.c_int, [V, V, I32, V, I32]),
    "crl_ddpg_get_params": (C.c_int, [V, V, V, V, V]),
    "crl_ddpg_get_adam_state": (C.c_int, [V, V, V, V, V, V]),
    "crl_ddpg_reset": (C.c_int, [V]),
    "crl_ddpg_run": (C.c_int, [V, I64, V]),
    "crl_ddpg_read_buffer": (C.c_int, [V] * 8),
    "crl_ddpg_forward_raw": (C.c_int, [V] * 6 + [I64, V]),
    "crl_ddpg_critic_loss_raw": (C.c_int, [V, V, V, I32] + [V] * 5 + [F64, V, V, V]),
    "crl_ddpg_actor_loss_raw": (C.c_int, [V, V, I32, V, V, V, V]),
}

# every symbol include/cleanrl_td3.h declares (the TD3 handle and its raw critic step)
TD3_SIGNATURES = {
    "crl_td3_create": (C.c_int, [C.POINTER(_abi.crl_td3_config), C.POINTER(V)]),
    "crl_td3_destroy": (C.c_int, [V]),
    "crl_td3_set_params": (C.c_int, [V, V, I32, V, I32, V, I32]),
    "crl_td3_get_params": (C.c_int, [V] * 7),
    "crl_td3_get_adam_state": (C.c_int, [V] * 8),
    "crl_td3_reset": (C.c_int, [V]),
    "crl_td3_run": (C.c_int, [V, I64, V]),
    "crl_td3_read_buffer": (C.c_int, [V] * 8),
    "crl_td3_critic_loss_raw": (C.c_int, [V] * 5 + [I32] + [V] * 5 + [F64, F64, F64, U64, U64] + [V] * 5),
}

# every symbol include/cleanrl_sac.h declares (the SAC handle and its raw kernels)
SAC_SIGNATURES = {
    "crl_sac_create": (C.c_int, [C.POINTER(_abi.crl_sac_config), C.POINTER(V)]),
    "crl_sac_destroy": (C.c_int, [V]),
    "crl_sac_set_params": (C.c_int, [V, V, I32, V, I32, V, I32]),
    "crl_sac_get_params": (C.c_int, [V] * 7),
    "crl_sac_get_adam_state": (C.c_int, [V] * 9),
    "crl_sac_reset": (C.c_int, [V]),
    "crl_sac_run": (C.c_int, [V, I64, V]),
    "crl_sac_read_buffer": (C.c_int, [V] * 8),
    "crl_sac_forward_raw": (C.c_int, [V] * 7 + [I64, V]),
    "crl_sac_critic_loss_raw": (C.c_int, [V] * 5 + [I32] + [V] * 5 + [F64, F64, U64, U64] + [V] * 5),
    "crl_sac_actor_loss_raw": (C.c_int, [V, V, V, I32, V, F64, U64, U64, V, V, V, V]),
}

# every symbol include/cleanrl_c51.h declares (the C51 handle and its raw kernels)
C51_SIGNATURES = {
    "crl_c51_create": (C.c_int, [C.POINTER(_abi.crl_c51_config), C.POINTER(V)]),
    "crl_c51_destroy": (C.c_int, [V]),
    "crl_c51_set_params": (C.c_int, [V, V, I32]),
    "crl_c51_get_params": (C.c_int, [V, V, V, I32]),
    "crl_c51_get_adam_state": (C.c_int, [V, V, V, V]),
    "crl_c51_reset": (C.c_int, [V]),
    "crl_c51_run": (C.c_int, [V, I64, V]),
    "crl_c51_read_buffer": (C.c_int, [V] * 8),
    "crl_c51_forward_raw": (C.c_int, [V, V, F64, F64, V, V, V, I64, V]),
    "crl_c51_loss_raw": (C.c_int, [V, V, I32] + [V] * 5 + [F64, F64, F64, V, V, V, V]),
}


def load():
    """dlopen the CUDA library and bind every entry point. Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CleanRLCudaError(-2, "%s is not built (run `python cleanrl.jl_b200/build.py` or "
                                   "__graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in list(SIGNATURES.items()) + list(DDPG_SIGNATURES.items()) + list(TD3_SIGNATURES.items()) + \
            list(SAC_SIGNATURES.items()) + list(C51_SIGNATURES.items()):
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.crl_version() != _abi.CRL_VERSION:
        raise CleanRLCudaError(-1, "version mismatch: library %d, binding %d" % (lib.crl_version(), _abi.CRL_VERSION))
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().crl_last_error()
        raise CleanRLCudaError(rc, msg.decode() if msg else "?")


def ptr(a):
    """host numpy array / torch tensor / int address -> void*"""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    return a


def device_count():
    n = C.c_int32()
    check(load().crl_device_count(C.byref(n)))
    return n.value
