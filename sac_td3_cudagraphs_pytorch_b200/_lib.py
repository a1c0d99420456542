"""ctypes binding of libb2rl.so (include/b2rl.h). There is NO fallback: if the library cannot be
loaded (or built with nvcc when absent) importing the update path raises."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

HID = 256
ROWS = 8  # batch rows per CTA group of the fused kernels (a batch need not be a multiple)
MAX_OUT = 64
MAX_SEG = 8
CTR_Q, CTR_PI, CTR_ALPHA, CTR_SAMPLE, CTR_TICKET, CTR_SIZE, CTR_CURSOR, CTR_XTICKET = 0, 1, 2, 3, 4, 5, 6, 7
OUT_QF_LOSS, OUT_ACTOR_LOSS, OUT_ALPHA_LOSS, OUT_ALPHA, OUT_LOGPI_MEAN = 0, 1, 2, 3, 4
REGION_P, REGION_T, REGION_M, REGION_V, REGION_G = range(5)


class Net(C.Structure):
    _fields_ = [("in_dim", C.c_int32), ("out_dim", C.c_int32), ("layer_norm", C.c_int32), ("reserved", C.c_int32),
                ("w1t", C.c_int64), ("b1", C.c_int64), ("g1", C.c_int64), ("be1", C.c_int64),
                ("w2t", C.c_int64), ("b2", C.c_int64), ("g2", C.c_int64), ("be2", C.c_int64),
                ("w3", C.c_int64), ("b3", C.c_int64), ("w2n", C.c_int64),
                ("begin", C.c_int64), ("end", C.c_int64)]


class RowFmt(C.Structure):
    _fields_ = [("ob_dim", C.c_int32), ("ac_dim", C.c_int32), ("row_stride", C.c_int32), ("reserved", C.c_int32)]


class Hyper(C.Structure):
    _fields_ = [("td3", C.c_int32), ("bcq_mix", C.c_int32), ("targ_smoothing", C.c_int32), ("autotune", C.c_int32),
                ("gamma", C.c_float), ("td3_std", C.c_float), ("td3_c", C.c_float), ("targ_ent", C.c_float),
                ("seed", C.c_uint64)]


class AgentHp(C.Structure):
    """b2rl_agent_hp_t: one 64-byte row of per-agent hyperparameters (lr indexed by CTR_Q / CTR_PI / CTR_ALPHA)."""
    _fields_ = [("lr", C.c_float * 3), ("gamma", C.c_float), ("polyak", C.c_float), ("td3_std", C.c_float),
                ("td3_c", C.c_float), ("targ_ent", C.c_float), ("clip_norm", C.c_float), ("explore_std", C.c_float),
                ("reserved", C.c_float * 6)]


class UpdateArgs(C.Structure):
    _fields_ = [("hp", Hyper), ("fmt", RowFmt), ("actor", Net), ("critic", Net * 2),
                ("batch", C.c_int32), ("n_agents", C.c_int32), ("agent_base", C.c_int32), ("reserved", C.c_int32),
                ("region_stride", C.c_int64), ("arena_agent_stride", C.c_int64),
                ("arena", C.c_void_p), ("rows", C.c_void_p), ("rows_agent_stride", C.c_int64),
                ("min_ac", C.c_void_p), ("max_ac", C.c_void_p), ("log_alpha", C.c_void_p),
                ("eps", C.c_void_p), ("eps2", C.c_void_p), ("eps_out", C.c_void_p), ("eps2_out", C.c_void_p),
                ("counters", C.c_void_p), ("workspace", C.c_void_p), ("workspace_agent_stride", C.c_int64),
                ("out", C.c_void_p), ("dbg_targ_q", C.c_void_p), ("dbg_q", C.c_void_p),
                ("storage", C.c_void_p), ("storage_agent_stride", C.c_int64), ("storage_size", C.c_int64),
                ("idx_out", C.c_void_p), ("new_rows", C.c_void_p), ("capacity", C.c_int64), ("n_new", C.c_int32),
                ("reserved2", C.c_int32), ("agent_hp", C.c_void_p)]


class Seg(C.Structure):
    _fields_ = [("begin", C.c_int64), ("end", C.c_int64), ("lr", C.c_float), ("do_adam", C.c_int32),
                ("do_polyak", C.c_int32), ("counter", C.c_int32), ("grad_scale", C.c_float), ("clip", C.c_int32)]


class AdamArgs(C.Structure):
    _fields_ = [("seg", Seg * MAX_SEG), ("n_seg", C.c_int32), ("n_agents", C.c_int32),
                ("polyak", C.c_float), ("clip_norm", C.c_float),
                ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("reserved", C.c_int32),
                ("region_stride", C.c_int64), ("arena_agent_stride", C.c_int64),
                ("arena", C.c_void_p), ("counters", C.c_void_p), ("grad_sumsq", C.c_void_p), ("lo", C.c_void_p), ("lo_agent_stride", C.c_int64),
                ("shadow_src", C.c_int64 * 3), ("shadow_dst", C.c_int64 * 3), ("n_shadow", C.c_int32), ("reserved2", C.c_int32),
                ("agent_hp", C.c_void_p)]


class WidePolicy(C.Structure):
    _fields_ = [("h2", C.c_void_p), ("w3", C.c_void_p), ("b3", C.c_void_p), ("rows", C.c_void_p), ("min_ac", C.c_void_p),
                ("max_ac", C.c_void_p), ("eps", C.c_void_p), ("eps_out", C.c_void_p), ("xn", C.c_void_p), ("logp", C.c_void_p),
                ("save", C.c_void_p), ("counters", C.c_void_p),
                ("M", C.c_int32), ("O", C.c_int32), ("A", C.c_int32), ("out_dim", C.c_int32), ("row_stride", C.c_int32),
                ("ldn", C.c_int32), ("src_off", C.c_int32), ("td3", C.c_int32), ("smoothing", C.c_int32),
                ("counter_idx", C.c_int32), ("stream_id", C.c_int32), ("td3_std", C.c_float), ("td3_c", C.c_float),
                ("seed", C.c_uint64), ("agent", C.c_uint32), ("reserved", C.c_uint32)]


class WidePredict(C.Structure):
    """b2rl_wide_predict_t"""
    _fields_ = [("h2", C.c_void_p), ("w3", C.c_void_p), ("b3", C.c_void_p), ("min_ac", C.c_void_p), ("max_ac", C.c_void_p),
                ("eps", C.c_void_p), ("eps_out", C.c_void_p), ("actions", C.c_void_p), ("counters", C.c_void_p),
                ("agent_hp", C.c_void_p), ("n", C.c_int32), ("A", C.c_int32), ("out_dim", C.c_int32), ("mode", C.c_int32),
                ("td3", C.c_int32), ("explore_std", C.c_float), ("seed", C.c_uint64), ("draw", C.c_uint64),
                ("agent", C.c_uint32), ("reserved", C.c_uint32)]


class WideQ(C.Structure):
    _fields_ = [("h2", C.c_void_p), ("w3", C.c_void_p), ("b3", C.c_void_p), ("q_out", C.c_void_p), ("qn0", C.c_void_p),
                ("qn1", C.c_void_p), ("logp", C.c_void_p), ("rows", C.c_void_p), ("log_alpha", C.c_void_p), ("dz3", C.c_void_p),
                ("sq_part", C.c_void_p), ("targ_out", C.c_void_p),
                ("M", C.c_int32), ("mode", C.c_int32), ("row_stride", C.c_int32), ("rd_off", C.c_int32), ("td3", C.c_int32),
                ("bcq_mix", C.c_int32), ("gamma", C.c_float), ("reserved", C.c_uint32)]


class ColsumJob(C.Structure):
    """b2rl_colsum_job_t"""
    _fields_ = [("part", C.c_void_p), ("off_b", C.c_int64), ("off_g", C.c_int64), ("off_be", C.c_int64),
                ("layer_norm", C.c_int32), ("reserved", C.c_int32)]


class Stack(C.Structure):
    """b2rl_stack_t: agents stacked along the row dimension of the wide path (NULL = one learner)."""
    _fields_ = [("n_agents", C.c_int32), ("agent_base", C.c_int32), ("param_stride", C.c_int64), ("lo_stride", C.c_int64),
                ("alpha_stride", C.c_int64), ("counters_stride", C.c_int64), ("out_stride", C.c_int64), ("agent_hp", C.c_void_p)]


_STK = C.POINTER(Stack)

# name -> (restype, argtypes); every symbol include/b2rl.h declares
SYMBOLS = {
    "b2rl_version": (C.c_int, []),
    "b2rl_last_error": (C.c_char_p, []),
    "b2rl_init": (C.c_int, []),
    "b2rl_workspace_floats": (C.c_int64, [C.c_int32]),
    "b2rl_replay_sample_gather": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, RowFmt, C.c_int32, C.c_int32,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                            C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "b2rl_replay_extend": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, RowFmt, C.c_void_p, C.c_int32, C.c_void_p]),
    "b2rl_replay_extend_dev": (C.c_int, [C.c_void_p, C.c_int64, RowFmt, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "b2rl_replay_extend_dev_stack": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, RowFmt, C.c_void_p, C.c_int32, C.c_int32,
                                               C.c_void_p, C.c_void_p]),
    "b2rl_critic_update_sac": (C.c_int, [C.POINTER(UpdateArgs), C.c_void_p]),
    "b2rl_critic_update_td3": (C.c_int, [C.POINTER(UpdateArgs), C.c_void_p]),
    "b2rl_actor_update_sac": (C.c_int, [C.POINTER(UpdateArgs), C.c_void_p]),
    "b2rl_actor_update_td3": (C.c_int, [C.POINTER(UpdateArgs), C.c_void_p]),
    "b2rl_tc_linear": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_tc_linear_q": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_tc_split_lo": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, _STK, C.c_void_p]),
    "b2rl_wide_first": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_tc_first": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, _STK, C.c_void_p]),
    "b2rl_tc_linear_bwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_void_p, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_wide_policy_head": (C.c_int, [C.POINTER(WidePolicy), _STK, C.c_void_p]),
    "b2rl_wide_actor_predict": (C.c_int, [C.POINTER(WidePredict), C.c_void_p]),
    "b2rl_copy_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "b2rl_wide_q_head": (C.c_int, [C.POINTER(WideQ), _STK, C.c_void_p]),
    "b2rl_wide_ln_bwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                  C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_wide_colsum_multi": (C.c_int, [C.POINTER(ColsumJob), C.c_int32, C.c_int32, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_wide_colsum": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _STK, C.c_void_p]),
    "b2rl_wide_critic_scalars": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                          C.c_int64, C.c_int64, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_wide_actor_loss": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, _STK, C.c_void_p]),
    "b2rl_wide_dqda": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_wide_actor_head_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                          C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_wide_actor_scalars": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                         C.c_void_p, C.c_int64, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_wide_alpha_grad": (C.c_int, [C.c_void_p, C.c_int32, C.c_float, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_tc_wgrad": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_int32, C.c_void_p, _STK, C.c_void_p]),
    "b2rl_tc_wgrad_scratch_floats": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "b2rl_wgrad": (C.c_int, [C.POINTER(UpdateArgs), C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "b2rl_publish_logs": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2rl_critic_update_opt": (C.c_int, [C.POINTER(UpdateArgs), C.POINTER(AdamArgs), C.c_void_p]),
    "b2rl_actor_update_opt": (C.c_int, [C.POINTER(UpdateArgs), C.POINTER(AdamArgs), C.c_void_p]),
    "b2rl_alpha_update": (C.c_int, [C.POINTER(UpdateArgs), C.c_float, C.c_void_p]),
    "b2rl_alpha_adam": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float, C.c_void_p, C.c_void_p]),
    "b2rl_alpha_adam_hp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]),
    "b2rl_grad_sumsq": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int32,
                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2rl_adam_polyak_multi": (C.c_int, [C.POINTER(AdamArgs), C.c_void_p]),
    "b2rl_bump_counter": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "b2rl_actor_predict": (C.c_int, [C.POINTER(UpdateArgs), C.c_void_p, C.c_int32, C.c_int32, C.c_float,
                                     C.c_uint64, C.c_void_p, C.c_void_p]),
    "b2rl_launch_single": (C.c_int, [C.POINTER(UpdateArgs), C.c_int32, C.c_void_p]),
    "b2rl_ffma_probe": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_double), C.c_void_p]),
}

LIB_PATH = Path(os.environ.get("B2RL_LIB") or Path(__file__).resolve().parent / "libb2rl.so")
_lib = None


class B2rlError(RuntimeError):
    pass


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first if the .so is absent and nvcc exists). Raises — never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if not build_if_missing:
            raise B2rlError(f"{LIB_PATH} is missing; run `python -m sac_td3_cudagraphs_pytorch_b200.build`")
        from .build import build_lib
        build_lib()
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError here = header and library disagree
        fn.restype, fn.argtypes = res, args
    if lib.b2rl_version() != 111:
        raise B2rlError(f"libb2rl version {lib.b2rl_version()} does not match the binding (111)")
    _lib = lib
    return lib


_inited = set()


def init_device(device) -> None:
    """b2rl_init() once per process and device (needs a live CUDA context)."""
    import torch
    dev = torch.device(device)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if idx in _inited:
        return
    with torch.cuda.device(idx):
        torch.zeros(1, device=dev)  # make sure the primary context exists
        check(load().b2rl_init(), "b2rl_init")
    _inited.add(idx)


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().b2rl_last_error().decode(errors="replace")
        raise B2rlError(f"{what or 'libb2rl'} failed ({rc}): {msg}")


def ptr(t) -> int | None:
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
