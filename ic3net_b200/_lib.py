"""ctypes binding of libic3net_b200.so (C ABI: include/ic3net_b200.h).

There is NO CPU fallback: if the shared library is missing, or a call returns a
non-zero status, this module raises.  PyTorch tensors are only the container for
device memory; the structs below carry their ``data_ptr()``s.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libic3net_b200.so")

MAX_AGENTS = 32
MAX_HEADS = 4
MAX_HEAD_DIM = 16
MAX_PASSES = 4
CELL_LSTM, CELL_TANH = 0, 1
LSTM_IMG_BYTES = 786432

ERR_EPISODE_DONE = 1
ERR_ROUTE_OVERRUN = 2
ERR_BAD_ACTION = 4
ERR_PIPELINE = 0x100
ERR_FP16_RANGE = 0x200

PP_MODES = {"mixed": 0, "cooperative": 1, "competitive": 2}

_p = C.c_void_p


class PPCfg(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("dim", C.c_int32), ("vision", C.c_int32),
                ("mode", C.c_int32), ("naction", C.c_int32), ("env_id0", C.c_uint32), ("enemy_comm", C.c_int32),
                ("seed", C.c_uint64)]


class PPState(C.Structure):
    _fields_ = [("loc", _p), ("reached", _p), ("done", _p), ("success", _p), ("episode", _p), ("tick", _p)]


class RolloutIO(C.Structure):
    _fields_ = [("t", C.c_int32), ("max_steps", C.c_int32), ("nheads", C.c_int32), ("hard_attn", C.c_int32),
                ("comm_action_one", C.c_int32), ("last", C.c_int32), ("action", _p), ("t_ep", _p), ("fresh", _p),
                ("comm_next", _p), ("alive_next", _p), ("rec_reward", _p), ("rec_episode_mask", _p),
                ("rec_mini_mask", _p), ("rec_alive", _p), ("stat_reward", _p), ("stat_comm", _p),
                ("stat_success", _p), ("stat_episodes", _p), ("stat_steps", _p), ("batch_size", C.c_int32),
                ("reserved0", C.c_int32), ("halted", _p), ("rec_valid", _p), ("snap_T", C.c_int32),
                ("reserved1", C.c_int32), ("snap_fresh", _p), ("snap_comm", _p), ("snap_alive", _p), ("snap_tep", _p),
                ("snap_pp_loc", _p), ("snap_tj_loc", _p), ("snap_tj_alive", _p), ("snap_tj_last_act", _p),
                ("snap_tj_route_id", _p)]


class TJCfg(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("vision", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
                ("G", C.c_int32), ("P", C.c_int32), ("Lmax", C.c_int32), ("outside_cls", C.c_int32),
                ("car_cls", C.c_int32), ("vocab", C.c_int32), ("npath", C.c_int32), ("spawn_thr", C.c_uint32),
                ("env_id0", C.c_uint32), ("seed", C.c_uint64), ("grid", _p), ("route_len", _p), ("route_cells", _p)]


class TJState(C.Structure):
    _fields_ = [("loc", _p), ("alive", _p), ("wait", _p), ("route_id", _p), ("route_pos", _p), ("last_act", _p),
                ("completed", _p), ("cars_in_sys", _p), ("has_failed", _p), ("tick", _p)]


class PolicyCfg(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("H", C.c_int32), ("O", C.c_int32), ("nheads", C.c_int32),
                ("head_dim", C.c_int32 * MAX_HEADS), ("hard_attn", C.c_int32), ("comm_avg", C.c_int32),
                ("comm_mask_zero", C.c_int32), ("env_id0", C.c_uint32), ("seed", C.c_uint64),
                ("obs_off", C.c_int32), ("obs_vocab", C.c_int32), ("obs_ncount", C.c_int32), ("cell", C.c_int32),
                ("passes", C.c_int32), ("x_tanh", C.c_int32), ("h_from_x", C.c_int32), ("reserved0", C.c_int32)]


class PolicyParams(C.Structure):
    _fields_ = [("encoder_w", _p), ("encoder_b", _p), ("c_w", _p), ("c_b", _p), ("w_ih", _p), ("w_hh", _p),
                ("b_ih", _p), ("b_hh", _p), ("value_w", _p), ("value_b", _p),
                ("head_w", _p * MAX_HEADS), ("head_b", _p * MAX_HEADS), ("c_w_pass", _p * MAX_PASSES),
                ("c_b_pass", _p * MAX_PASSES), ("f_w_pass", _p * MAX_PASSES), ("f_b_pass", _p * MAX_PASSES)]


class PolicyPacked(C.Structure):
    _fields_ = [("enc_wT", _p), ("enc_b", _p), ("c_wT", _p), ("c_b", _p), ("lstm_wT", _p), ("lstm_b", _p),
                ("head_w", _p), ("head_b", _p), ("lstm_img", _p), ("bias_cat", _p), ("f_wT", _p), ("f_b", _p), ("flags", _p)]


class PolicyIO(C.Structure):
    _fields_ = [("x", _p), ("h", _p), ("c", _p), ("comm_action", _p), ("alive", _p), ("fresh", _p), ("tick", _p),
                ("draws", _p), ("h_out", _p), ("c_out", _p), ("value", _p), ("logp", _p), ("action", _p),
                ("workspace", _p), ("err", _p), ("pp_env", _p), ("pp_state", _p), ("tj_env", _p), ("tj_state", _p),
                ("x_table", _p), ("pass_index", C.c_int32)]


class BpttPlan(C.Structure):
    _fields_ = [("cfg", C.POINTER(PolicyCfg)), ("w", C.POINTER(PolicyPacked)), ("pp_env", C.POINTER(PPCfg)),
                ("tj_env", C.POINTER(TJCfg)), ("x_table", _p), ("value_coeff", C.c_float), ("entr", C.c_float),
                ("workspace", _p)]


class BpttStepIO(C.Structure):
    _fields_ = [("t", C.c_int32), ("reserved0", C.c_int32), ("h_prev", _p), ("c_prev", _p), ("h_new", _p), ("fresh", _p), ("comm", _p), ("alive", _p), ("cut", _p),
                ("pp_loc", _p), ("tj_loc", _p), ("tj_alive", _p), ("tj_last_act", _p), ("tj_route_id", _p),
                ("logp", _p), ("action", _p), ("value", _p), ("ret", _p), ("adv", _p), ("alive_post", _p),
                ("valid", _p), ("dh", _p), ("dc", _p), ("err", _p)]


# every symbol include/ic3net_b200.h declares: name -> (restype, argtypes)
_PTR = C.c_void_p
SYMBOLS = {
    "ic3_version": (C.c_char_p, []),
    "ic3_strerror": (C.c_char_p, [C.c_int]),
    "ic3_launch_count": (C.c_uint64, []),
    "ic3_pp_reset": (C.c_int, [C.POINTER(PPCfg), C.POINTER(PPState), _PTR, _PTR, _PTR]),
    "ic3_pp_step": (C.c_int, [C.POINTER(PPCfg), C.POINTER(PPState), _PTR, C.c_int32, _PTR, _PTR, _PTR,
                              C.POINTER(RolloutIO), _PTR]),
    "ic3_pp_obs": (C.c_int, [C.POINTER(PPCfg), C.POINTER(PPState), _PTR, _PTR]),
    "ic3_tj_reset": (C.c_int, [C.POINTER(TJCfg), C.POINTER(TJState), _PTR, _PTR, _PTR]),
    "ic3_tj_step": (C.c_int, [C.POINTER(TJCfg), C.POINTER(TJState), _PTR, C.c_int32, _PTR, _PTR, _PTR, _PTR,
                              C.POINTER(RolloutIO), _PTR]),
    "ic3_tj_obs": (C.c_int, [C.POINTER(TJCfg), C.POINTER(TJState), _PTR, _PTR]),
    "ic3_policy_pack": (C.c_int, [C.POINTER(PolicyCfg), C.POINTER(PolicyParams), C.POINTER(PolicyPacked), _PTR]),
    "ic3_encoder_dense": (C.c_int, [C.POINTER(PolicyCfg), C.POINTER(PolicyPacked), _PTR, _PTR, _PTR]),
    "ic3_pp_encoder_index": (C.c_int, [C.POINTER(PPCfg), C.POINTER(PPState), C.POINTER(PolicyCfg),
                                       C.POINTER(PolicyPacked), _PTR, _PTR]),
    "ic3_tj_encoder_index": (C.c_int, [C.POINTER(TJCfg), C.POINTER(TJState), C.POINTER(PolicyCfg),
                                       C.POINTER(PolicyPacked), _PTR, _PTR]),
    "ic3_pp_encoder_table": (C.c_int, [C.POINTER(PPCfg), C.POINTER(PolicyCfg), C.POINTER(PolicyPacked), _PTR, _PTR]),
    "ic3_tj_encoder_table": (C.c_int, [C.POINTER(TJCfg), C.POINTER(PolicyCfg), C.POINTER(PolicyPacked), _PTR, _PTR]),
    "ic3_policy_workspace_bytes": (C.c_uint64, [C.POINTER(PolicyCfg)]),
    "ic3_policy_step": (C.c_int, [C.POINTER(PolicyCfg), C.POINTER(PolicyPacked), C.POINTER(PolicyIO), _PTR]),
    "ic3_policy_step_profile": (C.c_int, [C.POINTER(PolicyCfg), C.POINTER(PolicyPacked), C.POINTER(PolicyIO), _PTR,
                                          C.POINTER(C.c_float)]),
    "ic3_sample_actions": (C.c_int, [C.POINTER(PolicyCfg), _PTR, _PTR, _PTR, _PTR, _PTR]),
    "ic3_returns_scan": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float, _PTR, _PTR, _PTR, _PTR,
                                   _PTR]),
    "ic3_bptt_workspace_bytes": (C.c_uint64, [C.POINTER(BpttPlan)]),
    "ic3_bptt_begin": (C.c_int, [C.POINTER(BpttPlan), C.c_float, _PTR]),
    "ic3_bptt_step": (C.c_int, [C.POINTER(BpttPlan), C.POINTER(BpttStepIO), _PTR]),
    "ic3_bptt_prepare": (C.c_int, [C.POINTER(BpttPlan), C.POINTER(BpttStepIO), _PTR]),
    "ic3_bptt_finish": (C.c_int, [C.POINTER(BpttPlan), C.POINTER(PolicyParams), C.POINTER(PolicyParams), _PTR, _PTR]),
    "ic3_stat_reduce": (C.c_int, [C.c_int32, C.c_int32, _PTR, _PTR, _PTR, _PTR, _PTR, _PTR, _PTR, _PTR]),
    "ic3_rmsprop_step": (C.c_int, [C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, _PTR, _PTR, _PTR, _PTR]),
}

_lib = None


def load():
    """Load the CUDA library or raise (never falls back to a CPU path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("ic3net_b200: %s not found; run `python -m ic3net_b200.build` "
                           "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError("ic3net_b200 call failed (%d): %s" % (rc, load().ic3_strerror(rc).decode()))


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "ic3net_b200 needs contiguous CUDA tensors"
    return t.data_ptr()


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream():
    """cudaStream_t of torch's current stream on the current device (honours stream / graph-capture contexts)."""
    if _raw_stream is not None:          # one C call instead of building a torch.cuda.Stream object per launch
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("ic3net_b200 runs on a CUDA device only (no CPU fallback)")
    load()


def launch_count():
    return int(load().ic3_launch_count())
