"""ctypes binding of libcednerf_b200.so (include/cednerf_b200.h).

The library is the product: there is no CPU or PyTorch fallback.  If the shared object is missing the
import fails loudly with the build command; every op additionally refuses non-CUDA tensors.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# CEDNERF_B200_LIB: an instrumented build of the same library (make -C cednerf_b200/csrc debug), for profiles/tools only
LIB_PATH = os.environ.get("CEDNERF_B200_LIB") or os.path.join(_HERE, "libcednerf_b200.so")

MAX_LEVELS = 32
MLP_MAX_LAYERS = 5


class GridLevels(ctypes.Structure):
    _fields_ = [("n_levels", ctypes.c_int), ("scale", ctypes.c_float * MAX_LEVELS),
                ("res", ctypes.c_uint32 * MAX_LEVELS), ("size", ctypes.c_uint32 * MAX_LEVELS),
                ("offset", ctypes.c_uint32 * MAX_LEVELS), ("hashed", ctypes.c_uint32 * MAX_LEVELS)]


class MlpDesc(ctypes.Structure):
    _fields_ = [("n_layers", ctypes.c_int), ("dim_in", ctypes.c_int * MLP_MAX_LAYERS),
                ("dim_out", ctypes.c_int * MLP_MAX_LAYERS), ("param_off", ctypes.c_int * MLP_MAX_LAYERS),
                ("image_off", ctypes.c_int * MLP_MAX_LAYERS), ("image_bytes", ctypes.c_int)]


class FieldDesc(ctypes.Structure):
    _fields_ = [("aabb", ctypes.c_float * 6), ("moving_step", ctypes.c_float), ("use_div_offsets", ctypes.c_int),
                ("time_mode", ctypes.c_int), ("time_before_sigma", ctypes.c_int), ("f1", MlpDesc), ("f2", MlpDesc),
                ("f3", MlpDesc), ("f4", MlpDesc), ("levels", GridLevels)]


OPT_MAX_TENSORS = 8


class AdamTensors(ctypes.Structure):
    _fields_ = [("n_tensors", ctypes.c_int), ("p", ctypes.c_void_p * OPT_MAX_TENSORS),
                ("g", ctypes.c_void_p * OPT_MAX_TENSORS), ("m", ctypes.c_void_p * OPT_MAX_TENSORS),
                ("v", ctypes.c_void_p * OPT_MAX_TENSORS), ("p16", ctypes.c_void_p * OPT_MAX_TENSORS),
                ("n", ctypes.c_int64 * OPT_MAX_TENSORS), ("lr", ctypes.c_float * OPT_MAX_TENSORS),
                ("weight_decay", ctypes.c_float * OPT_MAX_TENSORS),
                ("chunk_begin", ctypes.c_int64 * (OPT_MAX_TENSORS + 1))]


DP_MAX_RANKS = 8


class DpCtrl(ctypes.Structure):
    _fields_ = [("arrive", ctypes.c_uint32 * DP_MAX_RANKS), ("found_inf", ctypes.c_float), ("timed_out", ctypes.c_uint32)]


class DpPeers(ctypes.Structure):
    _fields_ = [("world", ctypes.c_int), ("rank", ctypes.c_int), ("ctrl", ctypes.c_void_p * DP_MAX_RANKS)]


class DpAdam(ctypes.Structure):
    _fields_ = [("world", ctypes.c_int), ("rank", ctypes.c_int), ("grad", ctypes.c_void_p * DP_MAX_RANKS),
                ("n_out", ctypes.c_int), ("p32_out", ctypes.c_void_p * DP_MAX_RANKS),
                ("p16_out", ctypes.c_void_p * DP_MAX_RANKS), ("m", ctypes.c_void_p), ("v", ctypes.c_void_p),
                ("lo", ctypes.c_int64), ("hi", ctypes.c_int64), ("lr", ctypes.c_float), ("weight_decay", ctypes.c_float),
                ("grad_div", ctypes.c_float), ("grad_mc", ctypes.c_void_p), ("p16_mc", ctypes.c_void_p)]


class DpSmall(ctypes.Structure):
    _fields_ = [("world", ctypes.c_int), ("n_tensors", ctypes.c_int), ("grad", ctypes.c_void_p * DP_MAX_RANKS),
                ("p", ctypes.c_void_p * 8), ("m", ctypes.c_void_p * 8), ("v", ctypes.c_void_p * 8),
                ("off", ctypes.c_int64 * 8), ("n", ctypes.c_int64 * 8), ("lr", ctypes.c_float * 8),
                ("weight_decay", ctypes.c_float * 8), ("grad_div", ctypes.c_float), ("chunk_begin", ctypes.c_int64 * 9)]


class RenderRound(ctypes.Structure):
    _P, _I, _L, _F = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float
    _fields_ = [("rays_o", _P), ("rays_d", _P), ("n_rays", _L), ("occ_bits", _P), ("aabbs", _P), ("n_levels", _I),
                ("resolution", _I), ("near_term", _P), ("far_const", _F), ("step_size", _F), ("cone_angle", _F),
                ("early_stop_eps", _F), ("t_sorted", _P), ("t_indices", _P), ("hits", _P), ("state", _P), ("total", _P),
                ("n_samples", _P), ("run_t", _P), ("run_n", _P), ("n_runs", _P), ("occ_coarse", _P), ("capacity", _L),
                ("offsets", _P), ("totals", _P), ("scan_workspace", _P), ("t_starts", _P), ("t_ends", _P),
                ("ray_indices", _P), ("overflow", _P), ("timestamps", _P), ("image_deform", _P), ("image_density", _P),
                ("image_colour", _P), ("table_f16", _P), ("desc", ctypes.POINTER(FieldDesc)), ("sigma", _P), ("rgbs", _P),
                ("colors", _P), ("opacity", _P), ("depth", _P), ("alive_flags", _P), ("positions", _P),
                ("position_totals", _P), ("run_cap", _I), ("k_hint", _I), ("max_samples", _I), ("min_samples", _I)]


# p = pointer, i = int, l = int64, f = float, A = AdamTensors*, G = GridLevels*, M = MlpDesc*, F = FieldDesc*
_SIGNATURES = {
    "cednerf_ray_aabb_intersect": "pplpifffpppp",
    "cednerf_sort_boundaries": "pplippp",
    "cednerf_occ_pack_bits": "plpp",
    "cednerf_occ_threshold_pack": "plpppp",
    "cednerf_occ_mark_invisible": "pipiipiiiifpp",
    "cednerf_march": "ipplppiippffffippppppppppppppppppppppippp",
    "cednerf_occ_coarsen": "piipp",
    "cednerf_ray_coherence_keys": "plpp",
    "cednerf_ray_coherence_order": "plppp",
    "cednerf_march_fill_runs": "lppppiffppppp",
    "cednerf_exclusive_scan": "plppppp",
    "cednerf_exclusive_scan_capped": "pllpppp",
    "cednerf_march_fill_runs_capped": "lpppppiffppppp",
    "cednerf_compact_samples_capped": "pppppllpppp",
    "cednerf_hashgrid_fwd": "pilpGpip",
    "cednerf_hashgrid_bwd": "pilpGpiippp",
    "cednerf_hashgrid_bwd_table_lm": "pilGppp",
    "cednerf_hashgrid4d_fwd": "pilpGpiip",
    "cednerf_hashgrid4d_bwd": "pilGpiipip",
    "cednerf_cast_f32_to_f16": "pplp",
    "cednerf_frequency_fwd": "pilipiifp",
    "cednerf_frequency_bwd": "pilipiipp",
    "cednerf_sh2_fwd": "plpip",
    "cednerf_time_embed": "pplpp",
    "cednerf_mlp_pack_weights": "pMpp",
    "cednerf_mlp_fwd": "ppMlppp",
    "cednerf_mlp_bwd": "ppppMlpippp",
    "cednerf_field_fwd": "ppppppppilppppFpppp",
    "cednerf_occ_update_level": "plpppiffpppFpppp",
    "cednerf_field_train_fwd": "ppppppilpppppFpppppppp",
    "cednerf_field_train_bwd": "ppppppilpppppFpppppppppppppipp",
    "cednerf_ray_offsets": "pllpp",
    "cednerf_composite_fwd": "pppppppillpppppppifp",
    "cednerf_composite_bwd": "pppppppillppppppppppfp",
    "cednerf_visibility_mask": "ppppllffppp",
    "cednerf_compact_samples": "pppppllpppp",
    "cednerf_accumulate_fwd": "ppipllpip",
    "cednerf_accumulate_bwd": "ppiplppppp",
    "cednerf_render_round_begin": "pliippp",
    "cednerf_march_round": "ipplppiipfffppppppppppppppipp",
    "cednerf_march_fill_runs_round": "lpppppiffppppppp",
    "cednerf_render_round_composite": "pppppppplifppppp",
    "cednerf_render_round_compact":"ppplppliippp",
    "cednerf_render_round": "Rlppp",
    "cednerf_generate_rays": "ppppiffffiilpppp",
    "cednerf_distortion_fwd": "pppplpppp",
    "cednerf_distortion_bwd": "pppplpppp",
    "cednerf_importance_keys": "ppplpp",
    "cednerf_topk_select": "pllpppp",
    "cednerf_importance_batch": "pliiippiffffipppppppp",
    "cednerf_nonfinite_check": "App",
    "cednerf_training_loss_fwd": "ppplppplpiffpppp",
    "cednerf_training_loss_bwd": "pppplpppliffpppppp",
    "cednerf_adam_step": "Apippfffip",
    "cednerf_peer_alloc": "lp",
    "cednerf_peer_free": "p",
    "cednerf_ipc_export": "pp",
    "cednerf_ipc_open": "pp",
    "cednerf_ipc_close": "p",
    "cednerf_dp_barrier": "Puip",
    "cednerf_dp_found_inf": "Pppp",
    "cednerf_dp_adam": "Dpppfffip",
    "cednerf_dp_adam_small": "Spppfffip",
    "cednerf_ms_ssim": "ppppllllpffppp",
}
_CT = {"p": ctypes.c_void_p, "i": ctypes.c_int, "l": ctypes.c_int64, "f": ctypes.c_float,
       "G": ctypes.POINTER(GridLevels), "M": ctypes.POINTER(MlpDesc), "F": ctypes.POINTER(FieldDesc),
       "A": ctypes.POINTER(AdamTensors), "P": ctypes.POINTER(DpPeers), "D": ctypes.POINTER(DpAdam), "S": ctypes.POINTER(DpSmall),
       "u": ctypes.c_uint32, "R": ctypes.POINTER(RenderRound)}

_lib = None


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `make -C cednerf_b200/csrc` (or `python -c 'import "
            "__graft_entry__ as g; g.build()'`).  cednerf_b200 has no CPU / PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.cednerf_last_error.restype = ctypes.c_char_p
    lib.cednerf_scan_workspace_bytes.restype = ctypes.c_int64
    lib.cednerf_launch_count.restype = ctypes.c_int64
    lib.cednerf_dp_ctrl_bytes.restype = ctypes.c_int64
    for name in ("cednerf_field_saved_bytes", "cednerf_field_bwd_workspace_bytes"):
        getattr(lib, name).restype = ctypes.c_int64
        getattr(lib, name).argtypes = [ctypes.POINTER(FieldDesc), ctypes.c_int64]
    lib.cednerf_scan_workspace_bytes.argtypes = [ctypes.c_int64]
    lib.cednerf_topk_workspace_bytes.restype = ctypes.c_int64
    lib.cednerf_topk_workspace_bytes.argtypes = [ctypes.c_int64]
    lib.cednerf_render_round_bytes.restype = ctypes.c_int64
    lib.cednerf_render_round_bytes.argtypes = []
    if lib.cednerf_render_round_bytes() != ctypes.sizeof(RenderRound):
        raise ImportError("cednerf_b200: CednerfRenderRound layout mismatch between the library and _lib.RenderRound")
    lib.cednerf_distortion_workspace_bytes.restype = ctypes.c_int64
    lib.cednerf_distortion_workspace_bytes.argtypes = []
    lib.cednerf_ms_ssim_workspace_bytes.restype = ctypes.c_int64
    lib.cednerf_ms_ssim_workspace_bytes.argtypes = [ctypes.c_int64] * 4
    for name, sig in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = ctypes.c_int
        fn.argtypes = [_CT[c] for c in sig]
    _lib = lib
    return lib


def exported_symbols():
    return sorted(list(_SIGNATURES) + ["cednerf_last_error", "cednerf_abi_version", "cednerf_check_device",
                                       "cednerf_scan_workspace_bytes", "cednerf_launch_count", "cednerf_field_saved_bytes",
                                       "cednerf_field_bwd_workspace_bytes", "cednerf_dp_ctrl_bytes", "cednerf_topk_workspace_bytes", "cednerf_distortion_workspace_bytes", "cednerf_render_round_bytes",
                                       "cednerf_ms_ssim_workspace_bytes"])


def ptr(t: Optional[torch.Tensor]):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("cednerf_b200 ops need CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("cednerf_b200 ops need contiguous tensors")
    return t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


_timers = None  # bench.py's per-entry-point CUDA-event instrumentation (None = off)


def call(name: str, *args):
    lib = load()
    if _timers is not None:
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        rc = getattr(lib, name)(*args)
        end.record()
        _timers.append((name, start, end))
    else:
        rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {lib.cednerf_last_error().decode()}")


_device_checked = False


def launch_count() -> int:
    return int(load().cednerf_launch_count())


def check_device():
    global _device_checked
    if not _device_checked:
        lib = load()
        if not torch.cuda.is_available():
            raise RuntimeError("cednerf_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        rc = lib.cednerf_check_device()
        if rc != 0:
            raise RuntimeError(f"cednerf_check_device failed ({rc}): {lib.cednerf_last_error().decode()}")
        _device_checked = True
