"""ctypes binding of libiefvad.so (C ABI in include/iefvad.h).

There is no fallback: if the CUDA library has not been built, importing this module raises with the build
command; if no sm_100a device is present, the first compute call raises with the CUDA error text."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libiefvad.so")

ABI_VERSION = 1
F32, F16, BF16 = 0, 1, 2
NOISE = {"Gaussian": 0, "StudentT": 1}
PLANS = {"fp32": -1, "B": 6, "HH": 56}

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing - the IEF-VAD B200 path has no CPU or PyTorch fallback. Build it with "
        f"`python -c 'import __graft_entry__ as g; g.build()'` (or `python ief-vad_b200/build.py`) from the repo root.")

lib = C.CDLL(LIB_PATH)

_vp, _i, _i64, _f, _d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double

_SIGS = {
    "iefvad_abi_version": (_i, []),
    "iefvad_last_error": (C.c_char_p, []),
    "iefvad_model_create": (_i, [C.POINTER(_vp), _i, _i, _i, _i, _f, _i, _f, _f]),
    "iefvad_model_destroy": (None, [_vp]),
    "iefvad_model_set_param": (_i, [_vp, C.c_char_p, _vp, _i64, _vp]),
    "iefvad_model_set_plan": (_i, [_vp, _i]),
    "iefvad_model_get_plan": (_i, [_vp]),
    "iefvad_model_set_option": (_i, [_vp, C.c_char_p, _i64]),
    "iefvad_model_check_finite": (_i, [_vp, C.POINTER(C.c_int), _vp]),
    "iefvad_model_set_max_rows": (_i, [_vp, _i64]),
    "iefvad_model_forward": (_i, [_vp, _vp, _vp, _i, _i64, _i64] + [_vp] * 9 + [_vp]),
    "iefvad_model_forward_host": (_i, [_vp, _vp, _vp, _i, _i64, _i64, _vp, _vp, _vp]),
    "iefvad_model_forward_host_to_device": (_i, [_vp, _vp, _vp, _i, _i64, _i64, _vp, _vp, _vp]),
    "iefvad_model_set_host_part_rows": (_i, [_vp, _i64]),
    "iefvad_model_set_pad_dedup": (_i, [_vp, _i]),
    "iefvad_model_set_eval_outputs": (_i, [_vp] * 6),
    "iefvad_event_image": (_i, [_vp, _i64, _i, _i, _i, _f, _f, _vp, _vp, _vp]),
    "iefvad_model_forward_scores_ragged": (_i, [_vp, _vp, _vp, _i, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "iefvad_model_forward_scores": (_i, [_vp, _vp, _vp, _i, _i, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "iefvad_fuse": (_i, [_vp] * 4 + [_i64, _f, _f] + [_vp] * 3 + [_vp]),
    "iefvad_layernorm": (_i, [_vp, _i64, _i] + [_vp] * 4 + [_f, _vp, _vp]),
    "iefvad_linear": (_i, [_vp] * 4 + [_f, _i, _i64, _i, _i, _i, _i, _vp, _vp]),
    "iefvad_outproj_ln": (_i, [_vp] * 8 + [_f, _i64, _vp, _vp, _vp, _vp]),
    "iefvad_mha": (_i, [_vp] * 5 + [_i64, _i64, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "iefvad_classifier": (_i, [_vp, _i64, _i, _vp, _vp, _vp, _vp, _vp]),
    "iefvad_mil_topk_mean": (_i, [_vp, _vp, _i64, _i64, _i, _vp, _vp, _i, _vp]),
    "iefvad_clas2": (_i, [_vp, _vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp]),
    "iefvad_sort_scores": (_i, [_vp, _i64, _vp, _vp]),
    "iefvad_auc_ap": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp]),
    "iefvad_auc_ap_multi": (_i, [_vp, _vp, _vp, _i64, _i, _i, _vp, _vp, _vp]),
    "iefvad_segment_copy": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "iefvad_distance_adj": (_i, [_i64, _i, _vp, _vp]),
    "iefvad_similarity_adj": (_i, [_vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp]),
    "iefvad_graph_convolution": (_i, [_vp] * 4 + [_i, _vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp]),
    "iefvad_distance_scan": (_i, [_vp, _i64, _i, _i, _vp, _vp]),
    "iefvad_transformer": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "iefvad_clip_visual": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp]),
    "iefvad_process_split": (_i, [_vp, _i, _vp, _i64, _i, _i, _vp, _i64, _vp, _i, _vp]),
    "iefvad_process_feat": (_i, [_vp, _i, _vp, _i64, _i, _i, _vp, _vp, _i, _vp]),
    "iefvad_attention_train_fwd": (_i, [_vp, _i64, _i64, _i, _i, _f, C.c_uint64, _vp, _vp, _vp]),
    "iefvad_attention_train_bwd": (_i, [_vp, _vp, _vp, _vp, _i64, _i64, _i, _i, _f, C.c_uint64, _vp, _vp]),
    "iefvad_layernorm_bwd": (_i, [_vp, _vp, _vp, _i64, _i, _f, _vp, _vp, _vp, _vp]),
    "iefvad_colsum": (_i, [_vp, _vp, _i64, _i, _vp, _vp]),
    "iefvad_fuse_bwd": (_i, [_vp] * 11 + [_i64, _f, _f] + [_vp] * 5),
    "iefvad_relu_bwd": (_i, [_vp, _vp, _i64, _vp, _vp]),
    "iefvad_quickgelu": (_i, [_vp, _i64, _vp, _vp]),
    "iefvad_axpy": (_i, [_vp, _vp, _f, _i64, _vp]),
    "iefvad_outer": (_i, [_vp, _vp, _i64, _i, _vp, _vp]),
    "iefvad_wgrad": (_i, [_vp, _vp, _i64, _i, _i, _f, _vp, _vp]),
    "iefvad_transpose": (_i, [_vp, _i64, _i, _vp, _i64, _vp]),
    "iefvad_clas2_bwd": (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _i64, _i, _vp, _vp, _vp]),
    "iefvad_train_loss_fwd": (_i, [_vp, _vp, _i64, _vp, _i64, _i64] + [_vp] * 4 + [_i, _d, _d, _d, _vp, _vp, _i]
                              + [_vp] * 6),
    "iefvad_train_loss_bwd": (_i, [_vp, _vp, _vp, _i64, _vp, _i64, _i64, _i] + [_vp] * 4 + [_i, _vp, _d, _d, _d]
                              + [_vp] * 10),
    "iefvad_locmap_proposals": (_i, [_vp, _vp, _vp, _i64, _i, _i] + [_vp] * 5),
    "iefvad_locmap_match": (_i, [_vp, _vp, _vp, _i64, _i, _vp, _vp, _i64, C.c_double, _vp, _vp, _vp]),
    "iefvad_bench_gemm": (_i, [_i64, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "iefvad_launch_count": (C.c_uint64, []),
    "iefvad_alloc_generation": (C.c_uint64, []),
    "iefvad_add_launches": (None, [C.c_uint64]),
    "iefvad_profile_enable": (_i, [_i]),
    "iefvad_profile_read": (_i, [_vp, _vp, _vp]),
}

EXPORTS = tuple(_SIGS)

for _name, (_res, _args) in _SIGS.items():
    try:
        _fn = getattr(lib, _name)
    except AttributeError:
        continue  # reported by tests/test_abi.py, which checks every symbol of include/iefvad.h
    _fn.restype = _res
    _fn.argtypes = _args

if lib.iefvad_abi_version() != ABI_VERSION:
    raise ImportError(f"libiefvad.so ABI {lib.iefvad_abi_version()} != expected {ABI_VERSION}; rebuild it")


class IefvadError(RuntimeError):
    pass


def last_error() -> str:
    msg = lib.iefvad_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int) -> None:
    if rc != 0:
        msg = last_error()
        if msg.startswith("Unsupported noise_model"):
            raise ValueError(msg)      # same exception type and text as model/imf_vad.py:138
        raise IefvadError(f"libiefvad error {rc}: {msg}")


def ptr(t) -> int:
    """Device (or host) address of a torch tensor, 0 for None."""
    return 0 if t is None else t.data_ptr()


def stream_ptr(device=None) -> int:
    import torch
    return torch.cuda.current_stream(device).cuda_stream
