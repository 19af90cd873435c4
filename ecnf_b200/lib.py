"""ctypes binding of libecnf_b200.so (the C-ABI declared in include/ecnf_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, an exception is raised.
torch is used only as the provider of device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional

PKG = Path(__file__).resolve().parent
# ECNF_B200_LIB: load another build of the same library (the cycle-counter build of tools/tc_profile.py)
LIB_PATH = Path(os.environ["ECNF_B200_LIB"]) if os.environ.get("ECNF_B200_LIB") else PKG / "libecnf_b200.so"

MODE_VF, MODE_VF_DIV, MODE_SAMPLE, MODE_SAMPLE_LOGQ, MODE_LOGPROB = range(5)
MAX_SAVE_TIMES = 1024   # ECNF_MAX_SAVE_TIMES
TARGET_LJ, TARGET_DW = 0, 1


class EcnfError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [
        ("n_frames", C.c_int32), ("dim", C.c_int32), ("n_blocks", C.c_int32), ("n_layers", C.c_int32),
        ("mlp_units", C.c_int32), ("n_hidden", C.c_int32), ("time_dim", C.c_int32), ("n_features", C.c_int32),
        ("sigma_min", C.c_float), ("base_scale", C.c_float), ("normalization_constant", C.c_float),
        ("freqs", C.c_float * 8),
    ]


class SolveCtrl(C.Structure):
    _fields_ = [
        ("fixed", C.c_int32), ("step_size", C.c_float), ("rtol", C.c_float), ("atol", C.c_float),
        ("dtmin", C.c_float), ("max_steps", C.c_int32), ("safety", C.c_float), ("factormin", C.c_float),
        ("factormax", C.c_float), ("error_order", C.c_float), ("err_scale", C.c_float),
    ]


def make_ctrl(use_fixed_step_size=False, rtol=1e-5, atol=1e-5, step_size=0.05, dtmin=1e-5, max_steps=4096,
              safety=0.9, factormin=0.2, factormax=10.0, error_order=5.0, err_scale=1.0) -> SolveCtrl:
    """err_scale multiplies the embedded Dopri5 error estimate (1 = diffrax's b_hat weights, 1.5 = the classic
    Hairer-Wanner ones; SURVEY Appendix B) -- the same knob as oracle.SolveControl.err_scale."""
    return SolveCtrl(int(bool(use_fixed_step_size)), step_size, rtol, atol, dtmin, max_steps, safety, factormin,
                     factormax, error_order, err_scale)


# every exported symbol of include/ecnf_b200.h with (restype, argtypes)
_P, _I64, _I32, _F, _U64 = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_uint64
SIGNATURES = {
    "ecnf_last_error": (C.c_char_p, []),
    "ecnf_version": (C.c_int, []),
    "ecnf_model_create": (C.c_int, [C.POINTER(Config), _P, C.POINTER(_P)]),
    "ecnf_model_destroy": (None, [_P]),
    "ecnf_model_set_params": (C.c_int, [_P, _P]),
    "ecnf_model_clone": (C.c_int, [_P, _P, C.POINTER(_P)]),
    "ecnf_model_param_count": (_I64, [_P]),
    "ecnf_model_num_tensors": (C.c_int, [_P]),
    "ecnf_model_param_layout": (C.c_int, [_P, C.c_int, C.c_char_p, C.c_int, C.POINTER(_I64), C.POINTER(_I64),
                                          C.POINTER(_I64)]),
    "ecnf_solve_workspace_bytes": (_I64, [_P, C.c_int, _I64]),
    "ecnf_model_set_engine": (C.c_int, [_P, C.c_int]),
    "ecnf_model_set_fm_chunk": (C.c_int, [_P, C.c_int64]),
    "ecnf_solve_tensor_flops_per_eval": (C.c_int64, [C.c_void_p]),
    "ecnf_solve_engine_for": (C.c_int, [_P, C.c_int]),
    "ecnf_solve_tc_tile_table": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_uint32), C.c_int64]),
    "ecnf_vf_forward": (C.c_int, [_P, _P, _P, _P, _I64, _P, _P, _I64, _P]),
    "ecnf_vf_forward_div": (C.c_int, [_P, _P, _P, _P, _I64, _P, _P, _P, _I64, _P]),
    "ecnf_solve": (C.c_int, [_P, C.c_int, _P, _P, _I64, C.POINTER(SolveCtrl), _P, _P, _P, _P, _I64, _P]),
    "ecnf_solve_hutchinson": (C.c_int, [_P, C.c_int, _P, _P, _P, _I64, C.POINTER(SolveCtrl), _P, _P, _P, _P, _I64, _P]),
    "ecnf_solve_saveat_workspace_bytes": (_I64, [_P, C.c_int, _I64, C.c_int]),
    "ecnf_solve_saveat": (C.c_int, [_P, C.c_int, _P, _P, _P, _I64, C.POINTER(SolveCtrl), C.c_int, C.POINTER(_F), _P, _P, _P,
                                    _P, _P, _P, _I64, _P]),
    "ecnf_vf_forward_hutchinson": (C.c_int, [_P, _P, _P, _P, _P, _I64, _P, _P, _P, _I64, _P]),
    "ecnf_normal_noise": (C.c_int, [_P, _U64, _I64, _I64, C.c_uint32, _P, _P]),
    "ecnf_base_sample": (C.c_int, [_P, _U64, _I64, _I64, _P, _P]),
    "ecnf_base_sample_from_noise": (C.c_int, [_P, _P, _I64, _P, _P]),
    "ecnf_base_log_prob": (C.c_int, [_P, _P, _I64, _P, _P]),
    "ecnf_fm_workspace_bytes": (_I64, [_P, _I64]),
    "ecnf_fm_loss_grad": (C.c_int, [_P, _P, _P, _P, _P, _I64, _F, _P, _P, _P, _I64, _P]),
    "ecnf_fm_draw_noise": (C.c_int, [_P, _U64, _I64, _I64, _P, _P, _P]),
    "ecnf_adam_step": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I64, _F, _F, _F, _F, _F, _P, _P]),
    "ecnf_warmup_cosine_lr": (_F, [_I64, _F, _F, _I64, _I64, _F]),
    "ecnf_ess_stats": (C.c_int, [_P, _I64, _P, _P]),
    "ecnf_target_log_prob": (C.c_int, [C.c_int, _P, _I64, C.c_int, C.c_int, _P, _P]),
}

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load the CUDA library; raise loudly if it is not built (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise EcnfError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(or `python ecnf_b200/build.py`). ecnf_b200 has no CPU fallback.")
    lib = C.CDLL(os.fspath(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().ecnf_last_error().decode(errors="replace")
        raise EcnfError(f"{what} failed (code {rc}): {msg}")
