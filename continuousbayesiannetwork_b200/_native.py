"""ctypes binding of ``libcbn_b200.so`` (the C ABI declared in ``include/cbn_b200.h``).

There is no CPU fallback: importing this module without the built library, or
creating a context without a B200-class CUDA device, raises.  PyTorch is used by
the callers only to own device memory and streams; every argument crossing this
boundary is a raw pointer or a size.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Sequence

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libcbn_b200.so")

MAX_FAMILY_VARS = 12
MAX_CARD = 255
UNSEEN = 255
MAX_CONTRACT_DIMS = 24
MAX_CONTRACT_INPUTS = 16
MAX_GATHER_TABLES = 16
MAX_EVIDENCE_PTRS = 64
GATHER_MAX_CT = 8          # widest target the register-resident gather kernels (and the fused MAP epilogue) handle

OK, ERR_INVALID, ERR_CUDA, ERR_NOMEM, ERR_UNSUPPORTED = 0, -1, -2, -3, -4


class NativeLibraryMissing(ImportError):
    pass


class Family(C.Structure):
    _fields_ = [
        ("n_vars", C.c_int32),
        ("var", C.c_int32 * MAX_FAMILY_VARS),
        ("card", C.c_int32 * MAX_FAMILY_VARS),
        ("table_offset", C.c_int64),
    ]


class Contract(C.Structure):
    _fields_ = [
        ("n_out_dims", C.c_int32),
        ("out_card", C.c_int32 * MAX_CONTRACT_DIMS),
        ("sum_card", C.c_int32),
        ("n_in", C.c_int32),
        ("inp", C.c_void_p * MAX_CONTRACT_INPUTS),
        ("in_stride", (C.c_int32 * MAX_CONTRACT_DIMS) * MAX_CONTRACT_INPUTS),
        ("sum_stride", C.c_int32 * MAX_CONTRACT_INPUTS),
        ("out", C.c_void_p),
        ("normalize_last", C.c_int32),
        ("log_space", C.c_int32),
    ]


class GatherTable(C.Structure):
    _fields_ = [
        ("data", C.c_void_p),
        ("n_cells", C.c_int64),
        ("n_ev", C.c_int32),
        ("ev_slot", C.c_int32 * MAX_CONTRACT_DIMS),
        ("ev_stride", C.c_int32 * MAX_CONTRACT_DIMS),
        ("has_target", C.c_int32),
    ]


class RowInput(C.Structure):
    _fields_ = [
        ("data", C.c_void_p),
        ("n_cells", C.c_int64),
        ("n_ev", C.c_int32),
        ("ev_slot", C.c_int32 * MAX_CONTRACT_DIMS),
        ("ev_stride", C.c_int32 * MAX_CONTRACT_DIMS),
    ]


class RowStep(C.Structure):
    _fields_ = [
        ("out_size", C.c_int32),
        ("sum_card", C.c_int32),
        ("n_in", C.c_int32),
        ("in_id", C.c_int32 * MAX_CONTRACT_INPUTS),
        ("sum_stride", C.c_int32 * MAX_CONTRACT_INPUTS),
        ("offsets", C.c_void_p),
    ]


class MpeStep(C.Structure):
    _fields_ = [
        ("slot", C.c_int32),
        ("card", C.c_int32),
        ("argmax", C.c_void_p),
        ("n_cells", C.c_int64),
        ("n_ctx", C.c_int32),
        ("ctx_slot", C.c_int32 * MAX_CONTRACT_DIMS),
        ("ctx_stride", C.c_int32 * MAX_CONTRACT_DIMS),
    ]


class PsampleStep(C.Structure):
    _fields_ = [
        ("slot", C.c_int32),
        ("card", C.c_int32),
        ("cdf", C.c_void_p),
        ("n_cells", C.c_int64),
        ("n_ctx", C.c_int32),
        ("ctx_slot", C.c_int32 * MAX_CONTRACT_DIMS),
        ("ctx_stride", C.c_int32 * MAX_CONTRACT_DIMS),
        ("var", C.c_int32),
    ]


MPE_MAX_SLOTS = 512
ROWS_LOG_SPACE = 1
GATHER_NORMALIZE, GATHER_LOG_SPACE = 1, 2
HOST_OUT_DROP_LAST = 1
COMM_ID_BYTES = 128

# name -> (restype, argtypes); also the list the CPU test checks against the header
_P = C.c_void_p
SIGNATURES = {
    "cbn_abi_version": (C.c_int, []),
    "cbn_ctx_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "cbn_ctx_destroy": (None, [_P]),
    "cbn_last_error": (C.c_char_p, [_P]),
    "cbn_device_sm_count": (C.c_int, [_P]),
    "cbn_domain_f32": (C.c_int, [_P, _P, C.c_int64, _P, _P, _P]),
    "cbn_encode_f32": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int32, _P, _P, _P]),
    "cbn_domain_f32_multi": (C.c_int, [_P, C.POINTER(_P), C.c_int32, C.c_int64, _P, _P, _P]),
    "cbn_encode_f32_multi": (C.c_int, [_P, C.POINTER(_P), C.c_int32, C.c_int64, _P, _P, _P, C.c_int64, _P, _P]),
    "cbn_count_plan_create": (C.c_int, [_P, C.POINTER(Family), C.c_int32, C.c_int32, C.POINTER(_P)]),
    "cbn_count_plan_destroy": (None, [_P]),
    "cbn_count_run": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, _P]),
    "cbn_count_run_host": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, _P]),
    "cbn_count_plan_groups": (C.c_int, [_P]),
    "cbn_count_plan_updates_per_sample": (C.c_int, [_P]),
    "cbn_comm_unique_id": (C.c_int, [_P]),
    "cbn_comm_create": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "cbn_comm_destroy": (None, [_P]),
    "cbn_comm_size": (C.c_int, [_P]),
    "cbn_counts_allreduce": (C.c_int, [_P, _P, _P, C.c_int64, _P]),
    "cbn_cpt_from_counts": (C.c_int, [_P, _P, C.POINTER(Family), C.c_int32, C.c_longlong, _P, _P, _P]),
    "cbn_cpt_from_plan": (C.c_int, [_P, _P, _P, C.c_longlong, _P, _P, _P]),
    "cbn_cpt_from_plan_dev": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "cbn_mle_from_counts": (C.c_int, [_P, _P, C.POINTER(Family), C.POINTER(_P), C.c_longlong, _P, _P, _P]),
    "cbn_get_prob_f32": (C.c_int, [_P, _P, C.POINTER(Family), C.POINTER(_P), _P, C.c_int64, C.c_int32, _P,
                                   C.c_int64, _P, _P]),
    "cbn_factor_contract": (C.c_int, [_P, C.POINTER(Contract), _P]),
    "cbn_factor_rescale": (C.c_int, [_P, _P, C.c_longlong, C.c_int32, C.c_int32, _P]),
    "cbn_ve_plan_create_gather": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(GatherTable),
                                            C.c_int32, C.c_int32, _P, C.POINTER(_P)]),
    "cbn_ve_plan_create_rows": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(RowInput), C.c_int32,
                                          C.POINTER(RowStep), C.c_int32, C.c_int32, _P, C.POINTER(_P)]),
    "cbn_ve_plan_destroy": (None, [_P]),
    "cbn_ve_plan_fuse": (C.c_int, [_P, C.POINTER(_P), C.c_int32, _P, C.POINTER(_P)]),
    "cbn_ve_plan_set_static_evidence": (C.c_int, [_P, C.c_int32]),
    "cbn_ve_plan_outputs": (C.c_int, [_P]),
    "cbn_ve_run_codes_multi": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, C.POINTER(_P), _P]),
    "cbn_ve_run_codes": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, _P]),
    "cbn_ve_run_f32": (C.c_int, [_P, _P, C.POINTER(_P), C.POINTER(_P), C.c_int64, _P, _P]),
    "cbn_ve_run_codes_map": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, _P, _P]),
    "cbn_ve_run_f32_map": (C.c_int, [_P, _P, C.POINTER(_P), C.POINTER(_P), C.c_int64, _P, _P, _P]),
    "cbn_ve_run_codes_log_evidence": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, _P]),
    "cbn_loglik_plan_create": (C.c_int, [_P, C.POINTER(Family), C.c_int32, C.c_int32, _P, _P, C.POINTER(_P)]),
    "cbn_loglik_plan_destroy": (None, [_P]),
    "cbn_loglik_run": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, C.c_int32, _P]),
    "cbn_loglik_plan_tables": (C.c_int, [_P]),
    "cbn_factor_contract_max": (C.c_int, [_P, C.POINTER(Contract), _P, _P]),
    "cbn_mpe_plan_create": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(MpeStep), C.c_int32, _P,
                                      C.POINTER(_P)]),
    "cbn_mpe_plan_destroy": (None, [_P]),
    "cbn_mpe_run": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, _P, C.c_int64, _P]),
    "cbn_factor_contract_cdf": (C.c_int, [_P, C.POINTER(Contract), _P, _P]),
    "cbn_psample_plan_create": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(PsampleStep), C.c_int32,
                                          _P, C.POINTER(_P)]),
    "cbn_psample_plan_destroy": (None, [_P]),
    "cbn_psample_run": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P, C.c_uint64, C.c_int64, C.c_int32, _P, C.c_int64,
                                  _P]),
    "cbn_ve_run_codes_host": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P]),
    "cbn_ve_run_codes_host_multi": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, C.POINTER(_P)]),
    "cbn_ve_run_codes_host_multi_ex": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, C.POINTER(_P), C.c_int32]),
    "cbn_batch_max": (C.c_int, [_P, _P, C.c_int64, _P, _P]),
    "cbn_scale_by_inv": (C.c_int, [_P, _P, C.c_int64, _P, _P]),
    "cbn_sample_forward": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32), C.POINTER(Family), _P, C.c_uint64,
                                     C.c_int64, C.c_int64, _P, C.c_int64, _P]),
}

_lib = None


def lib() -> C.CDLL:
    """The loaded library.  Raises ``NativeLibraryMissing`` if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                f"{LIB_PATH} is missing: build it with `python -m continuousbayesiannetwork_b200.build` "
                "(nvcc, sm_100a).  There is no CPU fallback for this engine."
            )
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError here = header / library mismatch
            fn.restype = res
            fn.argtypes = args
        if handle.cbn_abi_version() != 2:
            raise NativeLibraryMissing("libcbn_b200.so has an unexpected ABI version; rebuild it")
        _lib = handle
    return _lib


class CbnError(RuntimeError):
    pass


def check(rc: int, ctx=None) -> None:
    """Map a status code to the exception class the reference would raise."""
    if rc == OK:
        return
    msg = lib().cbn_last_error(ctx)
    msg = msg.decode() if msg else f"cbn_b200 error {rc}"
    if rc == ERR_INVALID:
        raise ValueError(msg)
    if rc == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == ERR_NOMEM:
        raise MemoryError(msg)
    raise CbnError(msg)


class Context:
    """One ``cbn_ctx`` per CUDA device."""

    def __init__(self, device_index: int):
        self.device_index = int(device_index)
        h = _P()
        check(lib().cbn_ctx_create(self.device_index, C.byref(h)))
        self.handle = h
        self.sm_count = lib().cbn_device_sm_count(h)

    def __del__(self):
        try:
            if getattr(self, "handle", None) and _lib is not None:
                _lib.cbn_ctx_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


_contexts: Dict[int, Context] = {}


def context_for(device) -> Context:
    """Context of a torch device (``cuda`` / ``cuda:N``).  Anything but CUDA is an error."""
    import torch

    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(
            f"continuousbayesiannetwork_b200 runs on CUDA (sm_100a) only; got device '{device}'. "
            "There is no CPU path."
        )
    if not torch.cuda.is_available():
        raise RuntimeError("continuousbayesiannetwork_b200 needs a CUDA device (B200, sm_100a); none is visible.")
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if idx not in _contexts:
        _contexts[idx] = Context(idx)
    return _contexts[idx]


def make_family(vars_: Sequence[int], cards: Sequence[int], table_offset: int) -> Family:
    if not 1 <= len(vars_) <= MAX_FAMILY_VARS:
        raise ValueError(f"a family can have at most {MAX_FAMILY_VARS - 1} parents; got {len(vars_) - 1}")
    f = Family()
    f.n_vars = len(vars_)
    for j, (v, c) in enumerate(zip(vars_, cards)):
        f.var[j] = int(v)
        f.card[j] = int(c)
    f.table_offset = int(table_offset)
    return f


def ptr_array(ptrs: Sequence[int]):
    arr = (_P * max(len(ptrs), 1))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr


def stream_ptr(device=None) -> int:
    import torch

    return torch.cuda.current_stream(device).cuda_stream
