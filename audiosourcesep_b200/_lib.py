"""ctypes binding of libasep.so (include/asep.h) with DLPack tensor exchange.

PyTorch is only the tensor container: tensors are handed to the library as the ``DLTensor``
inside the DLPack capsule produced by ``torch.utils.dlpack.to_dlpack``.  There is no CPU
fallback: if the shared library is missing the import fails loudly, and every compute call
fails with ``RuntimeError`` when no sm_100 device is present.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch
from torch.utils import dlpack as _torch_dlpack

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libasep.so")

PREC_FP32 = 0
PREC_BF16 = 1
PREC_FP16 = 3       # Glow: tcgen05 with fp16 hidden activations in the forward network (closer to fp32, ~8 % slower)
PREC_BF16X3 = 2     # score networks: split-bf16 operands, three tcgen05 products per convolution
PREC_BF16X2 = 4     # Glow: tcgen05 "exact" mode, hidden activations as (hi + lo) bf16 pairs (round trip <= 1e-4)
PREC_FP16X2 = 5     # Glow: as BF16X2 with fp16 pairs (22 bits; hidden activations must stay below 65504)
PREC_FP16X3 = 6     # Glow: weights as (hi + lo) pairs too, three products per GEMM: score-exact on tensor cores


class AsepError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libasep error {code}: {msg}")
        self.code = code


class DLDevice(ctypes.Structure):
    _fields_ = [("device_type", ctypes.c_int32), ("device_id", ctypes.c_int32)]


class DLDataType(ctypes.Structure):
    _fields_ = [("code", ctypes.c_uint8), ("bits", ctypes.c_uint8), ("lanes", ctypes.c_uint16)]


class DLTensor(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("device", DLDevice), ("ndim", ctypes.c_int32), ("dtype", DLDataType),
                ("shape", ctypes.POINTER(ctypes.c_int64)), ("strides", ctypes.POINTER(ctypes.c_int64)),
                ("byte_offset", ctypes.c_uint64)]


class NcsnCfg(ctypes.Structure):
    _fields_ = [("version", ctypes.c_int32), ("H", ctypes.c_int32), ("W", ctypes.c_int32), ("C", ctypes.c_int32),
                ("ngf", ctypes.c_int32), ("num_classes", ctypes.c_int32)]


class GlowCfg(ctypes.Structure):
    _fields_ = [("H", ctypes.c_int32), ("W", ctypes.c_int32), ("C", ctypes.c_int32), ("L", ctypes.c_int32),
                ("K", ctypes.c_int32), ("n_filters", ctypes.c_int32), ("learntop", ctypes.c_int32),
                ("minval", ctypes.c_float), ("maxval", ctypes.c_float)]


_P = ctypes.POINTER(DLTensor)
_V = ctypes.c_void_p
_I = ctypes.c_int
_F = ctypes.c_float
_U64 = ctypes.c_uint64

# name -> argtypes; every function returns int status unless listed in _RESTYPES
_SIGNATURES = {
    "asep_init": [_I],
    "asep_glow_create": [ctypes.POINTER(GlowCfg), ctypes.POINTER(_V)],
    "asep_glow_destroy": [_V],
    "asep_glow_set_param": [_V, ctypes.c_char_p, _P],
    "asep_glow_get_param": [_V, ctypes.c_char_p, _P],
    "asep_glow_prepare": [_V, _I],
    "asep_glow_init_actnorm": [_V, _P, _V],
    "asep_glow_forward": [_V, _P, _P, _P, _V],
    "asep_glow_inverse": [_V, _P, _P, _V],
    "asep_glow_log_prob": [_V, _P, _P, _V],
    "asep_glow_grad_log_prob": [_V, _P, _P, _P, _V],
    "asep_glow_sample": [_V, _P, _P, _V],
    "asep_glow_enable_training": [_V],
    "asep_glow_num_trainable": [_V, ctypes.POINTER(ctypes.c_int64)],
    "asep_glow_train_grads": [_V, _P, _P, _F, _I, _P, _P, _V],
    "asep_glow_adamax_step": [_V, _P, _F, _F, _F, _F, _V],
    "asep_glow_adam_step": [_V, _P, _F, _F, _F, _F, _V],
    "asep_glow_get_flat": [_V, _P, _V],
    "asep_glow_set_flat": [_V, _P, _V],
    "asep_glow_sync_host": [_V],
    "asep_actnorm": [_P, _P, _P, _P, _I, _V],
    "asep_inv1x1": [_P, _P, _P, _V],
    "asep_coupling": [_P, _P, _P, _P, _I, _V],
    "asep_squeeze": [_P, _P, _I, _V],
    "asep_glow_coupling_nn": [_V, _I, _I, _P, _P, _V],
    "asep_glow_coupling_nn_backward": [_V, _I, _I, _P, _P, _P, _V],
    "asep_glow_coupling_tc": [_V, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _V],
    "asep_glow_wgrad_tc": [_P, _P, _I, _P, _V],
    "asep_philox_normal": [_P, _U64, _U64, _U64, _U64, _V],
    "asep_ncsn_create": [ctypes.POINTER(NcsnCfg), ctypes.POINTER(_V)],
    "asep_ncsn_destroy": [_V],
    "asep_ncsn_set_param": [_V, ctypes.c_char_p, _P],
    "asep_ncsn_set_sigmas": [_V, _P],
    "asep_ncsn_set_precision": [_V, _I],
    "asep_ncsn_prepare": [_V],
    "asep_ncsn_forward": [_V, _P, _P, _P, _V],
    "asep_ncsn_enable_training": [_V],
    "asep_ncsn_num_trainable": [_V, ctypes.POINTER(ctypes.c_int64)],
    "asep_ncsn_param_span": [_V, ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)],
    "asep_ncsn_train_grads": [_V, _P, _P, _P, _I, _P, _P, _V],
    "asep_ncsn_adam_step": [_V, _P, _F, _F, _F, _F, _V],
    "asep_ncsn_get_flat": [_V, _P, _V],
    "asep_ncsn_set_flat": [_V, _P, _V],
    "asep_mixing_db_k": [_I, _P, _P, _P, _V],
    "asep_langevin_step_k": [_I, _P, _P, _P, _P, _F, _F, _F, _U64, _U64, _U64, _P, _V],
    "asep_basis_glow_inner_k": [_I, ctypes.POINTER(_V), _P, _P, _I, _F, _F, _F, _P, _U64, _U64, _U64, _P, _P, _V],
    "asep_basis_ncsn_inner_k": [_I, ctypes.POINTER(_V), _P, _P, _I, _I, _F, _F, _F, _P, _U64, _U64, _U64, _P, _P, _V],
    "asep_basis_glow_run_k": [_I, ctypes.POINTER(_V), _I, _P, _P, _I, _I, ctypes.POINTER(ctypes.c_float),
                              ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float), _U64, _U64, _P, _P, _V],
    "asep_basis_ncsn_run_k": [_I, ctypes.POINTER(_V), _P, _P, _I, _I, ctypes.POINTER(ctypes.c_float),
                              ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float), _U64, _U64, _P, _P, _V],
    "asep_conv_profile": [_I],
    "asep_conv_profile_read": [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64),
                               ctypes.POINTER(ctypes.c_double)],
    "asep_conv_tc_image": [_P, _I, _I, _I, _P, _V],
    "asep_conv_tc_forward": [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _V],
    "asep_conv_wgrad_tc": [_P, _P, _P, _I, _I, _V],
    "asep_crc32c": [ctypes.c_char_p, ctypes.c_uint64, ctypes.c_uint32],
    "asep_bss_eval": [_P, _P, _I, ctypes.c_int64, ctypes.c_int64, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64),
                      _I, _I, _P, _V],
    "asep_ideal_mask": [_P, _P, _P, _I, _F, _V],
    "asep_stft": [_P, _I, _I, _P, _V],
    "asep_mel_db": [_P, _P, _P, _P, _P, _F, _F, _F, _F, _V],
    "asep_mel_to_stft": [_P, _P, _P, _P, _P, _P, _F, _I, _V],
    "asep_stft_filter": [_P, _P, _P, _I, _V],
    "asep_istft": [_P, _I, _P, _V],
    "asep_istft_track": [_P, _I, _I, _P, _V],
    "asep_griffinlim_update": [_P, _P, _P, _P, _F, _V],
    "asep_track_psd": [_P, _I, _I, _I, _I, _I, _I, _I, _P, _V],
    "asep_mwf": [_P, _P, _I, _P, _V],
    "asep_resample": [_P, _P, _P, _P, ctypes.c_double, _I, _P, _V],
    "asep_basis_graphs": [_I],
    "asep_hbm_profile": [_I],
    "asep_hbm_profile_read": [_I, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64),
                              ctypes.POINTER(ctypes.c_double)],
    "asep_tc_profile": [_I],
    "asep_tc_profile_read": [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64),
                             ctypes.POINTER(ctypes.c_double)],
}
_RESTYPES = {"asep_last_error": ctypes.c_char_p, "asep_abi_version": ctypes.c_int, "asep_launch_count": ctypes.c_int64,
             "asep_crc32c": ctypes.c_uint32}
EXPORTED_SYMBOLS = sorted(set(_SIGNATURES) | set(_RESTYPES))

_lib = None
_initialised_device: Optional[int] = None


def load() -> ctypes.CDLL:
    """dlopen libasep.so and declare the prototypes (no CUDA call is made here)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `make` (or __graft_entry__.build()). "
            "audiosourcesep_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, args in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = ctypes.c_int
    for name, res in _RESTYPES.items():
        fn = getattr(lib, name)
        if name not in _SIGNATURES:
            fn.argtypes = []
        fn.restype = res
    _lib = lib
    return lib


def check(status: int):
    if status != 0:
        raise AsepError(status, load().asep_last_error().decode("utf-8", "replace"))


def init(device: Optional[int] = None) -> int:
    """asep_init on ``device`` (default: torch's current CUDA device)."""
    global _initialised_device
    if not torch.cuda.is_available():
        raise RuntimeError("audiosourcesep_b200 needs a CUDA (sm_100a) device; there is no CPU fallback")
    if device is None:
        device = torch.cuda.current_device()
    if _initialised_device != device:
        check(load().asep_init(int(device)))
        _initialised_device = device
    return device


def launch_count() -> int:
    return int(load().asep_launch_count())


def conv_profile(on: bool) -> None:
    check(load().asep_conv_profile(int(on)))


def conv_profile_read():
    ms, n, fl = ctypes.c_double(), ctypes.c_int64(), ctypes.c_double()
    check(load().asep_conv_profile_read(ctypes.byref(ms), ctypes.byref(n), ctypes.byref(fl)))
    return ms.value, n.value, fl.value


HBM_CATEGORIES = {"flow_step": 0, "langevin": 1, "ncsn_prep": 2, "ncsn_pool_resize": 3, "gather": 4}


def hbm_profile(on: bool) -> None:
    check(load().asep_hbm_profile(int(on)))


def basis_graphs(on: bool) -> None:
    """CUDA-graph replay of the Langevin steps inside basis_*_inner (default on); off = eager launches."""
    check(load().asep_basis_graphs(int(on)))


def hbm_profile_read(category: int):
    """(summed kernel ms, launches, algorithmic bytes) of one HBM-bound kernel category since hbm_profile(True)."""
    ms, n, by = ctypes.c_double(), ctypes.c_int64(), ctypes.c_double()
    check(load().asep_hbm_profile_read(int(category), ctypes.byref(ms), ctypes.byref(n), ctypes.byref(by)))
    return ms.value, n.value, by.value


def tc_profile(on: bool) -> None:
    check(load().asep_tc_profile(int(on)))


def tc_profile_read():
    """(summed kernel ms, launches, algorithmic FLOPs) of the tcgen05 launches recorded since tc_profile(True)."""
    ms, n, fl = ctypes.c_double(), ctypes.c_int64(), ctypes.c_double()
    check(load().asep_tc_profile_read(ctypes.byref(ms), ctypes.byref(n), ctypes.byref(fl)))
    return ms.value, n.value, fl.value


# ------------------------------------------------------------------ DLPack plumbing
_PyCapsule_GetPointer = ctypes.pythonapi.PyCapsule_GetPointer
_PyCapsule_GetPointer.restype = ctypes.c_void_p
_PyCapsule_GetPointer.argtypes = [ctypes.py_object, ctypes.c_char_p]
_PyCapsule_GetName = ctypes.pythonapi.PyCapsule_GetName
_PyCapsule_GetName.restype = ctypes.c_char_p
_PyCapsule_GetName.argtypes = [ctypes.py_object]


class DL:
    """Keeps a DLPack capsule alive and exposes the ``DLTensor*`` inside it."""

    __slots__ = ("capsule", "ptr", "tensor")

    def __init__(self, t: Optional[torch.Tensor]):
        self.tensor = t
        if t is None:
            self.capsule = None
            self.ptr = ctypes.cast(None, _P)
            return
        self.capsule = _torch_dlpack.to_dlpack(t)
        name = _PyCapsule_GetName(self.capsule)
        addr = _PyCapsule_GetPointer(self.capsule, name)
        if name == b"dltensor":
            off = 0                       # DLManagedTensor starts with its DLTensor
        elif name == b"dltensor_versioned":
            off = 8 + 8 + 8 + 8           # DLPackVersion(2xu32) + manager_ctx + deleter + flags(u64)
        else:
            raise RuntimeError(f"unexpected DLPack capsule {name!r}")
        self.ptr = ctypes.cast(addr + off, _P)


def dl(t: Optional[torch.Tensor]) -> DL:
    return DL(t)


def stream_ptr(stream: Optional[torch.cuda.Stream] = None) -> ctypes.c_void_p:
    s = torch.cuda.current_stream() if stream is None else stream
    return ctypes.c_void_p(s.cuda_stream)
