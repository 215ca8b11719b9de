"""ctypes binding of the C-ABI library (include/nerf_b200.h).

The library is built in-tree by ``nerficg_b200/csrc/build.py`` (``__graft_entry__.build()``).
There is NO fallback: a missing library or a non-sm_100 device raises.
"""
from __future__ import annotations

import ctypes
from ctypes import c_float, c_int, c_int64, c_size_t, c_void_p
from pathlib import Path

import torch

LIB_PATH = Path(__file__).resolve().parent / 'libnerf_b200.so'

_PROTOTYPES = {
    # name: (restype, argtypes)
    'nerf_abi_version': (c_int, []),
    'nerf_last_error': (ctypes.c_char_p, []),
    'nerf_device_check': (c_int, [c_int]),
    'nerf_param_layout': (c_int, [ctypes.POINTER(c_int64), ctypes.POINTER(c_int64), ctypes.POINTER(c_int64)]),
    'nerf_sample_stratified': (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_void_p]),
    'nerf_sample_importance': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    'nerf_composite_forward': (c_int, [c_void_p] * 8 + [c_int, c_int, c_void_p]),
    'nerf_composite_backward': (c_int, [c_void_p] * 8 + [c_int, c_int, c_int, c_float, c_void_p]),
    'nerf_mlp_packed_bytes': (c_size_t, []),
    'nerf_mlp_pack': (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    'nerf_mlp_stash_bytes': (c_size_t, [c_int64]),
    'nerf_mlp_forward': (c_int, [c_void_p] * 9 + [c_int, c_int, c_void_p]),
    'nerf_mlp_backward_workspace_bytes': (c_size_t, [c_int64]),
    'nerf_mlp_backward': (c_int, [c_void_p] * 7 + [c_int, c_int, c_float, c_void_p]),
    'nerf_mlp_backward_dgrad': (c_int, [c_void_p] * 6 + [c_int, c_int, c_void_p]),
    'nerf_mlp_backward_wgrad': (c_int, [c_void_p] * 3 + [c_int, c_int, c_float, c_void_p]),
    'nerf_mlp_backward_inputs': (c_int, [c_void_p] * 6 + [c_int64, c_float, c_void_p]),
    'nerf_mlp_backward_rays_scratch_bytes': (c_size_t, [c_int, c_int]),
    'nerf_mlp_backward_rays': (c_int, [c_void_p] * 12 + [c_int, c_int, c_float, c_void_p]),
    'nerf_adam_tick': (c_int, [c_void_p, c_float, c_float, c_void_p]),
    'nerf_adam_update': (c_int, [c_void_p] * 6 + [c_float, c_float, c_float, c_int64, c_void_p]),
    'nerf_adam_update_ex': (c_int, [c_void_p] * 6 + [c_float, c_float, c_float, c_float, c_int, c_int64, c_void_p]),
    'nerf_generate_rays': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, ctypes.POINTER(ctypes.c_double), c_int, c_int,
                                   ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, c_void_p]),
    'nerf_gather_rays': (c_int, [c_void_p] * 11 + [c_int64, c_void_p]),
    'nerf_loss_mse': (c_int, [c_void_p] * 12 + [c_int, c_float, c_float, c_void_p]),
    'nerf_debug_set_timing': (c_int, [c_void_p]),
    'nerf_selftest_umma': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    'nerf_selftest_umma2': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    'nerf_selftest_umma2_mn': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    'nerf_selftest_tmem_read': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p]),
    'nerf_selftest_umma2_rate': (c_int, [c_void_p, c_int, c_int, c_void_p]),
    'nerf_selftest_l2_stream': (c_int, [c_void_p, c_void_p, ctypes.c_uint32, c_int, c_int, c_int, c_void_p]),
    'nerf_selftest_l2_stream_lsu': (c_int, [c_void_p, c_void_p, ctypes.c_uint32, c_int, c_int, c_int, c_int, c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_PROTOTYPES)
_lib = None


class NativeLibraryError(RuntimeError):
    """The CUDA extension is missing, stale or running on an unsupported device."""


def load() -> ctypes.CDLL:
    """Loads libnerf_b200.so and declares every prototype.  Raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise NativeLibraryError(
            f'{LIB_PATH} not found: build it with `python nerficg_b200/csrc/build.py` '
            '(there is no CPU or PyTorch fallback for the NeRF hot path)')
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (res, args) in _PROTOTYPES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise NativeLibraryError(f'{LIB_PATH} does not export {name}; rebuild the extension') from e
        fn.restype = res
        fn.argtypes = args
    if lib.nerf_abi_version() != 1:
        raise NativeLibraryError('ABI version mismatch; rebuild the extension')
    _lib = lib
    return lib


def last_error() -> str:
    return load().nerf_last_error().decode()


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise NativeLibraryError(f'{what} failed ({rc}): {last_error()}')


_checked_devices: set[int] = set()


def require_device(t: torch.Tensor) -> None:
    """Fails loudly unless ``t`` lives on an sm_100 GPU."""
    if not t.is_cuda:
        raise NativeLibraryError('nerficg_b200 kernels need CUDA tensors on a B200 (sm_100); there is no CPU path')
    idx = t.device.index if t.device.index is not None else torch.cuda.current_device()
    if idx not in _checked_devices:
        check(load().nerf_device_check(idx), 'nerf_device_check')
        _checked_devices.add(idx)


def ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def param_layout() -> tuple[list[int], list[int], int]:
    off = (c_int64 * 24)()
    size = (c_int64 * 24)()
    total = c_int64()
    check(load().nerf_param_layout(off, size, ctypes.byref(total)), 'nerf_param_layout')
    return list(off), list(size), total.value
