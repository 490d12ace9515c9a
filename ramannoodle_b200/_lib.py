"""ctypes binding of ``libramannoodle_b200.so`` (the C-ABI in ``include/ramannoodle_b200.h``).

There is NO fallback: if the shared library is missing, cannot be loaded, or no sm_100
device is present, the product path raises ``NativeLibraryError`` loudly.
"""
from __future__ import annotations

import ctypes
import os

from .exceptions import NativeLibraryError

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libramannoodle_b200.so")

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int32_p = ctypes.POINTER(ctypes.c_int32)
c_int64_p = ctypes.POINTER(ctypes.c_int64)

RN_MODEL_DEFAULT = 0
RN_MODEL_FORCE_DENSE = 1

# name -> (restype, argtypes); must list every symbol include/ramannoodle_b200.h declares
PROTOTYPES = {
    "rn_last_error": (ctypes.c_char_p, []),
    "rn_device_info": (ctypes.c_int, [ctypes.c_int] + [ctypes.POINTER(ctypes.c_int)] * 4),
    "rn_model_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "rn_model_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "rn_model_info": (ctypes.c_int, [ctypes.c_void_p, c_int64_p]),
    "rn_calc_polarizabilities": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                                ctypes.c_void_p, ctypes.c_void_p]),
    "rn_get_polarizability": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                             ctypes.c_void_p, ctypes.c_void_p]),
    "rn_calc_polarizabilities_host": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]),
    "rn_calc_polarizabilities_multi": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                                      ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]),
    "rn_calc_polarizabilities_host_multi": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                                           ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                           ctypes.c_void_p]),
    "rn_calc_polarizabilities_routed": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                                       ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                       ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p]),
    "rn_routed_phases_supported": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,
                                                  ctypes.c_int64]),
    "rn_calc_polarizabilities_routed_phase": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                                             ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                                             ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                                                             ctypes.c_int64, ctypes.c_int, ctypes.c_void_p]),
    "rn_calc_polarizabilities_host_routed": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                                            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                                            ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                                                            ctypes.c_int64, ctypes.c_void_p]),
    "rn_apply_pbc": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    "rn_spectrum_plan_create": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "rn_spectrum_plan_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "rn_spectrum_num_points": (ctypes.c_int64, [ctypes.c_int64]),
    "rn_md_spectrum": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double, ctypes.c_int,
                                      ctypes.c_double, ctypes.c_int, ctypes.c_double, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_void_p]),
    "rn_spectrum_plan_create_batched": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, ctypes.c_int,
                                                       ctypes.POINTER(ctypes.c_void_p)]),
    "rn_md_spectrum_windows": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,
                                              ctypes.c_double, ctypes.c_int, ctypes.c_double, ctypes.c_int,
                                              ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "rn_md_cross_spectra": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_double,
                                           ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_double,
                                           ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "rn_vdos": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                               ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_double, ctypes.c_void_p,
                               ctypes.c_void_p, ctypes.c_void_p]),
    "rn_spectrum_plan_create_dist": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                    ctypes.POINTER(ctypes.c_void_p)]),
    "rn_spectrum_plan_info": (ctypes.c_int, [ctypes.c_void_p, c_int64_p]),
    "rn_spectrum_dist_sizes": (ctypes.c_int, [ctypes.c_void_p, c_int64_p, c_int64_p, c_int64_p]),
    "rn_spectrum_dist_route": (ctypes.c_int, [ctypes.c_void_p, c_int64_p, c_int64_p]),
    "rn_spectrum_dist_stripe": (ctypes.c_int, [ctypes.c_void_p, c_int64_p]),
    "rn_spectrum_dist_pack": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                             ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "rn_spectrum_dist_transform": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                                  ctypes.c_void_p]),
    "rn_spectrum_dist_final": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                              ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_double,
                                              ctypes.c_int, ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p]),
    "rn_spectrum_dist_finish": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double, ctypes.c_void_p,
                                               ctypes.c_void_p, ctypes.c_void_p]),
    "rn_signal_spectrum": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double, ctypes.c_void_p,
                                          ctypes.c_void_p, ctypes.c_void_p]),
    "rn_convolve_workspace_size": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int64]),
    "rn_convolve_spectrum": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                            ctypes.c_double, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                                            ctypes.c_void_p, ctypes.c_void_p]),
    "rn_convolve_spectra_workspace_size": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int64, ctypes.c_int64]),
    "rn_convolve_spectra": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,
                                           ctypes.c_int, ctypes.c_double, ctypes.c_void_p, ctypes.c_int64,
                                           ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "rn_calc_polarizabilities_sweep":(ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int64,
                                                      ctypes.c_void_p, ctypes.c_void_p]),
    "rn_calc_polarizabilities_host_sweep": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                                           ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64]),
    "rn_calc_polarizabilities_sweep_routed": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                                             ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                                             ctypes.c_int, ctypes.c_int64, ctypes.c_int64,
                                                             ctypes.c_int64, ctypes.c_void_p]),
    "rn_calc_polarizabilities_host_sweep_routed": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                                                  ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                                                  ctypes.c_int, ctypes.c_int64, ctypes.c_int64,
                                                                  ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p]),
    "rn_xdatcar_scan": (ctypes.c_int, [ctypes.c_char_p, c_int64_p, c_int64_p, ctypes.c_void_p]),
    "rn_xdatcar_read": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,
                                       ctypes.c_int, ctypes.c_int]),
    "rn_outcar_scan": (ctypes.c_int, [ctypes.c_char_p, c_int64_p, c_int64_p, ctypes.c_void_p, ctypes.c_void_p]),
    "rn_outcar_read": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,
                                      ctypes.c_void_p, ctypes.c_int, ctypes.c_int]),
    "rn_vasprun_scan": (ctypes.c_int, [ctypes.c_char_p, c_int64_p, c_int64_p, c_double_p]),
    "rn_vasprun_read": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,
                                       ctypes.c_int, ctypes.c_int]),
    "rn_host_apply_pbc": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int]),
    "rn_host_register": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_size_t]),
    "rn_host_unregister": (ctypes.c_int, [ctypes.c_void_p]),
    "rn_bspline_to_pp": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "rn_launch_count": (ctypes.c_int64, []),
}

# test / tuning hooks: include/ramannoodle_b200_debug.h
DEBUG_PROTOTYPES = {
    "rn_debug_force_generic_affine": (None, [ctypes.c_int]),
    "rn_debug_set_affine_config": (None, [ctypes.c_int, ctypes.c_int]),
    "rn_debug_set_dense_config": (None, [ctypes.c_int, ctypes.c_int]),
    "rn_debug_phase_tiles": (ctypes.c_int64, [ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, c_int64_p,
                                              ctypes.c_int64]),
    "rn_debug_set_dense_split": (None, [ctypes.c_int]),
    "rn_debug_set_sweep_fused": (None, [ctypes.c_int]),
    "rn_debug_set_sweep_min_run": (None, [ctypes.c_int]),
    "rn_debug_fft_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "rn_debug_fft_convolve": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
}

_lib = None


def lib() -> ctypes.CDLL:
    """Load the shared library once; bind every prototype."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryError(
                f"{LIB_PATH} not found — build it with `python -m ramannoodle_b200._build` "
                "(there is no CPU fallback)")
        try:
            handle = ctypes.CDLL(LIB_PATH)
        except OSError as exc:
            raise NativeLibraryError(f"cannot load {LIB_PATH}: {exc}") from exc
        for name, (restype, argtypes) in PROTOTYPES.items():
            try:
                fn = getattr(handle, name)
            except AttributeError as exc:
                raise NativeLibraryError(f"{LIB_PATH} does not export {name}") from exc
            fn.restype = restype
            fn.argtypes = argtypes
        for name, (restype, argtypes) in DEBUG_PROTOTYPES.items():
            fn = getattr(handle, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


def last_error() -> str:
    return lib().rn_last_error().decode("utf-8", "replace")


def check(status: int, what: str) -> None:
    """Raise on a non-zero ``rn_status``."""
    if status == 0:
        return
    message = last_error()
    if status == -1:
        raise ValueError(f"{what}: {message}")
    if status == -4:
        raise MemoryError(f"{what}: {message}")
    raise NativeLibraryError(f"{what} failed ({status}): {message}")


def require_device(device: int = 0) -> dict:
    """Fail loudly unless ``device`` is an sm_100 GPU the library can drive."""
    rt = ctypes.c_int()
    count = ctypes.c_int()
    cc = ctypes.c_int()
    sms = ctypes.c_int()
    status = lib().rn_device_info(device, ctypes.byref(rt), ctypes.byref(count), ctypes.byref(cc), ctypes.byref(sms))
    if status != 0:
        raise NativeLibraryError(f"no usable CUDA device {device}: {last_error()} (there is no CPU fallback)")
    if cc.value // 10 != 10:
        raise NativeLibraryError(f"device {device} is sm_{cc.value}; ramannoodle_b200 is built for sm_100a only")
    return {"runtime": rt.value, "devices": count.value, "compute_capability": cc.value, "sm_count": sms.value}


def launch_count() -> int:
    return int(lib().rn_launch_count())


def is_torch_tensor(obj) -> bool:
    """Whether ``obj`` is a torch tensor (checked without importing torch)."""
    return type(obj).__module__.startswith("torch") and hasattr(obj, "data_ptr")


def current_stream(device: int) -> ctypes.c_void_p:
    """torch's current CUDA stream on ``device``, as the ``void* stream`` argument of the C-ABI."""
    import torch  # pylint: disable=import-outside-toplevel

    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
