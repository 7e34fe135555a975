"""Loader of the product C-ABI library (csrc/libspartacus_b200.so).

There is no CPU fallback: if the library is missing this raises, and every
solve entry point of the library itself returns SSB200_ERR_NOGPU when no CUDA
device is visible.
"""
import ctypes as C
import os

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
# SSB200_LIB: alternative build of the same library (kernel tuning experiments)
LIB_PATH = os.environ.get("SSB200_LIB") or os.path.join(_HERE, "csrc", "libspartacus_b200.so")

_lib = None


class LibraryMissing(RuntimeError):
    pass


def _declare(lib):
    P = C.POINTER
    lib.ssb200_version.restype = C.c_char_p
    lib.ssb200_last_error.restype = C.c_char_p
    lib.ssb200_abi_sizes.argtypes = [P(C.c_int64)]
    lib.ssb200_device_count.restype = C.c_int
    lib.ssb200_set_device.argtypes = [C.c_int]
    lib.ssb200_legendre_gauss_init.argtypes = [C.c_int32, P(_abi.LegendreGauss)]
    radsurf_args = [P(_abi.Config), P(_abi.CanopyProperties), P(_abi.SwSpectralProperties),
                    P(_abi.LwSpectralProperties), P(_abi.BoundaryCondsOut), C.c_int32, C.c_int32,
                    P(_abi.CanopyFlux), P(_abi.CanopyFlux), P(_abi.CanopyFlux), P(_abi.CanopyFlux)]
    lib.ssb200_radsurf.argtypes = radsurf_args
    lib.ssb200_radsurf.restype = C.c_int
    lib.ssb200_radsurf_sp.argtypes = radsurf_args  # (the _sp structs are layout-identical)
    lib.ssb200_radsurf_sp.restype = C.c_int
    lib.ssb200_radsurf_device.argtypes = radsurf_args + [C.c_void_p, P(C.c_int32)]
    lib.ssb200_radsurf_device.restype = C.c_int
    lib.ssb200_radsurf_fluxes.argtypes = (radsurf_args[:4] + [P(_abi.DriverInputs)] + radsurf_args[4:7]
                                          + [P(_abi.CanopyFlux), P(_abi.CanopyFlux)])
    lib.ssb200_radsurf_fluxes.restype = C.c_int
    # (the _sp structs, ssb200_driver_inputs_sp included, are layout-identical to the double ones)
    lib.ssb200_radsurf_fluxes_sp.argtypes = lib.ssb200_radsurf_fluxes.argtypes
    lib.ssb200_radsurf_fluxes_sp.restype = C.c_int
    lib.ssb200_radsurf_device_sp.argtypes = lib.ssb200_radsurf_device.argtypes
    lib.ssb200_radsurf_device_sp.restype = C.c_int
    lib.ssb200_radsurf_fluxes_device.argtypes = lib.ssb200_radsurf_fluxes.argtypes + [C.c_void_p, P(C.c_int32)]
    lib.ssb200_radsurf_fluxes_device.restype = C.c_int
    lib.ssb200_radsurf_fluxes_device_sp.argtypes = lib.ssb200_radsurf_fluxes_device.argtypes
    lib.ssb200_radsurf_fluxes_device_sp.restype = C.c_int
    lib.ssb200_kernel_launch_count.restype = C.c_int64
    lib.ssb200_set_profiling.argtypes = [C.c_int]
    lib.ssb200_last_kernel_times_ms.argtypes = [P(C.c_double)]
    lib.ssb200_last_kernel_counts.argtypes = [P(C.c_int64)]
    lib.ssb200_release.restype = C.c_int
    lib.ssb200_set_option.argtypes = [C.c_char_p, C.c_int64]
    lib.ssb200_canopy_flux_scale_device.argtypes = [P(_abi.CanopyFlux), P(C.c_int32), P(C.c_int32),
                                                    C.c_void_p, C.c_void_p]
    lib.ssb200_canopy_flux_sum_device.argtypes = [P(_abi.CanopyFlux), P(_abi.CanopyFlux),
                                                  P(_abi.CanopyFlux), C.c_void_p]
    lib.ssb200_canopy_flux_check_device.argtypes = [P(_abi.CanopyFlux), P(_abi.CanopyProperties),
                                                    C.c_void_p, C.c_void_p]
    lib.ssb200_calc_simple_spectrum_lw_device.argtypes = ([P(_abi.LwSpectralProperties)] + [C.c_int32] * 6
                                                          + [C.c_void_p] * 7)
    lib.ssb200_measure_fp64_peak_tflops.argtypes = [C.c_int]
    lib.ssb200_measure_fp64_peak_tflops.restype = C.c_double
    return lib


def load():
    """Return the ctypes handle of libspartacus_b200.so (built by __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LibraryMissing(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)")
        lib = _declare(C.CDLL(LIB_PATH))
        sizes = (C.c_int64 * 7)()
        lib.ssb200_abi_sizes(sizes)
        mirror = [C.sizeof(t) for t in (_abi.LegendreGauss, _abi.Config, _abi.CanopyProperties,
                                       _abi.SwSpectralProperties, _abi.LwSpectralProperties,
                                       _abi.CanopyFlux, _abi.BoundaryCondsOut)]
        if list(sizes) != mirror:
            raise RuntimeError(f"ctypes mirror out of date: library {list(sizes)} vs _abi.py {mirror}")
        _lib = lib
    return _lib


def last_error():
    return load().ssb200_last_error().decode()
