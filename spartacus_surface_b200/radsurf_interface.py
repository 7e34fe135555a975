"""radsurf: the public entry of the path (radsurf/radsurf_interface.F90:20-25).

Same argument list and meaning as the reference subroutine; the body is the
B200 library (ssb200_radsurf for host arrays, ssb200_radsurf_device when the
members are torch CUDA tensors; radsurf_fluxes likewise picks ssb200_radsurf_fluxes or
ssb200_radsurf_fluxes_device; the _sp wrappers below take float32 arrays and pick the host or device
single-precision entry the same way).  The reference aborts on error
(utilities/radiation_io.F90:46-54); here errors raise RadsurfError.
"""
import ctypes as C

from ._arrays import dptr, is_torch
from ._lib import load, last_error


class RadsurfError(RuntimeError):
    pass


def marshal(config, canopy_props, sw_spectral_props, lw_spectral_props, bc_out,
            sw_norm_dir=None, sw_norm_diff=None, lw_internal=None, lw_norm=None, ptr=dptr):
    """Build the C structs of include/spartacus_b200.h from the API objects.

    Returned objects own no array memory: the caller's arrays must outlive
    the call (same ownership rule as the Fortran allocatables).  `ptr` maps
    an array member to the address stored in its struct slot.
    """
    s = lambda o: o.as_struct(ptr) if o is not None else None
    structs = dict(
        config=config.as_struct(),
        canopy=canopy_props.as_struct(ptr),
        sw=s(sw_spectral_props),
        lw=s(lw_spectral_props),
        bc=bc_out.as_struct(ptr),
        sw_norm_dir=s(sw_norm_dir),
        sw_norm_diff=s(sw_norm_diff),
        lw_internal=s(lw_internal),
        lw_norm=s(lw_norm),
    )
    return structs


def _ref(s):
    return C.byref(s) if s is not None else None


def call_radsurf(fn, structs, istartcol, iendcol, extra=()):
    s = structs
    return fn(_ref(s["config"]), _ref(s["canopy"]), _ref(s["sw"]), _ref(s["lw"]), _ref(s["bc"]),
              int(istartcol or 0), int(iendcol or 0), _ref(s["sw_norm_dir"]), _ref(s["sw_norm_diff"]),
              _ref(s["lw_internal"]), _ref(s["lw_norm"]), *extra)


def radsurf(config, canopy_props, sw_spectral_props, lw_spectral_props, bc_out,
            istartcol=None, iendcol=None, sw_norm_dir=None, sw_norm_diff=None,
            lw_internal=None, lw_norm=None, stream=None):
    """Solve columns istartcol..iendcol (1-based inclusive, default all)."""
    lib = load()
    structs = marshal(config, canopy_props, sw_spectral_props, lw_spectral_props, bc_out,
                      sw_norm_dir, sw_norm_diff, lw_internal, lw_norm)
    device = is_torch(canopy_props.dz) if canopy_props.dz is not None else is_torch(bc_out.sw_albedo
                                                                                    if bc_out.sw_albedo is not None
                                                                                    else bc_out.lw_emissivity)
    if device:
        rc = call_radsurf(lib.ssb200_radsurf_device, structs, istartcol, iendcol,
                          extra=(C.c_void_p(stream or 0), None))
    else:
        rc = call_radsurf(lib.ssb200_radsurf, structs, istartcol, iendcol)
    if rc < 0:
        raise RadsurfError(f"ssb200_radsurf failed (rc={rc}): {last_error()}")
    return rc


def radsurf_fluxes(config, canopy_props, sw_spectral_props, lw_spectral_props, bc_out, istartcol=None, iendcol=None,
                   sw_flux=None, lw_flux=None, top_flux_dn_sw=None, top_flux_dn_direct_sw=None, top_flux_dn_lw=None,
                   ground_temperature=None, roof_temperature=None, wall_temperature=None,
                   clear_air_temperature=None, veg_temperature=None, veg_air_temperature=None, stream=None):
    """The reference driver's sequence for a block of columns in one call
    (driver/spartacus_surface_driver.F90:206-261): calc_simple_spectrum_lw, radsurf,
    scale of the normalised fluxes by the top-of-canopy fluxes and sum into `sw_flux` / `lw_flux`.
    The four normalised flux objects are never returned; members of the spectral property
    objects that are None take read_input's defaults or are derived from the temperatures
    (include/spartacus_b200.h: ssb200_radsurf_fluxes).  numpy members: ssb200_radsurf_fluxes (host
    arrays).  torch CUDA float64 members, top-of-canopy fluxes and temperatures included:
    ssb200_radsurf_fluxes_device, enqueued on `stream` (cudaStream_t as an int, None = default stream)
    without synchronising.  A mix of numpy arrays and tensors, or a float32 tensor, raises RadsurfError."""
    from . import _abi
    lib = load()
    keep = [np_ for np_ in (top_flux_dn_sw, top_flux_dn_direct_sw, top_flux_dn_lw, ground_temperature,
                            roof_temperature, wall_temperature, clear_air_temperature, veg_temperature,
                            veg_air_temperature)]
    members = list(_float_members(canopy_props, sw_spectral_props, lw_spectral_props, bc_out, sw_flux, lw_flux))
    members += [a for a in keep if a is not None]
    if any(is_torch(v) for v in members):
        return _radsurf_fluxes_device(lib, members, keep, config, canopy_props, sw_spectral_props,
                                      lw_spectral_props, bc_out, istartcol, iendcol, sw_flux, lw_flux, stream)
    structs = marshal(config, canopy_props, sw_spectral_props, lw_spectral_props, bc_out)
    drv = _abi.DriverInputs(*[_abi.dptr(a) for a in keep])
    fsw = sw_flux.as_struct() if sw_flux is not None else None
    flw = lw_flux.as_struct() if lw_flux is not None else None
    s = structs
    rc = lib.ssb200_radsurf_fluxes(_ref(s["config"]), _ref(s["canopy"]), _ref(s["sw"]), _ref(s["lw"]), C.byref(drv),
                                   _ref(s["bc"]), int(istartcol or 0), int(iendcol or 0), _ref(fsw), _ref(flw))
    if rc < 0:
        raise RadsurfError(f"ssb200_radsurf_fluxes failed (rc={rc}): {last_error()}")
    return rc


def _radsurf_fluxes_device(lib, members, keep, config, canopy_props, sw_spectral_props, lw_spectral_props, bc_out,
                           istartcol, iendcol, sw_flux, lw_flux, stream):
    from . import _abi
    if not all(is_torch(v) for v in members):
        raise RadsurfError("radsurf_fluxes: members mix numpy arrays and torch tensors")
    ptr = f64_cuda_ptr("radsurf_fluxes")
    structs = marshal(config, canopy_props, sw_spectral_props, lw_spectral_props, bc_out, ptr=ptr)
    drv = _abi.DriverInputs(*[ptr(a) for a in keep])
    fsw = sw_flux.as_struct(ptr) if sw_flux is not None else None
    flw = lw_flux.as_struct(ptr) if lw_flux is not None else None
    s = structs
    rc = lib.ssb200_radsurf_fluxes_device(_ref(s["config"]), _ref(s["canopy"]), _ref(s["sw"]), _ref(s["lw"]),
                                          C.byref(drv), _ref(s["bc"]), int(istartcol or 0), int(iendcol or 0),
                                          _ref(fsw), _ref(flw), C.c_void_p(stream or 0), None)
    if rc < 0:
        raise RadsurfError(f"ssb200_radsurf_fluxes_device failed (rc={rc}): {last_error()}")
    return rc


def f64_cuda_ptr(where):
    """Address function for the double-precision device entries that check their members: contiguous float64
    torch CUDA tensors only; anything else raises RadsurfError."""
    _dp = C.POINTER(C.c_double)

    def ptr(a):
        if a is None:
            return C.cast(None, _dp)
        import torch
        if is_torch(a) and a.is_cuda and a.dtype == torch.float64 and a.is_contiguous():
            return C.cast(a.data_ptr(), _dp)
        raise RadsurfError(f"{where}: every real member must be a contiguous float64 CUDA tensor")
    return ptr


def _float_members(*objs):
    """Every real array member of the objects: numpy arrays of a float dtype and floating torch tensors."""
    import numpy as np
    for o in objs:
        if o is None:
            continue
        for v in vars(o).values():
            if (isinstance(v, np.ndarray) and v.dtype.kind == "f") or (is_torch(v) and v.is_floating_point()):
                yield v


def _is_f32(a):
    import numpy as np
    if is_torch(a):
        import torch
        return a.dtype == torch.float32
    return a.dtype == np.float32


def f32_ptr(device, where):
    """Address function for the single-precision entries: the _sp structs of the header are
    layout-identical to the double-precision ones, so the same ctypes structs carry float32 addresses.
    device=False accepts C-contiguous float32 numpy arrays, device=True contiguous float32 torch CUDA
    tensors; anything else raises RadsurfError (the double-precision entries keep their own checks)."""
    import numpy as np
    _dp = C.POINTER(C.c_double)

    def ptr(a):
        if a is None:
            return C.cast(None, _dp)
        if device:
            if is_torch(a) and a.is_cuda and _is_f32(a) and a.is_contiguous():
                return C.cast(a.data_ptr(), _dp)
            raise RadsurfError(f"{where}: every real member must be a contiguous float32 CUDA tensor")
        if isinstance(a, np.ndarray) and a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]:
            return a.ctypes.data_as(_dp)
        raise RadsurfError(f"{where}: every real member must be a C-contiguous float32 numpy array")
    return ptr


def to_single(obj):
    """Copy of an API object with every float64 numpy member converted to float32 (what a
    -DSINGLE_PRECISION build of the reference holds: jprb = real32, utilities/parkind1.F90:45-49)."""
    import copy
    import numpy as np
    out = copy.copy(obj)
    for k, v in vars(obj).items():
        if isinstance(v, np.ndarray) and v.dtype == np.float64:
            setattr(out, k, np.ascontiguousarray(v.astype(np.float32)))
    return out


def radsurf_sp(config, canopy_props, sw_spectral_props, lw_spectral_props, bc_out,
               istartcol=None, iendcol=None, sw_norm_dir=None, sw_norm_diff=None,
               lw_internal=None, lw_norm=None, stream=None):
    """radsurf for single-precision (float32) arrays.  numpy members: ssb200_radsurf_sp (the arrays cross
    PCIe as float32).  torch CUDA members: ssb200_radsurf_device_sp, enqueued on `stream` (cudaStream_t
    as an int, None = default stream) without synchronising.  The solve runs in FP64 on the device and
    every output is the FP64 result rounded to float32."""
    lib = load()
    objs = (canopy_props, sw_spectral_props, lw_spectral_props, bc_out, sw_norm_dir, sw_norm_diff, lw_internal, lw_norm)
    members = list(_float_members(*objs))
    device = any(is_torch(v) for v in members)
    if device and not all(is_torch(v) for v in members):
        raise RadsurfError("radsurf_sp: members mix numpy arrays and torch tensors")
    if not all(_is_f32(v) for v in members):
        raise RadsurfError("radsurf_sp: every real array member must be float32")
    structs = marshal(config, canopy_props, sw_spectral_props, lw_spectral_props, bc_out,
                      sw_norm_dir, sw_norm_diff, lw_internal, lw_norm, ptr=f32_ptr(device, "radsurf_sp"))
    if device:
        rc = call_radsurf(lib.ssb200_radsurf_device_sp, structs, istartcol, iendcol,
                          extra=(C.c_void_p(stream or 0), None))
    else:
        rc = call_radsurf(lib.ssb200_radsurf_sp, structs, istartcol, iendcol)
    if rc < 0:
        name = "ssb200_radsurf_device_sp" if device else "ssb200_radsurf_sp"
        raise RadsurfError(f"{name} failed (rc={rc}): {last_error()}")
    return rc


def radsurf_fluxes_sp(config, canopy_props, sw_spectral_props, lw_spectral_props, bc_out, istartcol=None,
                      iendcol=None, sw_flux=None, lw_flux=None, top_flux_dn_sw=None, top_flux_dn_direct_sw=None,
                      top_flux_dn_lw=None, ground_temperature=None, roof_temperature=None, wall_temperature=None,
                      clear_air_temperature=None, veg_temperature=None, veg_air_temperature=None, stream=None):
    """radsurf_fluxes for single-precision (float32) arrays.  Same arguments and defaults as radsurf_fluxes;
    every real member, top-of-canopy flux and temperature must be float32.  numpy arrays:
    ssb200_radsurf_fluxes_sp (the arrays cross PCIe as float32).  torch CUDA tensors:
    ssb200_radsurf_fluxes_device_sp, enqueued on `stream` (cudaStream_t as an int, None = default stream)
    without synchronising.  The solve, emission and scale + sum run in FP64 and every output is the FP64
    result rounded to float32.  A mix of numpy arrays and tensors, or a float64 member, raises RadsurfError."""
    from . import _abi
    lib = load()
    keep = (top_flux_dn_sw, top_flux_dn_direct_sw, top_flux_dn_lw, ground_temperature, roof_temperature,
            wall_temperature, clear_air_temperature, veg_temperature, veg_air_temperature)
    members = list(_float_members(canopy_props, sw_spectral_props, lw_spectral_props, bc_out, sw_flux, lw_flux))
    members += [a for a in keep if a is not None]
    device = any(is_torch(v) for v in members)
    if device and not all(is_torch(v) for v in members):
        raise RadsurfError("radsurf_fluxes_sp: members mix numpy arrays and torch tensors")
    if not all(_is_f32(v) for v in members):
        raise RadsurfError("radsurf_fluxes_sp: every real array member must be float32")
    ptr = f32_ptr(device, "radsurf_fluxes_sp")
    structs = marshal(config, canopy_props, sw_spectral_props, lw_spectral_props, bc_out, ptr=ptr)
    drv = _abi.DriverInputs(*[ptr(a) for a in keep])
    fsw = sw_flux.as_struct(ptr) if sw_flux is not None else None
    flw = lw_flux.as_struct(ptr) if lw_flux is not None else None
    s = structs
    args = (_ref(s["config"]), _ref(s["canopy"]), _ref(s["sw"]), _ref(s["lw"]), C.byref(drv), _ref(s["bc"]),
            int(istartcol or 0), int(iendcol or 0), _ref(fsw), _ref(flw))
    if device:
        name = "ssb200_radsurf_fluxes_device_sp"
        rc = lib.ssb200_radsurf_fluxes_device_sp(*args, C.c_void_p(stream or 0), None)
    else:
        name = "ssb200_radsurf_fluxes_sp"
        rc = lib.ssb200_radsurf_fluxes_sp(*args)
    if rc < 0:
        raise RadsurfError(f"{name} failed (rc={rc}): {last_error()}")
    return rc
