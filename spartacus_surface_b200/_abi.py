"""ctypes mirror of include/spartacus_b200.h (the C ABI of the product library).

Field order and types must match the header exactly; tests/test_abi.py checks
sizes against the compiled library.
"""
import ctypes as C

MAX_NSTREAM = 16

TILE_FLAT, TILE_FOREST, TILE_URBAN, TILE_VEGETATED_URBAN, TILE_SIMPLE_URBAN, TILE_INFINITE_STREET = range(6)

OK = 0
ERR_ARG, ERR_SHAPE, ERR_UNSUPPORTED, ERR_CUDA, ERR_NOGPU, ERR_SIMPLE_URBAN_LAYERS = -1, -2, -3, -4, -5, -6

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_darr = C.c_double * MAX_NSTREAM


class LegendreGauss(C.Structure):
    _fields_ = [
        ("nstream", C.c_int32), ("pad_", C.c_int32),
        ("mu", _darr), ("sin_ang", _darr), ("tan_ang", _darr),
        ("weight", _darr), ("hweight", _darr), ("vweight", _darr),
        ("vadjustment", C.c_double), ("vadjustment2", C.c_double),
    ]


class Config(C.Structure):
    _fields_ = [
        ("do_sw", C.c_int32), ("do_lw", C.c_int32), ("use_sw_direct_albedo", C.c_int32),
        ("do_vegetation", C.c_int32), ("do_urban", C.c_int32),
        ("n_vegetation_region_forest", C.c_int32), ("n_vegetation_region_urban", C.c_int32),
        ("nsw", C.c_int32), ("nlw", C.c_int32),
        ("use_symmetric_vegetation_scale_forest", C.c_int32),
        ("use_symmetric_vegetation_scale_urban", C.c_int32),
        ("iverbose", C.c_int32),
        ("vegetation_isolation_factor_forest", C.c_double),
        ("vegetation_isolation_factor_urban", C.c_double),
        ("min_vegetation_fraction", C.c_double),
        ("min_building_fraction", C.c_double),
        ("lg_sw_forest", LegendreGauss), ("lg_sw_urban", LegendreGauss),
        ("lg_lw_forest", LegendreGauss), ("lg_lw_urban", LegendreGauss),
    ]


class CanopyProperties(C.Structure):
    _fields_ = [
        ("ncol", C.c_int32), ("ntotlay", C.c_int32),
        ("nlay", _ip), ("istartlay", _ip), ("i_representation", _ip),
        ("cos_sza", _dp), ("dz", _dp),
        ("building_fraction", _dp), ("building_scale", _dp),
        ("veg_fraction", _dp), ("veg_scale", _dp), ("veg_ext", _dp),
        ("veg_fsd", _dp), ("veg_contact_fraction", _dp),
    ]


class SwSpectralProperties(C.Structure):
    _fields_ = [
        ("nspec", C.c_int32), ("pad_", C.c_int32),
        ("air_ext", _dp), ("air_ssa", _dp), ("veg_ssa", _dp), ("ground_albedo", _dp),
        ("roof_albedo", _dp), ("wall_albedo", _dp), ("wall_specular_frac", _dp),
        ("ground_albedo_dir", _dp), ("roof_albedo_dir", _dp),
    ]


class LwSpectralProperties(C.Structure):
    _fields_ = [
        ("nspec", C.c_int32), ("pad_", C.c_int32),
        ("air_ext", _dp), ("air_ssa", _dp), ("clear_air_planck", _dp),
        ("veg_ssa", _dp), ("veg_planck", _dp), ("veg_air_planck", _dp),
        ("ground_emissivity", _dp), ("ground_emission", _dp),
        ("roof_emissivity", _dp), ("wall_emissivity", _dp),
        ("roof_emission", _dp), ("wall_emission", _dp),
    ]


FLUX_COL_FIELDS = ["ground_dn", "ground_net", "ground_vertical_diff", "top_dn", "top_net"]
FLUX_COL_DIR_FIELDS = ["ground_dn_dir", "top_dn_dir"]
FLUX_LAY_URBAN_FIELDS = ["roof_in", "roof_net", "wall_in", "wall_net"]
FLUX_LAY_URBAN_DIR_FIELDS = ["roof_in_dir", "wall_in_dir"]
FLUX_LAY_VEG_FIELDS = ["veg_abs", "veg_air_abs"]
FLUX_PROFILE_FIELDS = ["flux_dn_layer_top", "flux_up_layer_top", "flux_dn_layer_base", "flux_up_layer_base"]
FLUX_PROFILE_DIR_FIELDS = ["flux_dn_dir_layer_top", "flux_dn_dir_layer_base"]


class CanopyFlux(C.Structure):
    _fields_ = [
        ("nspec", C.c_int32), ("ncol", C.c_int32), ("ntotlay", C.c_int32), ("pad_", C.c_int32),
        ("ground_dn", _dp), ("ground_net", _dp), ("ground_vertical_diff", _dp),
        ("top_dn", _dp), ("top_net", _dp),
        ("ground_dn_dir", _dp), ("top_dn_dir", _dp), ("ground_sunlit_frac", _dp),
        ("roof_in", _dp), ("roof_net", _dp), ("wall_in", _dp), ("wall_net", _dp),
        ("roof_in_dir", _dp), ("wall_in_dir", _dp),
        ("roof_sunlit_frac", _dp), ("wall_sunlit_frac", _dp),
        ("clear_air_abs", _dp), ("veg_abs", _dp), ("veg_air_abs", _dp),
        ("veg_abs_dir", _dp), ("veg_sunlit_frac", _dp),
        ("flux_dn_layer_top", _dp), ("flux_up_layer_top", _dp),
        ("flux_dn_layer_base", _dp), ("flux_up_layer_base", _dp),
        ("flux_dn_dir_layer_top", _dp), ("flux_dn_dir_layer_base", _dp),
    ]


class BoundaryCondsOut(C.Structure):
    _fields_ = [
        ("sw_albedo", _dp), ("sw_albedo_dir", _dp),
        ("lw_emissivity", _dp), ("lw_emission", _dp),
    ]


# Every symbol include/spartacus_b200.h declares (tests check the built library
# exports all of them).
class DriverInputs(C.Structure):
    """ssb200_driver_inputs: what the reference driver feeds around radsurf (top-of-canopy
    fluxes for scale/sum, temperatures for the LW emission stage)."""
    _fields_ = [(k, _dp) for k in ("top_flux_dn_sw", "top_flux_dn_direct_sw", "top_flux_dn_lw",
                                   "ground_temperature", "roof_temperature", "wall_temperature",
                                   "clear_air_temperature", "veg_temperature", "veg_air_temperature")]


EXPORTED_SYMBOLS = [
    "ssb200_version", "ssb200_abi_sizes", "ssb200_last_error", "ssb200_device_count", "ssb200_set_device",
    "ssb200_legendre_gauss_init", "ssb200_radsurf", "ssb200_radsurf_device", "ssb200_radsurf_fluxes",
    "ssb200_radsurf_sp", "ssb200_radsurf_fluxes_sp", "ssb200_radsurf_device_sp", "ssb200_radsurf_fluxes_device",
    "ssb200_radsurf_fluxes_device_sp", "ssb200_kernel_launch_count", "ssb200_set_profiling",
    "ssb200_last_kernel_times_ms", "ssb200_last_kernel_counts",
    "ssb200_release", "ssb200_set_option", "ssb200_canopy_flux_scale_device", "ssb200_canopy_flux_sum_device",
    "ssb200_canopy_flux_check_device", "ssb200_calc_simple_spectrum_lw_device", "ssb200_measure_fp64_peak_tflops",
]


def dptr(arr):
    """double* of a numpy float64 C-contiguous array (or NULL for None)."""
    if arr is None:
        return C.cast(None, _dp)
    return arr.ctypes.data_as(_dp)


def iptr(arr):
    if arr is None:
        return C.cast(None, _ip)
    return arr.ctypes.data_as(_ip)
