"""sw_spectral_properties_type (radsurf/radsurf_sw_spectral_properties.F90:24-49)."""
from . import _abi
from ._arrays import dptr

_MEMBERS = ("air_ext", "air_ssa", "veg_ssa", "ground_albedo", "roof_albedo", "wall_albedo",
            "wall_specular_frac", "ground_albedo_dir", "roof_albedo_dir")


class sw_spectral_properties_type:
    """Members are (ntotlay, nsw) or (ncol, nsw) C-contiguous float64 arrays
    (= Fortran (nsw, ntotlay) / (nsw, ncol)); None when not allocated."""

    def __init__(self, nspec=1):
        self.nspec = nspec
        for name in _MEMBERS:
            setattr(self, name, None)

    def as_struct(self, ptr=dptr):
        """C struct of the members; `ptr` maps an array to the address stored (default: dptr)."""
        c = _abi.SwSpectralProperties()
        c.nspec = int(self.nspec)
        for name in _MEMBERS:
            setattr(c, name, ptr(getattr(self, name)))
        return c
