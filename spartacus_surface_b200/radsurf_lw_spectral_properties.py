"""lw_spectral_properties_type (radsurf/radsurf_lw_spectral_properties.F90:24-57)."""
from . import _abi
from ._arrays import dptr

StefanBoltzmann = 5.67037321e-8  # radtool/radiation_constants.F90:26

_MEMBERS = ("air_ext", "air_ssa", "clear_air_planck", "veg_ssa", "veg_planck", "veg_air_planck",
            "ground_emissivity", "ground_emission", "roof_emissivity", "wall_emissivity",
            "roof_emission", "wall_emission")


class lw_spectral_properties_type:
    def __init__(self, nspec=1):
        self.nspec = nspec
        for name in _MEMBERS:
            setattr(self, name, None)

    def calc_monochromatic_emission(self, canopy_props):
        """radsurf_lw_spectral_properties.F90:161-199 (host-side input preparation)."""
        cp = canopy_props
        if cp.ground_temperature is not None and self.ground_emissivity is not None:
            self.ground_emission = (StefanBoltzmann * self.ground_emissivity[:, :1]
                                    * cp.ground_temperature[:, None] ** 4).copy()
        if cp.roof_temperature is not None and self.roof_emissivity is not None:
            self.roof_emission = (StefanBoltzmann * self.roof_emissivity[:, :1]
                                  * cp.roof_temperature[:, None] ** 4).copy()
            self.wall_emission = (StefanBoltzmann * self.wall_emissivity[:, :1]
                                  * cp.wall_temperature[:, None] ** 4).copy()

    def as_struct(self, ptr=dptr):
        """C struct of the members; `ptr` maps an array to the address stored (default: dptr)."""
        c = _abi.LwSpectralProperties()
        c.nspec = int(self.nspec)
        for name in _MEMBERS:
            setattr(c, name, ptr(getattr(self, name)))
        return c
