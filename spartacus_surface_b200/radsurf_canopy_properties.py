"""canopy_properties_type (radsurf/radsurf_canopy_properties.F90:53-110)."""
import numpy as np

from . import _abi
from ._arrays import dptr, iptr

# Tile representation codes (radsurf_canopy_properties.F90:26-33)
ITileFlat, ITileForest, ITileUrban, ITileVegetatedUrban, ITileSimpleUrban, ITileInfiniteStreet = range(6)
TileRepresentationName = ("Flat", "Forest", "Urban", "VegetatedUrban", "SimpleUrban", "InfiniteStreet")

_REAL_LAYER = ("dz", "building_fraction", "building_scale", "veg_fraction", "veg_scale", "veg_ext",
               "veg_fsd", "veg_contact_fraction")
_TEMPERATURES = ("roof_temperature", "wall_temperature", "clear_air_temperature", "veg_temperature",
                 "veg_air_temperature")


class canopy_properties_type:
    """Geometric / spectrally independent canopy description.

    nlay, istartlay (1-based, like the reference) and i_representation are
    int32 host arrays (ncol); the per-layer members are packed ragged
    (ntotlay) arrays; temperatures are only used upstream of radsurf
    (radsurf_simple_spectrum.F90:41-66).
    """

    def __init__(self):
        self.ncol = 0
        self.ntotlay = 0
        self.nlay = self.istartlay = self.i_representation = None
        self.cos_sza = None
        self.ground_temperature = None
        for name in _REAL_LAYER + _TEMPERATURES:
            setattr(self, name, None)

    def set_layers(self, nlay):
        """Fill ncol/ntotlay/istartlay from nlay (driver/spartacus_surface_read_input.F90:73-92)."""
        self.nlay = np.ascontiguousarray(nlay, dtype=np.int32)
        self.ncol = int(self.nlay.size)
        self.ntotlay = int(self.nlay.sum())
        start = np.ones(self.ncol, dtype=np.int64)
        start[1:] = 1 + np.cumsum(self.nlay.astype(np.int64))[:-1]
        self.istartlay = start.astype(np.int32)
        return self

    def as_struct(self, ptr=dptr):
        """C struct of the members; `ptr` maps an array to the address stored (default: dptr)."""
        c = _abi.CanopyProperties()
        c.ncol, c.ntotlay = int(self.ncol), int(self.ntotlay)
        c.nlay, c.istartlay = iptr(self.nlay), iptr(self.istartlay)
        c.i_representation = iptr(self.i_representation)
        c.cos_sza = ptr(self.cos_sza)
        for name in _REAL_LAYER:
            setattr(c, name, ptr(getattr(self, name)))
        return c
