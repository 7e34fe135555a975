"""canopy_flux_type (radsurf/radsurf_canopy_flux.F90:27-91) with the same
type-bound procedures: allocate (:95-166), zero_all, scale (:212-282),
sum (:399-460) and check (:465-542).

scale/sum/check operate with numpy on host arrays; for device-resident
(torch CUDA) members they call the library's device entry points
(ssb200_canopy_flux_*_device), which is the fused "next row" f1 of SURVEY §8.
"""
import ctypes as C

import numpy as np

from . import _abi
from ._arrays import dptr, iptr, is_torch, zeros
from .radsurf_canopy_properties import (ITileFlat, ITileForest, ITileUrban, ITileVegetatedUrban,
                                        ITileSimpleUrban, ITileInfiniteStreet)

COL_FIELDS = ("ground_dn", "ground_net", "ground_vertical_diff", "top_dn", "top_net")
COL_DIR_FIELDS = ("ground_dn_dir", "top_dn_dir")
LAY_URBAN_FIELDS = ("roof_in", "roof_net", "wall_in", "wall_net")
LAY_URBAN_DIR_FIELDS = ("roof_in_dir", "wall_in_dir")
LAY_VEG_FIELDS = ("veg_abs", "veg_air_abs")
PROFILE_FIELDS = ("flux_dn_layer_top", "flux_up_layer_top", "flux_dn_layer_base", "flux_up_layer_base")
PROFILE_DIR_FIELDS = ("flux_dn_dir_layer_top", "flux_dn_dir_layer_base")
SUNLIT_LAY_FIELDS = ("roof_sunlit_frac", "wall_sunlit_frac", "veg_sunlit_frac")
ALL_FIELDS = (COL_FIELDS + COL_DIR_FIELDS + ("ground_sunlit_frac",) + LAY_URBAN_FIELDS + LAY_URBAN_DIR_FIELDS
              + ("roof_sunlit_frac", "wall_sunlit_frac", "clear_air_abs") + LAY_VEG_FIELDS
              + ("veg_abs_dir", "veg_sunlit_frac") + PROFILE_FIELDS + PROFILE_DIR_FIELDS)
SPECTRAL_LAYER_FIELDS = (LAY_URBAN_FIELDS + LAY_URBAN_DIR_FIELDS + ("clear_air_abs",) + LAY_VEG_FIELDS
                         + ("veg_abs_dir",) + PROFILE_FIELDS + PROFILE_DIR_FIELDS)


class canopy_flux_type:
    def __init__(self):
        self.nspec = self.ncol = self.ntotlay = 0
        for name in ALL_FIELDS:
            setattr(self, name, None)

    # -- allocate_canopy_flux (radsurf_canopy_flux.F90:95-166) ---------------
    def allocate(self, config, ncol, ntotlay, nspec, use_direct=True, do_save_flux_profile=True,
                 device=None):
        self.__init__()
        col = lambda: zeros((ncol, nspec), device=device)
        lay = lambda: zeros((ntotlay, nspec), device=device)
        for name in COL_FIELDS:
            setattr(self, name, col())
        if use_direct:
            for name in COL_DIR_FIELDS:
                setattr(self, name, col())
            self.ground_sunlit_frac = zeros((ncol,), device=device)
        if config.do_urban:
            for name in LAY_URBAN_FIELDS:
                setattr(self, name, lay())
            if use_direct:
                for name in LAY_URBAN_DIR_FIELDS:
                    setattr(self, name, lay())
                self.roof_sunlit_frac = zeros((ntotlay,), device=device)
                self.wall_sunlit_frac = zeros((ntotlay,), device=device)
        self.clear_air_abs = lay()
        if config.do_vegetation:
            for name in LAY_VEG_FIELDS:
                setattr(self, name, lay())
            if use_direct:
                self.veg_abs_dir = lay()
                self.veg_sunlit_frac = zeros((ntotlay,), device=device)
        if do_save_flux_profile:
            for name in PROFILE_FIELDS:
                setattr(self, name, lay())
            if use_direct:
                for name in PROFILE_DIR_FIELDS:
                    setattr(self, name, lay())
        self.nspec, self.ncol, self.ntotlay = nspec, ncol, ntotlay
        return self

    def zero_all(self):
        for name in ALL_FIELDS:
            a = getattr(self, name)
            if a is not None:
                if is_torch(a):
                    a.zero_()
                else:
                    a[...] = 0.0

    def fill(self, value):
        """Test helper: poison every allocated member."""
        for name in ALL_FIELDS:
            a = getattr(self, name)
            if a is not None:
                if is_torch(a):
                    a.fill_(value)
                else:
                    a[...] = value

    def is_device(self):
        return is_torch(self.ground_dn)

    def as_struct(self, ptr=dptr):
        """C struct of the members; `ptr` maps an array to the address stored (default: dptr)."""
        c = _abi.CanopyFlux()
        c.nspec, c.ncol, c.ntotlay = int(self.nspec), int(self.ncol), int(self.ntotlay)
        for name in ALL_FIELDS:
            setattr(c, name, ptr(getattr(self, name)))
        return c

    # -- scale_canopy_flux (radsurf_canopy_flux.F90:212-282) -----------------
    def scale(self, nlay, factor):
        """Multiply every flux by factor(nspec, ncol) (array shape (ncol, nspec));
        sunlit fractions are not scaled, as in the reference."""
        if factor.shape[-1] != self.nspec:
            raise ValueError("spectral resolution mismatch when scaling canopy fluxes")
        if self.is_device():
            from ._lib import load, last_error
            nlay = np.ascontiguousarray(nlay, dtype=np.int32)
            start = np.ones(nlay.size, dtype=np.int64)
            start[1:] = 1 + np.cumsum(nlay.astype(np.int64))[:-1]
            start = start.astype(np.int32)
            s = self.as_struct()
            rc = load().ssb200_canopy_flux_scale_device(C.byref(s), iptr(nlay), iptr(start),
                                                        C.c_void_p(factor.data_ptr()), None)
            if rc != 0:
                raise RuntimeError(f"ssb200_canopy_flux_scale_device failed ({rc}): {last_error()}")
            return
        indcol = np.repeat(np.arange(self.ncol), np.asarray(nlay))
        for name in COL_FIELDS + COL_DIR_FIELDS:
            a = getattr(self, name)
            if a is not None:
                a *= factor
        for name in SPECTRAL_LAYER_FIELDS:
            a = getattr(self, name)
            if a is not None:
                a *= factor[indcol]

    # -- sum_canopy_flux (radsurf_canopy_flux.F90:399-460) -------------------
    def sum(self, flux1, flux2):
        if self.ground_dn is None:
            raise RuntimeError("Attempt to sum canopy fluxes to an unallocated canopy flux object")
        if self.is_device():
            from ._lib import load, last_error
            so, s1, s2 = self.as_struct(), flux1.as_struct(), flux2.as_struct()
            rc = load().ssb200_canopy_flux_sum_device(C.byref(so), C.byref(s1), C.byref(s2), None)
            if rc != 0:
                raise RuntimeError(f"ssb200_canopy_flux_sum_device failed ({rc}): {last_error()}")
            return
        for name in ALL_FIELDS:
            out = getattr(self, name)
            a, b = getattr(flux1, name), getattr(flux2, name)
            if out is not None and a is not None and b is not None:
                out[...] = a + b

    # -- check_canopy_flux (radsurf_canopy_flux.F90:465-542) -----------------
    def check(self, canopy_props, istartcol=None, iendcol=None, iverbose=3, file=None):
        """Return the per-column energy-budget table
        [ground, air, wall, roof, veg, air-veg, top, residual] and optionally print it."""
        icol1 = 1 if istartcol is None else istartcol
        icol2 = self.ncol if iendcol is None else iendcol
        get = (lambda a: a.cpu().numpy()) if self.is_device() else (lambda a: a)
        rows = []
        if iverbose >= 3:
            print("Column  Ground      Air     Wall     Roof      Veg  Air-veg      Top   Residual", file=file)
        for jcol in range(icol1 - 1, icol2):
            l1 = int(canopy_props.istartlay[jcol]) - 1
            l2 = l1 + int(canopy_props.nlay[jcol])
            irep = int(canopy_props.i_representation[jcol])
            ground_net = float(get(self.ground_net)[jcol].sum())
            top_net = float(get(self.top_net)[jcol].sum())
            clear_air_net = float(get(self.clear_air_abs)[l1:l2].sum()) if irep != ITileFlat else 0.0
            if irep in (ITileUrban, ITileVegetatedUrban, ITileSimpleUrban, ITileInfiniteStreet):
                roof_net = float(get(self.roof_net)[l1:l2].sum())
                wall_net = float(get(self.wall_net)[l1:l2].sum())
            else:
                roof_net = wall_net = 0.0
            if irep in (ITileForest, ITileVegetatedUrban):
                veg_net = float(get(self.veg_abs)[l1:l2].sum())
                veg_air_net = float(get(self.veg_air_abs)[l1:l2].sum())
            else:
                veg_net = veg_air_net = 0.0
            residual = ground_net + clear_air_net + wall_net + roof_net + veg_net + veg_air_net - top_net
            rows.append([ground_net, clear_air_net, wall_net, roof_net, veg_net, veg_air_net, top_net, residual])
            if iverbose >= 3:
                print("%5d%9.3f%9.3f%9.3f%9.3f%9.3f%9.3f%9.3f%11.3e" % ((jcol + 1,) + tuple(rows[-1])), file=file)
        return np.array(rows)
