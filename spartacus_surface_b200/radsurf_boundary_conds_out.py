"""boundary_conds_out_type (radsurf/radsurf_boundary_conds_out.F90:24-39)."""
from . import _abi
from ._arrays import dptr, zeros


class boundary_conds_out_type:
    def __init__(self):
        self.sw_albedo = self.sw_albedo_dir = self.lw_emissivity = self.lw_emission = None

    def allocate(self, ncol, nsw, nlw, device=None):
        if nsw > 0:
            self.sw_albedo = zeros((ncol, nsw), device=device)
            self.sw_albedo_dir = zeros((ncol, nsw), device=device)
        if nlw > 0:
            self.lw_emissivity = zeros((ncol, nlw), device=device)
            self.lw_emission = zeros((ncol, nlw), device=device)
        return self

    def as_struct(self, ptr=dptr):
        """C struct of the members; `ptr` maps an array to the address stored (default: dptr)."""
        c = _abi.BoundaryCondsOut()
        for name in ("sw_albedo", "sw_albedo_dir", "lw_emissivity", "lw_emission"):
            setattr(c, name, ptr(getattr(self, name)))
        return c
