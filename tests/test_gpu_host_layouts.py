"""GPU tests of the host entries (ssb200_radsurf, ssb200_radsurf_sp) on packed layouts whose layers are not
contiguous over a call's columns: the per-layer outputs are then uploaded before the solve, so that layers no
selected column owns come back unchanged."""
import copy

import numpy as np
import pytest

from mixed_case import make_mixed, mixed_config
from spartacus_surface_b200 import radsurf, canopy_flux_type, boundary_conds_out_type
from spartacus_surface_b200.radsurf_canopy_flux import ALL_FIELDS
from spartacus_surface_b200.radsurf_interface import radsurf_sp, to_single

pytestmark = pytest.mark.gpu

POISON = 7.0
BC_FIELDS = ("sw_albedo", "sw_albedo_dir", "lw_emissivity", "lw_emission")


def _shuffled_blocks(cp, seed):
    """Start (0-based) of every column's block of layers when the blocks are packed in a seeded shuffled
    order, and the new row of every row of the contiguous packing."""
    order = np.random.default_rng(seed).permutation(cp.ncol)
    start = np.empty(cp.ncol, dtype=np.int64)
    start[order] = np.concatenate(([0], np.cumsum(cp.nlay[order])[:-1]))
    rows = np.concatenate([start[j] + np.arange(cp.nlay[j]) for j in range(cp.ncol)])
    return start, rows


def _solve(cfg, cp, sw, lw, c1, c2, single):
    """Outputs of one host-entry call on outputs poisoned beforehand, as {object: {member: array}}."""
    cast = to_single if single else (lambda o: o)
    bc = cast(boundary_conds_out_type().allocate(cp.ncol, cfg.nsw, cfg.nlw))
    fl = [cast(canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, n, use_direct=d))
          for n, d in ((cfg.nsw, True), (cfg.nsw, True), (cfg.nlw, False), (cfg.nlw, False))]
    for obj in [bc] + fl:
        for v in vars(obj).values():
            if isinstance(v, np.ndarray) and v.dtype.kind == "f":
                v[...] = POISON
    solve = radsurf_sp if single else radsurf
    assert solve(cfg, cast(cp), cast(sw), cast(lw), bc, c1, c2, *fl) == 0
    names = ("sw_norm_dir", "sw_norm_diff", "lw_internal", "lw_norm")
    out = {n: {k: getattr(f, k) for k in ALL_FIELDS if getattr(f, k) is not None} for n, f in zip(names, fl)}
    out["bc"] = {k: getattr(bc, k) for k in BC_FIELDS}
    return out


@pytest.mark.parametrize("single", [False, True], ids=["radsurf", "radsurf_sp"])
def test_non_contiguous_packed_layers(single):
    """The column blocks of packed layers in a shuffled order, so that the layer span of a column sub-range
    holds layers of unselected columns (mixed tiles: Flat, single-layer urban, ragged layers): the outputs
    equal those of the contiguous layout row for row, and every packed layer no selected column owns keeps
    its poison."""
    cfg = mixed_config(2).consolidate()
    cp, sw, lw = make_mixed(cfg, ncol=300)
    assert cp.ntotlay != cp.ncol
    start, rows = _shuffled_blocks(cp, 23)
    inv = np.empty_like(rows)
    inv[rows] = np.arange(rows.size)

    def permuted(obj):
        out = copy.copy(obj)
        for k, v in vars(obj).items():
            if isinstance(v, np.ndarray) and v.dtype == np.float64 and v.shape[0] == cp.ntotlay:
                setattr(out, k, np.ascontiguousarray(v[inv]))
        return out
    pcp = permuted(cp)
    pcp.istartlay = (start + 1).astype(np.int32)
    for c1, c2 in ((None, None), (37, 263)):
        ref = _solve(cfg, cp, sw, lw, c1, c2, single)
        got = _solve(cfg, pcp, permuted(sw), permuted(lw), c1, c2, single)
        lo, hi = (c1 or 1) - 1, c2 or cp.ncol
        owned = np.zeros(cp.ntotlay, dtype=bool)
        owned[np.concatenate([start[j] + np.arange(cp.nlay[j]) for j in range(lo, hi)])] = True
        if c1 is not None:  # the span of the sub-range holds layers of unselected columns
            span = np.nonzero(owned)[0]
            assert not owned[span[0]:span[-1]].all()
        for n, fields in ref.items():
            for k, v in fields.items():
                g = got[n][k]
                if v.shape[0] == cp.ntotlay:
                    assert np.all(g[~owned] == POISON), (n, k)
                    g = g[rows]
                assert np.array_equal(g, v), (n, k)
