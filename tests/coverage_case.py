"""Configuration matrix with asymmetric inputs, shared by the CPU (host check) and GPU coverage tests.

The dispatcher picks a register-resident kernel per (pass, regions, streams, urban) of every column
class (csrc/ssb_fast_kernels.cuh) and the generic kernels for 5-8 streams.  SPECS lists a few
configurations that together reach every register-resident shape (pass x NREG 1-3 x NS 1-4 x URBAN)
and every generic stream count 5-8 in both passes, on forest and on urban tiles; `shapes(spec)` says
which ones a spec reaches, derived the way build_plan / class_cfg derive the column classes
(csrc/ssb_driver.hpp): forest columns get n_vegetation_region_forest + 1 regions, urban columns 1,
vegetated-urban columns n_vegetation_region_urban + 1.

`make_case` starts from the mixed case (tests/mixed_case.py: every tile type, ragged layers, night
columns, several spectral intervals) and breaks the symmetries that would let a kernel confuse one
input with another: vegetation, vegetation-air and clear-air Planck functions all differ (and vary
from layer to layer), longwave air scatters, clear air absorbs far above the small-field floor of
tests/parity.py, the direct roof and ground albedos differ from the diffuse ones and the wall
reflection is partly specular.
"""
import functools

import numpy as np

import oracle_lib
from mixed_case import make_mixed
from spartacus_surface_b200 import config_type, canopy_flux_type, boundary_conds_out_type
from spartacus_surface_b200.radsurf_canopy_flux import ALL_FIELDS
from spartacus_surface_b200.radsurf_canopy_properties import (ITileForest, ITileUrban,
                                                              ITileVegetatedUrban)

NCOL = 40
POISON = 7.0
FLUX_NAMES = ("sw_norm_dir", "sw_norm_diff", "lw_internal", "lw_norm")
BC_FIELDS = ("sw_albedo", "sw_albedo_dir", "lw_emissivity", "lw_emission")
FAST_NS = (1, 2, 3, 4)
GENERIC_NS = (5, 6, 7, 8)


def _spec(name, nvf, forest_ns, nvu, urban_ns, **extra):
    s = dict(name=name, n_vegetation_region_forest=nvf, n_vegetation_region_urban=nvu,
             n_stream_sw_forest=forest_ns[0], n_stream_lw_forest=forest_ns[1],
             n_stream_sw_urban=urban_ns[0], n_stream_lw_urban=urban_ns[1])
    s.update(extra)
    return s


# (forest regions - 1, (SW, LW) forest streams, urban vegetation regions, (SW, LW) urban streams)
SPECS = [
    _spec("default", 1, (4, 4), 1, (4, 4)),  # the reference's defaults: one vegetation region, 4 streams
    _spec("r3_s2_iso05_asym", 2, (2, 2), 2, (2, 2), vegetation_isolation_factor_forest=0.5,
          vegetation_isolation_factor_urban=0.5, use_symmetric_vegetation_scale_forest=False,
          use_symmetric_vegetation_scale_urban=False),
    _spec("r3_s4_iso10", 2, (4, 4), 2, (4, 4), vegetation_isolation_factor_forest=1.0,
          vegetation_isolation_factor_urban=1.0, use_symmetric_vegetation_scale_urban=False),
    _spec("r3_s1_u13", 2, (1, 1), 2, (1, 3)),
    _spec("r3_s3_u31", 2, (3, 3), 2, (3, 1)),
    _spec("f1r_s12_u2r_s23", 0, (1, 2), 1, (2, 3)),
    _spec("f1r_s21_u2r_s31", 0, (2, 1), 1, (3, 1)),
    _spec("f1r_s34_u2r_s12", 0, (3, 4), 1, (1, 2)),
    _spec("f1r_s43_u1r_s65", 0, (4, 3), 0, (6, 5), use_sw_direct_albedo=False),
    _spec("f2r_s13_u1r_s87", 1, (1, 3), 0, (8, 7)),
    _spec("f2r_s21_u1r_s24", 1, (2, 1), 0, (2, 4)),
    _spec("f2r_s32_u3r_s34", 1, (3, 2), 2, (3, 4)),
    _spec("f3r_s56_u2r_s11", 2, (5, 6), 1, (1, 1), use_sw_direct_albedo=False),
    _spec("f2r_s78_u3r_s21", 1, (7, 8), 2, (2, 1), vegetation_isolation_factor_urban=0.5),
]
BY_NAME = {s["name"]: s for s in SPECS}
DEFAULT = "default"


def full_shape_set():
    """Every register-resident shape the dispatcher has a kernel for."""
    return {(p, nreg, ns, urban) for p in ("sw", "lw") for nreg in (1, 2, 3) for ns in FAST_NS for urban in (0, 1)}


def classes(spec):
    """(urban, nreg) of the column classes of a spec's mixed case (build_plan)."""
    return {(0, spec["n_vegetation_region_forest"] + 1), (1, 1), (1, spec["n_vegetation_region_urban"] + 1)}


def streams(spec, pass_, urban):
    kind = "urban" if urban else "forest"
    return spec[f"n_stream_{pass_}_{kind}"]


def shapes(spec):
    """(pass, nreg, ns, urban) of every register-resident kernel shape the spec launches."""
    return {(p, nreg, streams(spec, p, urban), urban) for urban, nreg in classes(spec) for p in ("sw", "lw")
            if streams(spec, p, urban) in FAST_NS}


def generic_uses(spec):
    """(pass, ns, urban) of every class and pass that runs the generic kernels (5-8 streams)."""
    return {(p, streams(spec, p, urban), urban) for urban, _ in classes(spec) for p in ("sw", "lw")
            if streams(spec, p, urban) in GENERIC_NS}


def make_config(spec, nsw=2, nlw=3, legendre_gauss_init=oracle_lib.legendre_gauss_init):
    kw = {k: v for k, v in spec.items() if k != "name"}
    kw.setdefault("use_sw_direct_albedo", True)
    cfg = config_type(do_sw=True, do_lw=True, nsw=nsw, nlw=nlw, **kw)
    return cfg.consolidate(legendre_gauss_init)


def make_case(spec, ncol=NCOL, nsw=2, nlw=3):
    """(config, canopy_props, sw, lw): the mixed case under `spec` with the input symmetries broken.
    Deterministic (fixed seeds); the quadrature tables are the oracle's."""
    cfg = make_config(spec, nsw, nlw)
    cp, sw, lw = make_mixed(cfg, ncol=ncol, seed=11)
    rng = np.random.default_rng(2024)
    nt = cp.ntotlay
    # longwave Planck functions: vegetation warmer, vegetation air cooler than clear air, both by a few
    # percent that differ from layer to layer and between intervals
    base = lw.clear_air_planck
    lw.veg_planck = np.ascontiguousarray(base * (1.0 + rng.uniform(0.03, 0.08, size=base.shape)))
    lw.veg_air_planck = np.ascontiguousarray(base * (1.0 - rng.uniform(0.02, 0.06, size=base.shape)))
    lw.clear_air_planck = np.ascontiguousarray(base * (1.0 + rng.uniform(-0.01, 0.01, size=base.shape)))
    # scattering, absorbing air (optical depths of order 0.1-1 over a column)
    lw.air_ssa = np.ascontiguousarray(rng.uniform(0.2, 0.4, size=(nt, cfg.nlw)))
    lw.air_ext = np.ascontiguousarray(rng.uniform(0.01, 0.04, size=(nt, cfg.nlw)))
    sw.air_ext = np.ascontiguousarray(rng.uniform(0.005, 0.02, size=(nt, cfg.nsw)))
    sw.air_ssa = np.ascontiguousarray(rng.uniform(0.6, 0.95, size=(nt, cfg.nsw)))
    # direct albedos differ from the diffuse ones; partly specular walls
    sw.roof_albedo_dir = np.ascontiguousarray(sw.roof_albedo * rng.uniform(0.5, 0.8, size=sw.roof_albedo.shape))
    sw.ground_albedo_dir = np.ascontiguousarray(sw.ground_albedo * rng.uniform(0.6, 0.9, size=sw.ground_albedo.shape))
    sw.wall_specular_frac = np.ascontiguousarray(rng.uniform(0.2, 0.6, size=(nt, cfg.nsw)))
    return cfg, cp, sw, lw


def run(cfg, cp, sw, lw, solver):
    """(outputs {object: {field: array}}, status) of one call; every output entry starts at POISON."""
    bc = boundary_conds_out_type().allocate(cp.ncol, cfg.nsw, cfg.nlw)
    for k in BC_FIELDS:
        getattr(bc, k)[...] = POISON
    fl = [canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, n, use_direct=d)
          for n, d in ((cfg.nsw, True), (cfg.nsw, True), (cfg.nlw, False), (cfg.nlw, False))]
    for f in fl:
        f.fill(POISON)
    status = solver(cfg, cp, sw, lw, bc, None, None, *fl)
    out = {n: {k: getattr(f, k) for k in ALL_FIELDS if getattr(f, k) is not None} for n, f in zip(FLUX_NAMES, fl)}
    out["bc"] = {k: getattr(bc, k) for k in BC_FIELDS}
    return out, status


@functools.lru_cache(maxsize=None)
def oracle_runs(name):
    """{"fma", "nofma", "quad"}: the oracle's outputs for a spec (computed once per session; read-only)."""
    cfg, cp, sw, lw = make_case(BY_NAME[name])
    res = {}
    for tag, kw in (("fma", {}), ("nofma", dict(nofma=True)), ("quad", dict(quad=True))):
        out, status = run(cfg, cp, sw, lw, oracle_lib.make_solver(**kw))
        assert status == 0, (name, tag, status)
        for fields in out.values():
            for v in fields.values():
                v.setflags(write=False)
        res[tag] = out
    return res


def poison_mismatches(got, ref):
    """(object, field) whose entries left at POISON differ from those of `ref`."""
    return [(n, k) for n, f in ref.items() for k, v in f.items()
            if not np.array_equal(np.asarray(got[n][k]) == POISON, v == POISON)]


def unpoison(out, ref):
    """`out` with the entries `ref` leaves at POISON set to zero (they would otherwise set the field
    scale of the parity measure)."""
    return {n: {k: np.where(v == POISON, 0.0, np.asarray(out[n][k], dtype=np.float64)) for k, v in f.items()}
            for n, f in ref.items()}


def columns(cp, urban, nreg, spec):
    """Column indices of the class (urban, nreg) of a spec's mixed case."""
    rep = cp.i_representation
    if urban:
        m = np.zeros(cp.ncol, dtype=bool)
        if nreg == 1:
            m |= rep == ITileUrban
        if spec["n_vegetation_region_urban"] + 1 == nreg:
            m |= rep == ITileVegetatedUrban
        return np.nonzero(m)[0]
    return np.nonzero(rep == ITileForest)[0] if spec["n_vegetation_region_forest"] + 1 == nreg else np.array([], int)
