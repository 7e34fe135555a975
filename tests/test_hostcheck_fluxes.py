"""The summing scatter of ssb200_radsurf_fluxes_device on the CPU: the serial Dispatcher of tests/hostcheck
run with the sum descriptor (hostcheck_radsurf_summed, tests/hostcheck/hostcheck_summed.cpp), against
hostcheck_radsurf followed by canopy_flux_type.scale / .sum in numpy, the steps of the reference driver
(driver:250-261).  Both run the register-resident bodies through the level-major staging; the summed run
writes the scaled sum of the two normalised objects straight from the staging buffers, so every per-layer
member must match bit for bit.
The per-column members, which the device entry scales and sums in a separate launch, are summed here in
numpy from the normalised objects the summed run leaves."""
import copy
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import golden_io
import hostcheck_lib
import oracle_lib
from degenerate_case import make_degenerate
from mixed_case import mixed_config, make_mixed
from spartacus_surface_b200 import config_type, canopy_flux_type, boundary_conds_out_type
from spartacus_surface_b200 import _abi
from spartacus_surface_b200.radsurf_canopy_flux import (COL_FIELDS, COL_DIR_FIELDS,
                                                        SPECTRAL_LAYER_FIELDS, SUNLIT_LAY_FIELDS)
from spartacus_surface_b200.radsurf_canopy_properties import (ITileFlat, ITileForest, ITileUrban, ITileSimpleUrban,
                                                              ITileInfiniteStreet)
from spartacus_surface_b200.radsurf_interface import marshal
from spartacus_surface_b200.synthetic import make_synthetic

POISON = 7.0
NOT_STAGED = -100
PER_COLUMN = COL_FIELDS + COL_DIR_FIELDS


SUMMED_SRC = os.path.join(os.path.dirname(hostcheck_lib.SRC), "hostcheck_summed.cpp")
SUMMED_SO = os.path.join(os.path.dirname(hostcheck_lib.SO), "libhostcheck_summed.so")
_summed_handle = None


def _summed_lib():
    """tests/_build/libhostcheck_summed.so: the host check plus hostcheck_radsurf_summed, built with the flags
    of libhostcheck.so (no FMA contraction)."""
    global _summed_handle
    if _summed_handle is None:
        deps = [SUMMED_SRC, hostcheck_lib.SRC, os.path.join(os.path.dirname(SUMMED_SRC), "asymtx_qr.hpp"),
                os.path.join(hostcheck_lib.ROOT, "include", "spartacus_b200.h")]
        deps += [os.path.join(hostcheck_lib.CSRC, f) for f in os.listdir(hostcheck_lib.CSRC) if f.endswith((".cuh", ".hpp"))]
        if not (os.path.exists(SUMMED_SO) and all(os.path.getmtime(SUMMED_SO) >= os.path.getmtime(d) for d in deps)):
            os.makedirs(os.path.dirname(SUMMED_SO), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                                   "-Wno-maybe-uninitialized", "-o", SUMMED_SO, SUMMED_SRC])
        lib = C.CDLL(SUMMED_SO)
        P = C.POINTER
        lib.hostcheck_radsurf_summed.argtypes = (
            [P(_abi.Config), P(_abi.CanopyProperties), P(_abi.SwSpectralProperties), P(_abi.LwSpectralProperties),
             P(_abi.BoundaryCondsOut), C.c_int32, C.c_int32] + [P(_abi.CanopyFlux)] * 6
            + [P(C.c_double)] * 3 + [C.c_int64])
        _summed_handle = lib
    return _summed_handle


def _ptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _ref(s):
    return C.byref(s) if s is not None else None


def _factors(cfg, ncol, seed):
    rng = np.random.default_rng(seed)
    top_sw = rng.uniform(200.0, 900.0, size=(ncol, cfg.nsw))
    top_dir = np.ascontiguousarray(top_sw * rng.uniform(0.2, 0.9, size=(ncol, cfg.nsw)))
    top_lw = rng.uniform(250.0, 400.0, size=(ncol, cfg.nlw))
    return top_sw, top_dir, top_lw


def _flux(cfg, ncol, ntot, nspec, direct, profiles):
    return canopy_flux_type().allocate(cfg, ncol, ntot, nspec, use_direct=direct, do_save_flux_profile=profiles)


def _owned_layers(cp, c1, c2):
    """Mask of the packed layers owned by the non-Flat columns c1..c2 (1-based)."""
    owned = np.zeros(cp.ntotlay, dtype=bool)
    for j in range(c1 - 1, c2):
        if cp.i_representation[j] != ITileFlat:
            s = int(cp.istartlay[j]) - 1
            owned[s:s + int(cp.nlay[j])] = True
    return owned


def _reference(cfg, cp, sw, lw, c1, c2, shapes, factors, budget):
    """hostcheck_radsurf on zeroed normalised objects, then scale and sum in numpy."""
    top_sw, top_dir, top_lw = factors
    bc = boundary_conds_out_type().allocate(cp.ncol, cfg.nsw, cfg.nlw)
    norm = [_flux(cfg, cp.ncol, cp.ntotlay, *s) for s in shapes for _ in range(2)]
    rc = hostcheck_lib.make_solver(budget_doubles=budget, fast=True)(cfg, cp, sw, lw, bc, c1, c2, *norm)
    assert rc == 0
    norm[0].scale(cp.nlay, top_dir)
    norm[1].scale(cp.nlay, top_sw - top_dir)
    norm[3].scale(cp.nlay, top_lw)
    out = [_flux(cfg, cp.ncol, cp.ntotlay, *s) for s in shapes]
    out[0].sum(norm[0], norm[1])
    out[1].sum(norm[2], norm[3])
    return bc, out


def _summed(cfg, cp, sw, lw, c1, c2, shapes, factors, budget):
    """hostcheck_radsurf_summed on poisoned summed objects; per-column members summed in numpy."""
    top_sw, top_dir, top_lw = factors
    bc = boundary_conds_out_type().allocate(cp.ncol, cfg.nsw, cfg.nlw)
    out = [_flux(cfg, cp.ncol, cp.ntotlay, *s) for s in shapes]
    for o in out:
        o.fill(POISON)
    norm = []
    for o in out:  # per-column members zeroed, per-layer members: the summed object's arrays (markers only)
        for _ in range(2):
            n = copy.copy(o)
            for k in PER_COLUMN + ("ground_sunlit_frac",):
                if getattr(o, k) is not None:
                    setattr(n, k, np.zeros_like(getattr(o, k)))
            norm.append(n)
    s = marshal(cfg, cp, sw, lw, bc, *norm)
    fsw, flw = out[0].as_struct(), out[1].as_struct()
    rc = _summed_lib().hostcheck_radsurf_summed(
        _ref(s["config"]), _ref(s["canopy"]), _ref(s["sw"]), _ref(s["lw"]), _ref(s["bc"]), int(c1 or 0),
        int(c2 or 0), _ref(s["sw_norm_dir"]), _ref(s["sw_norm_diff"]), _ref(s["lw_internal"]), _ref(s["lw_norm"]),
        C.byref(fsw), C.byref(flw), _ptr(top_sw), _ptr(top_dir), _ptr(top_lw), budget)
    if rc == NOT_STAGED:
        return None
    assert rc == 0
    for o, a, b, fa, fb in ((out[0], norm[0], norm[1], top_dir, top_sw - top_dir),
                            (out[1], norm[2], norm[3], None, top_lw)):
        for k in PER_COLUMN:
            if getattr(o, k) is not None:
                xa = getattr(a, k) if fa is None else fa * getattr(a, k)
                getattr(o, k)[...] = xa + fb * getattr(b, k)
        if o.ground_sunlit_frac is not None:
            o.ground_sunlit_frac[...] = a.ground_sunlit_frac + b.ground_sunlit_frac
    return bc, out


def _compare(cfg, cp, sw, lw, c1=None, c2=None, profiles=True, seed=1, budget=0):
    """Summed run against the reference; per-layer entries of layers no in-range column owns keep the poison.
    Returns False when the plan does not take the staged route."""
    shapes = ((cfg.nsw, True, profiles), (cfg.nlw, False, profiles))
    factors = _factors(cfg, cp.ncol, seed)
    got = _summed(cfg, cp, sw, lw, c1, c2, shapes, factors, budget)
    if got is None:
        return False
    bc_ref, ref = _reference(cfg, cp, sw, lw, c1, c2, shapes, factors, budget)
    owned = _owned_layers(cp, c1 or 1, c2 or cp.ncol)
    lo, hi = (c1 or 1) - 1, c2 or cp.ncol
    n = 0
    for name, a, b, on in (("sw", ref[0], got[1][0], cfg.do_sw), ("lw", ref[1], got[1][1], cfg.do_lw)):
        if not on:
            continue
        for k in SPECTRAL_LAYER_FIELDS + SUNLIT_LAY_FIELDS:
            x, y = getattr(a, k), getattr(b, k)
            if x is None:
                continue
            assert np.array_equal(x[owned], y[owned]), (name, k, float(np.abs(x[owned] - y[owned]).max()))
            assert np.all(y[~owned] == POISON), (name, k)
            n += 1
        for k in PER_COLUMN + ("ground_sunlit_frac",):
            x, y = getattr(a, k), getattr(b, k)
            if x is not None:
                assert np.array_equal(x[lo:hi], y[lo:hi]), (name, k)
    for k in golden_io.BC_FIELDS:
        x, y = getattr(bc_ref, k), getattr(got[0], k)
        if x is not None and (cfg.do_sw if k.startswith("sw") else cfg.do_lw):
            assert np.array_equal(x[lo:hi], y[lo:hi]), k
    assert n > 0
    return True


def _cfg(streams=2, nsw=1, nlw=1, **kw):
    return config_type(nsw=nsw, nlw=nlw, n_vegetation_region_urban=2, n_vegetation_region_forest=2,
                       n_stream_sw_urban=streams, n_stream_lw_urban=streams, n_stream_sw_forest=streams,
                       n_stream_lw_forest=streams, **kw).consolidate()


@pytest.mark.parametrize("streams,nsw,nlw", [(1, 1, 1), (2, 1, 1), (4, 1, 1), (2, 2, 3)])
def test_summed_scatter_synthetic(streams, nsw, nlw):
    """9 layers: both the vector and the scalar branch of the one-value-per-layer scatter run; nsw = 2,
    nlw = 3 runs the tiled scatter.  A small budget forces several chunks."""
    cfg = _cfg(streams, nsw, nlw)
    cp, sw, lw = make_synthetic(cfg, 300, 9)
    assert _compare(cfg, cp, sw, lw)
    assert _compare(cfg, cp, sw, lw, budget=1)


def test_summed_scatter_mixed_tiles_and_sub_range():
    """Ragged layers, Flat, forest and urban tiles, night columns, several spectral intervals (the
    single-layer urban columns, which the staging does not cover, made Urban)."""
    cfg = mixed_config(2).consolidate()
    cp, sw, lw = make_mixed(cfg, ncol=200)
    rep = cp.i_representation
    assert not _compare(cfg, cp, sw, lw)  # SimpleUrban / InfiniteStreet present: not the staged route
    cp.i_representation = np.where((rep == ITileSimpleUrban) | (rep == ITileInfiniteStreet), ITileUrban, rep).astype(np.int32)
    assert _compare(cfg, cp, sw, lw)
    assert _compare(cfg, cp, sw, lw, 37, 151)


def test_summed_scatter_member_subsets():
    """Without flux profiles, and with urban or vegetation members absent: only the allocated members of
    the summed objects are paired and written."""
    for kw in (dict(), dict(do_urban=False), dict(do_vegetation=False)):
        cfg = _cfg(2, **kw)
        cp, sw, lw = make_synthetic(cfg, 120, 6)
        if not cfg.do_urban:
            cp.i_representation[:] = ITileForest
        if not cfg.do_vegetation:
            cp.i_representation[:] = ITileUrban
        assert _compare(cfg, cp, sw, lw, profiles=False)


def test_summed_scatter_degenerate_regions():
    cfg, cp, sw, lw = make_degenerate(2)
    assert _compare(cfg, cp, sw, lw)


@pytest.mark.parametrize("case", golden_io.list_cases())
def test_summed_scatter_golden(case):
    """Every golden fixture with seeded top-of-canopy fluxes; cases with single-layer urban columns or more
    than 4 streams do not take the staged route."""
    r, _ = golden_io.load_case(case, legendre_gauss_init=oracle_lib.legendre_gauss_init)
    cfg, cp = r.config, r.canopy_props
    staged = _compare(cfg, cp, r.sw_spectral_props if cfg.do_sw else None,
                      r.lw_spectral_props if cfg.do_lw else None, seed=len(case))
    simple = np.isin(cp.i_representation[:cp.ncol], (ITileSimpleUrban, ITileInfiniteStreet)).any()
    streams = max(cfg.n_stream_sw_urban, cfg.n_stream_lw_urban, cfg.n_stream_sw_forest, cfg.n_stream_lw_forest)
    assert staged == (not simple and streams <= 4)
