"""The summing scatter of ssb200_radsurf_fluxes_device_sp on the CPU: hostcheck_radsurf_summed_sp
(tests/hostcheck/hostcheck_summed_sp.cpp) stages float per-layer inputs and scatters the FP64 sums, rounded to
nearest, into float summed objects.  It must equal hostcheck_radsurf_summed on the same (float-valued) inputs
held as doubles, cast to float, for every per-layer member of the summed objects.
Some per-layer inputs are kept double in the single-precision run, as the device entry keeps read_input's
defaults, sigma T^4 and the default contact fraction in double buffers: one pass then stages float and double
arrays side by side, and those inputs keep values that are not floats."""
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
from spartacus_surface_b200 import _abi, boundary_conds_out_type
from spartacus_surface_b200.radsurf_canopy_flux import (COL_FIELDS, COL_DIR_FIELDS, SPECTRAL_LAYER_FIELDS,
                                                        SUNLIT_LAY_FIELDS)
from spartacus_surface_b200.radsurf_canopy_properties import (ITileForest, ITileUrban, ITileSimpleUrban,
                                                              ITileInfiniteStreet)
from spartacus_surface_b200.radsurf_interface import marshal
from spartacus_surface_b200.synthetic import make_synthetic
from test_hostcheck_fluxes import POISON, NOT_STAGED, _ptr, _ref, _factors, _flux, _owned_layers, _summed, _cfg

PER_COLUMN = COL_FIELDS + COL_DIR_FIELDS

SP_SRC = os.path.join(os.path.dirname(hostcheck_lib.SRC), "hostcheck_summed_sp.cpp")
SP_SO = os.path.join(os.path.dirname(hostcheck_lib.SO), "libhostcheck_summed_sp.so")
_sp_handle = None


def _sp_lib():
    """tests/_build/libhostcheck_summed_sp.so: the host check plus hostcheck_radsurf_summed_sp, built with the
    flags of libhostcheck.so (no FMA contraction)."""
    global _sp_handle
    if _sp_handle is None:
        deps = [SP_SRC, hostcheck_lib.SRC, os.path.join(os.path.dirname(SP_SRC), "asymtx_qr.hpp"),
                os.path.join(hostcheck_lib.ROOT, "include", "spartacus_b200.h")]
        deps += [os.path.join(hostcheck_lib.CSRC, f) for f in os.listdir(hostcheck_lib.CSRC) if f.endswith((".cuh", ".hpp"))]
        if not (os.path.exists(SP_SO) and all(os.path.getmtime(SP_SO) >= os.path.getmtime(d) for d in deps)):
            os.makedirs(os.path.dirname(SP_SO), exist_ok=True)
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off",
                                   "-Wno-maybe-uninitialized", "-o", SP_SO, SP_SRC])
        lib = C.CDLL(SP_SO)
        P = C.POINTER
        lib.hostcheck_radsurf_summed_sp.argtypes = (
            [P(_abi.Config), P(_abi.CanopyProperties), P(_abi.SwSpectralProperties), P(_abi.LwSpectralProperties),
             P(_abi.BoundaryCondsOut), C.c_int32, C.c_int32] + [P(_abi.CanopyFlux)] * 6
            + [P(C.c_double)] * 3 + [C.c_int64, C.c_int64])
        _sp_handle = lib
    return _sp_handle


def _double_members(struct):
    return [k for k, t in struct._fields_ if t is _abi._dp]


# the per-layer inputs in the order of the bits of hostcheck_radsurf_summed_sp's f64_mask
MEMBERS = ([("cp", k) for k in _double_members(_abi.CanopyProperties)]
           + [("sw", k) for k in _double_members(_abi.SwSpectralProperties)]
           + [("lw", k) for k in _double_members(_abi.LwSpectralProperties)])
# the members the device entry may hold in double buffers
DRIVER_DEFAULTS = {("cp", "veg_contact_fraction"), ("sw", "air_ext"), ("sw", "air_ssa"),
                   ("sw", "wall_specular_frac"), ("lw", "air_ext"), ("lw", "air_ssa"), ("lw", "clear_air_planck"),
                   ("lw", "veg_planck"), ("lw", "veg_air_planck"), ("lw", "roof_emission"), ("lw", "wall_emission")}


def _mask(kept):
    return sum(1 << i for i, m in enumerate(MEMBERS) if m in kept)


def _to_float_values(cp, sw, lw, kept):
    """Copies whose float64 members hold float values, except the per-layer members in `kept`."""
    out = {}
    for key, obj in (("cp", cp), ("sw", sw), ("lw", lw)):
        if obj is None:
            out[key] = None
            continue
        o = copy.copy(obj)
        for k, v in vars(obj).items():
            if isinstance(v, np.ndarray) and v.dtype == np.float64 and (key, k) not in kept:
                setattr(o, k, v.astype(np.float32).astype(np.float64))
        out[key] = o
    return out["cp"], out["sw"], out["lw"]


def _summed_sp(cfg, cp, sw, lw, c1, c2, shapes, factors, budget, mask):
    """hostcheck_radsurf_summed_sp on poisoned summed objects; per-layer members only."""
    top_sw, top_dir, top_lw = factors
    lib = _sp_lib()
    bc = boundary_conds_out_type().allocate(cp.ncol, cfg.nsw, cfg.nlw)
    out = [_flux(cfg, cp.ncol, cp.ntotlay, *s) for s in shapes]
    for o in out:
        o.fill(POISON)
    norm = []
    for o in out:
        for _ in range(2):
            n = copy.copy(o)
            for k in PER_COLUMN + ("ground_sunlit_frac",):
                if getattr(o, k) is not None:
                    setattr(n, k, np.zeros_like(getattr(o, k)))
            norm.append(n)
    s = marshal(cfg, cp, sw, lw, bc, *norm)
    fsw, flw = out[0].as_struct(), out[1].as_struct()
    rc = lib.hostcheck_radsurf_summed_sp(
        _ref(s["config"]), _ref(s["canopy"]), _ref(s["sw"]), _ref(s["lw"]), _ref(s["bc"]), int(c1 or 0),
        int(c2 or 0), _ref(s["sw_norm_dir"]), _ref(s["sw_norm_diff"]), _ref(s["lw_internal"]), _ref(s["lw_norm"]),
        C.byref(fsw), C.byref(flw), _ptr(top_sw), _ptr(top_dir), _ptr(top_lw), budget, mask)
    if rc == NOT_STAGED:
        return None
    assert rc == 0
    return bc, out


def _compare_sp(cfg, cp, sw, lw, c1=None, c2=None, profiles=True, seed=1, budget=0, kept=DRIVER_DEFAULTS):
    """Single-precision summed run against the double one, cast to float; layers no in-range column owns keep
    the poison.  Returns False when the plan does not take the staged route."""
    cp, sw, lw = _to_float_values(cp, sw, lw, kept)
    shapes = ((cfg.nsw, True, profiles), (cfg.nlw, False, profiles))
    factors = _factors(cfg, cp.ncol, seed)
    got = _summed_sp(cfg, cp, sw, lw, c1, c2, shapes, factors, budget, _mask(kept))
    if got is None:
        return False
    bc_ref, ref = _summed(cfg, cp, sw, lw, c1, c2, shapes, factors, budget)
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
            want = x[owned].astype(np.float32).astype(np.float64)
            assert np.array_equal(want, y[owned]), (name, k, float(np.abs(want - y[owned]).max()))
            assert np.all(y[~owned] == POISON), (name, k)
            n += 1
    for k in golden_io.BC_FIELDS:  # (per-column: double in both runs, as the device entry widens them)
        x, y = getattr(bc_ref, k), getattr(got[0], k)
        if x is not None and (cfg.do_sw if k.startswith("sw") else cfg.do_lw):
            assert np.array_equal(x[lo:hi], y[lo:hi]), k
    assert n > 0
    return True


@pytest.mark.parametrize("streams,nsw,nlw", [(1, 1, 1), (2, 1, 1), (4, 1, 1), (2, 2, 3)])
def test_summed_scatter_sp_synthetic(streams, nsw, nlw):
    """9 layers: both the float4 and the scalar branch of the one-value-per-layer scatter run; nsw = 2,
    nlw = 3 runs the tiled scatter.  Every input float, then the driver defaults kept double; a small budget
    forces several chunks."""
    cfg = _cfg(streams, nsw, nlw)
    cp, sw, lw = make_synthetic(cfg, 300, 9)
    assert _compare_sp(cfg, cp, sw, lw, kept=set())
    assert _compare_sp(cfg, cp, sw, lw)
    assert _compare_sp(cfg, cp, sw, lw, budget=1)


def test_summed_scatter_sp_mixed_tiles_and_sub_range():
    cfg = mixed_config(2).consolidate()
    cp, sw, lw = make_mixed(cfg, ncol=200)
    rep = cp.i_representation
    assert not _compare_sp(cfg, cp, sw, lw)  # SimpleUrban / InfiniteStreet present: not the staged route
    cp.i_representation = np.where((rep == ITileSimpleUrban) | (rep == ITileInfiniteStreet), ITileUrban, rep).astype(np.int32)
    assert _compare_sp(cfg, cp, sw, lw)
    assert _compare_sp(cfg, cp, sw, lw, 37, 151)


def test_summed_scatter_sp_member_subsets():
    for kw in (dict(), dict(do_urban=False), dict(do_vegetation=False)):
        cfg = _cfg(2, **kw)
        cp, sw, lw = make_synthetic(cfg, 120, 6)
        if not cfg.do_urban:
            cp.i_representation[:] = ITileForest
        if not cfg.do_vegetation:
            cp.i_representation[:] = ITileUrban
        assert _compare_sp(cfg, cp, sw, lw, profiles=False)


def test_summed_scatter_sp_degenerate_regions():
    cfg, cp, sw, lw = make_degenerate(2)
    assert _compare_sp(cfg, cp, sw, lw)


@pytest.mark.parametrize("case", golden_io.list_cases())
def test_summed_scatter_sp_golden(case):
    r, _ = golden_io.load_case(case, legendre_gauss_init=oracle_lib.legendre_gauss_init)
    cfg, cp = r.config, r.canopy_props
    staged = _compare_sp(cfg, cp, r.sw_spectral_props if cfg.do_sw else None,
                         r.lw_spectral_props if cfg.do_lw else None, seed=len(case))
    simple = np.isin(cp.i_representation[:cp.ncol], (ITileSimpleUrban, ITileInfiniteStreet)).any()
    streams = max(cfg.n_stream_sw_urban, cfg.n_stream_lw_urban, cfg.n_stream_sw_forest, cfg.n_stream_lw_forest)
    assert staged == (not simple and streams <= 4)
