"""GPU tests on the configuration matrix of tests/coverage_case.py: every register-resident kernel
shape the dispatcher can launch (pass x NREG 1-3 x NS 1-4 x URBAN) and the generic kernels at 5-8
streams, on inputs whose regions and boundary conditions cannot be confused with one another, held to
the oracle's _Float128 truth with the rule of tests/parity.py.  Also: the device-resident entry is
bit-equal to the host entry on every spec; the driver-sequence entries with distinct air, vegetation
and vegetation-air temperatures are bit-equal to sigma T^4 in numpy followed by radsurf, scale and sum;
the single-precision entries are bit-equal to the float64 result rounded to float32.  Every parity run
appends its numbers to the parity table through tests/test_gpu_parity.py's _record."""
import copy

import numpy as np
import pytest

import coverage_case as cc
import parity
from spartacus_surface_b200 import radsurf, canopy_flux_type, boundary_conds_out_type
from spartacus_surface_b200._lib import load
from spartacus_surface_b200.radsurf_canopy_flux import ALL_FIELDS
from spartacus_surface_b200.radsurf_interface import radsurf_fluxes, radsurf_fluxes_sp, radsurf_sp, to_single
from spartacus_surface_b200.radsurf_lw_spectral_properties import StefanBoltzmann
from test_gpu_fluxes_device import _dev, _tops
from test_gpu_fluxes_device_sp import _dev as _dev32, _single, _wide
from test_gpu_parity import _record

pytestmark = pytest.mark.gpu

NAMES = [s["name"] for s in cc.SPECS]


@pytest.fixture
def fast_kernels():
    """Sets the fast_kernels option for one test and restores the default (1) afterwards."""
    lib = load()
    assert lib.ssb200_device_count() > 0
    yield lambda value: lib.ssb200_set_option(b"fast_kernels", value)
    lib.ssb200_set_option(b"fast_kernels", 1)


@pytest.mark.parametrize("fast", [1, 0], ids=["register_resident", "generic"])
@pytest.mark.parametrize("name", NAMES)
def test_host_entry_vs_truth(name, fast, fast_kernels):
    """ssb200_radsurf on a spec of the matrix against the truth: REF_FACTOR for the product kernels,
    4 for the generic kernels (the reference's operation order compiled by nvcc)."""
    assert fast_kernels(fast) == 0
    got, status = cc.run(*cc.make_case(cc.BY_NAME[name]), radsurf)
    o = cc.oracle_runs(name)
    ref = o["fma"]
    assert status == 0
    assert not cc.poison_mismatches(got, ref), cc.poison_mismatches(got, ref)
    got, truth, ora, orb = (cc.unpoison(x, ref) for x in (got, o["quad"], o["fma"], o["nofma"]))
    ok, worst, lines = parity.check(got, truth, ora, orb, factor=parity.REF_FACTOR if fast else 4.0)
    row = dict(case=f"coverage_{name}", kernels="register-resident" if fast else "generic",
               **parity.summary(got, truth, ora, orb))
    _record(row)
    print(f"{name} fast={fast}: err_gpu = {row['err_gpu']:.3e}, err_ref_fp64 = {row['err_ref_fp64']:.3e}, "
          f"worst err/bound = {worst:.3e}")
    if not ok and not fast and row["err_ref_fp64"] > 1e-2:
        pytest.skip(f"reference FP64 arithmetic is off by {row['err_ref_fp64']:.2e} of the field maximum here")
    assert ok, "\n".join(lines)


@pytest.mark.parametrize("name", NAMES)
def test_device_entry_equals_host_entry(name):
    """ssb200_radsurf_device on torch CUDA tensors gives the bits of ssb200_radsurf, poison included."""
    import torch
    cfg, cp, sw, lw = cc.make_case(cc.BY_NAME[name])
    host, status = cc.run(cfg, cp, sw, lw, radsurf)
    assert status == 0
    bc = boundary_conds_out_type().allocate(cp.ncol, cfg.nsw, cfg.nlw)
    for k in cc.BC_FIELDS:
        getattr(bc, k)[...] = cc.POISON
    fl = [canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, n, use_direct=d)
          for n, d in ((cfg.nsw, True), (cfg.nsw, True), (cfg.nlw, False), (cfg.nlw, False))]
    for f in fl:
        f.fill(cc.POISON)
    dbc, dfl = _dev(bc), [_dev(f) for f in fl]
    assert radsurf(cfg, _dev(cp), _dev(sw), _dev(lw), dbc, None, None, *dfl) == 0
    torch.cuda.synchronize()
    for n, f in zip(cc.FLUX_NAMES, dfl):
        for k, v in host[n].items():
            x = getattr(f, k).cpu().numpy()
            assert np.array_equal(x, v), (n, k, float(np.abs(x - v).max()))
    for k, v in host["bc"].items():
        assert np.array_equal(getattr(dbc, k).cpu().numpy(), v), ("bc", k)


# ---- driver sequence ---------------------------------------------------------------------------

def _driver_case(name, ncol=cc.NCOL):
    """A spec's case with one longwave interval (the simple spectrum of the driver) and distinct
    temperatures: vegetation warmer and vegetation air cooler than clear air, by amounts that vary."""
    cfg, cp, sw, lw = cc.make_case(cc.BY_NAME[name], ncol, nsw=2, nlw=1)
    rng = np.random.default_rng(99)
    t_air = rng.uniform(275.0, 295.0, size=cp.ntotlay)
    temps = dict(ground_temperature=rng.uniform(270.0, 300.0, size=cp.ncol),
                 roof_temperature=rng.uniform(270.0, 310.0, size=cp.ntotlay),
                 wall_temperature=rng.uniform(270.0, 305.0, size=cp.ntotlay),
                 clear_air_temperature=t_air,
                 veg_temperature=t_air + rng.uniform(2.0, 6.0, size=cp.ntotlay),
                 veg_air_temperature=t_air - rng.uniform(1.0, 4.0, size=cp.ntotlay))
    return cfg, cp, sw, lw, dict(_tops(cfg, cp.ncol, 17), **temps)


def _step_by_step(cfg, cp, sw, lw, drv):
    """sigma T^4 in numpy, then radsurf, scale and sum: what the reference driver holds in memory."""
    p4 = lambda t: (t * t) * (t * t)
    lw = copy.copy(lw)
    lw.ground_emission = (StefanBoltzmann * lw.ground_emissivity[:, 0] * p4(drv["ground_temperature"]))[:, None].copy()
    lw.roof_emission = (StefanBoltzmann * lw.roof_emissivity[:, 0] * p4(drv["roof_temperature"]))[:, None].copy()
    lw.wall_emission = (StefanBoltzmann * lw.wall_emissivity[:, 0] * p4(drv["wall_temperature"]))[:, None].copy()
    for k, t in (("clear_air_planck", "clear_air_temperature"), ("veg_planck", "veg_temperature"),
                 ("veg_air_planck", "veg_air_temperature")):
        setattr(lw, k, (StefanBoltzmann * p4(drv[t]))[:, None].copy())
    assert np.all(lw.veg_planck != lw.clear_air_planck) and np.all(lw.veg_air_planck != lw.clear_air_planck)
    bc = boundary_conds_out_type().allocate(cp.ncol, cfg.nsw, cfg.nlw)
    fl = [canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, n, use_direct=d)
          for n, d in ((cfg.nsw, True), (cfg.nsw, True), (cfg.nlw, False), (cfg.nlw, False))]
    assert radsurf(cfg, cp, sw, lw, bc, None, None, *fl) == 0
    top_sw, top_dir = drv["top_flux_dn_sw"], drv["top_flux_dn_direct_sw"]
    fl[0].scale(cp.nlay, top_dir)
    fl[1].scale(cp.nlay, top_sw - top_dir)
    fl[3].scale(cp.nlay, drv["top_flux_dn_lw"])
    sw_ref = canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, cfg.nsw, use_direct=True)
    lw_ref = canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, cfg.nlw, use_direct=False)
    sw_ref.sum(fl[0], fl[1])
    lw_ref.sum(fl[2], fl[3])
    return bc, sw_ref, lw_ref


def _driver_outputs(cfg, cp):
    """(bc_out, sw_flux, lw_flux) of the driver sequence, zeroed."""
    return (boundary_conds_out_type().allocate(cp.ncol, cfg.nsw, cfg.nlw),
            canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, cfg.nsw, use_direct=True),
            canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, cfg.nlw, use_direct=False))


def _without_emission(lw):
    lw = copy.copy(lw)
    for k in ("ground_emission", "roof_emission", "wall_emission", "clear_air_planck", "veg_planck", "veg_air_planck"):
        setattr(lw, k, None)
    return lw


def _assert_same(got, want, tag):
    """got, want: (bc_out, sw_flux, lw_flux), host arrays or CUDA tensors in `got`."""
    host = lambda a: a.cpu().numpy() if hasattr(a, "cpu") else a
    for name, a, b in (("sw", got[1], want[1]), ("lw", got[2], want[2])):
        for k in ALL_FIELDS:
            w = getattr(b, k)
            if w is not None:
                g = host(getattr(a, k))
                assert np.array_equal(g, w), (tag, name, k, float(np.abs(g - w).max()))
    for k in cc.BC_FIELDS:
        assert np.array_equal(host(getattr(got[0], k)), getattr(want[0], k)), (tag, k)


@pytest.mark.parametrize("name", [cc.DEFAULT, "r3_s3_u31"])
def test_driver_sequence_with_distinct_temperatures(name):
    """ssb200_radsurf_fluxes (host arrays) and ssb200_radsurf_fluxes_device (CUDA tensors) with the
    emission and Planck members None and distinct air / vegetation / vegetation-air temperatures:
    bit-equal to sigma T^4 in numpy followed by radsurf, scale and sum.  (The two entries share the
    staging of the driver inputs, so comparing them with each other alone would not catch a wrong
    temperature behind a Planck member.)"""
    import torch
    cfg, cp, sw, lw, drv = _driver_case(name)
    want = _step_by_step(cfg, cp, sw, lw, drv)
    lw0 = _without_emission(lw)
    outputs = lambda: _driver_outputs(cfg, cp)
    bc, swf, lwf = outputs()
    assert radsurf_fluxes(cfg, cp, sw, lw0, bc, None, None, swf, lwf, **drv) == 0
    _assert_same((bc, swf, lwf), want, "host")
    dbc, dswf, dlwf = (_dev(o) for o in outputs())
    assert radsurf_fluxes(cfg, _dev(cp), _dev(sw), _dev(lw0), dbc, None, None, dswf, dlwf,
                          **{k: _dev(v) for k, v in drv.items()}) == 0
    torch.cuda.synchronize()
    _assert_same((dbc, dswf, dlwf), want, "device")


# ---- single precision --------------------------------------------------------------------------

def test_single_precision_entries_default_spec():
    """radsurf_sp and radsurf_fluxes_sp on float32 CUDA tensors (device entries) of the default spec:
    bit-equal to the float64 entries on the widened inputs, rounded to float32."""
    import torch
    cfg, cp, sw, lw = cc.make_case(cc.BY_NAME[cc.DEFAULT])
    cp, sw, lw = _single(cp), _single(sw), _single(lw)
    want, status = cc.run(cfg, _wide(cp), _wide(sw), _wide(lw), radsurf)
    assert status == 0
    bc = to_single(boundary_conds_out_type().allocate(cp.ncol, cfg.nsw, cfg.nlw))
    fl = [to_single(canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, n, use_direct=d))
          for n, d in ((cfg.nsw, True), (cfg.nsw, True), (cfg.nlw, False), (cfg.nlw, False))]
    for o in [bc] + fl:
        for v in vars(o).values():
            if isinstance(v, np.ndarray) and v.dtype.kind == "f":
                v[...] = cc.POISON
    dbc, dfl = _dev32(bc), [_dev32(f) for f in fl]
    assert radsurf_sp(cfg, _dev32(cp), _dev32(sw), _dev32(lw), dbc, None, None, *dfl) == 0
    torch.cuda.synchronize()
    for n, f in zip(cc.FLUX_NAMES, dfl):
        for k, v in want[n].items():
            x = getattr(f, k).cpu().numpy()
            assert x.dtype == np.float32 and np.array_equal(x, v.astype(np.float32)), (n, k)
    for k, v in want["bc"].items():
        assert np.array_equal(getattr(dbc, k).cpu().numpy(), v.astype(np.float32)), ("bc", k)

    # the driver sequence: distinct temperatures, emission and Planck members None
    cfg, cp, sw, lw, drv = _driver_case(cc.DEFAULT)
    cp, sw, lw0 = _single(cp), _single(sw), _single(_without_emission(lw))
    drv = {k: _single(v) for k, v in drv.items()}
    outputs = lambda: _driver_outputs(cfg, cp)
    ref = outputs()
    assert radsurf_fluxes(cfg, _wide(cp), _wide(sw), _wide(lw0), ref[0], None, None, ref[1], ref[2],
                          **{k: _wide(v) for k, v in drv.items()}) == 0
    got = [_dev32(to_single(o)) for o in outputs()]
    assert radsurf_fluxes_sp(cfg, _dev32(cp), _dev32(sw), _dev32(lw0), got[0], None, None, got[1], got[2],
                             **{k: _dev32(v) for k, v in drv.items()}) == 0
    torch.cuda.synchronize()
    n = 0
    for a, b in zip(got, ref):
        for k, v in vars(b).items():
            if isinstance(v, np.ndarray) and v.dtype == np.float64:
                x = getattr(a, k).cpu().numpy()
                assert x.dtype == np.float32 and np.array_equal(x, v.astype(np.float32)), k
                n += 1
    assert n > 0
