"""GPU tests of the single-precision forms of the driver-sequence and device-resident entries
(ssb200_radsurf_fluxes_sp, ssb200_radsurf_device_sp).  Both take float32 arrays, solve in FP64 and
round every output to nearest float32, so each must be bit-equal to its double-precision twin called
on the widened inputs, followed by a cast: every comparison below is np.array_equal against
double_output.astype(float32).  Outputs start from a finite poison value, so entries the solve leaves
untouched and columns outside istartcol..iendcol are checked too."""
import copy
import ctypes as C

import numpy as np
import pytest

import golden_io
from degenerate_case import make_degenerate
from mixed_case import mixed_config, make_mixed
from spartacus_surface_b200 import (radsurf, RadsurfError, config_type, canopy_flux_type,
                                    boundary_conds_out_type)
from spartacus_surface_b200._lib import load
from spartacus_surface_b200.radsurf_canopy_properties import ITileSimpleUrban, ITileInfiniteStreet, ITileUrban
from spartacus_surface_b200.radsurf_interface import (call_radsurf, f32_ptr, marshal, radsurf_fluxes,
                                                      radsurf_fluxes_sp, radsurf_sp, to_single)
from spartacus_surface_b200.synthetic import make_synthetic

pytestmark = pytest.mark.gpu

POISON = 7.0
NLAY = 9  # istartlay - 1 + l0 is not always a multiple of 4: vector and scalar float staging both run

# library defaults (include/spartacus_b200.h, ssb200_set_option)
DEFAULTS = {b"stage_layers": 1, b"fast_kernels": 1, b"sort_columns": 1, b"scratch_budget_bytes": 0}


@pytest.fixture
def options():
    """Sets library options for one test and restores the defaults afterwards."""
    lib = load()
    touched = []

    def set_option(name, value):
        touched.append(name)
        assert lib.ssb200_set_option(name, value) == 0

    yield set_option
    for name in touched:
        lib.ssb200_set_option(name, DEFAULTS[name])


def _cfg(streams=2, nsw=1, nlw=1):
    return config_type(nsw=nsw, nlw=nlw, n_vegetation_region_urban=2, n_vegetation_region_forest=2,
                       n_stream_sw_urban=streams, n_stream_lw_urban=streams, n_stream_sw_forest=streams,
                       n_stream_lw_forest=streams).consolidate()


def _wide(obj):
    """Copy with every float32 numpy member widened to float64 (the double twin's inputs)."""
    if obj is None:
        return None
    out = copy.copy(obj)
    for k, v in vars(obj).items():
        if isinstance(v, np.ndarray) and v.dtype == np.float32:
            setattr(out, k, np.ascontiguousarray(v.astype(np.float64)))
    return out


def _dev(obj, dtype):
    """Copy with every real numpy member as a torch CUDA tensor of `dtype`."""
    import torch
    if obj is None:
        return None
    out = copy.copy(obj)
    for k, v in vars(obj).items():
        if isinstance(v, np.ndarray) and v.dtype.kind == "f":
            setattr(out, k, torch.from_numpy(np.ascontiguousarray(v.astype(dtype))).cuda())
    return out


def _host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else a


def _poison(objs):
    for o in objs:
        for v in vars(o).values() if o is not None else ():
            if isinstance(v, np.ndarray) and v.dtype.kind == "f":
                v[...] = POISON


def _poisoned(cfg, ncol, ntot):
    bc = boundary_conds_out_type().allocate(ncol, cfg.nsw, cfg.nlw)
    fl = [canopy_flux_type().allocate(cfg, ncol, ntot, n, use_direct=d)
          for n, d in ((cfg.nsw, True), (cfg.nsw, True), (cfg.nlw, False), (cfg.nlw, False))]
    _poison([bc] + fl)
    return bc, fl


def _assert_cast_equal(objs32, objs64):
    """Every float32 member equals the double twin's member cast to float32, bit for bit."""
    n = 0
    for a, b in zip(objs32, objs64):
        if a is None:
            continue
        for k, v in vars(a).items():
            if v is None or isinstance(v, (int, float)) or _host(v).dtype != np.float32:
                continue
            x, y = _host(v), _host(getattr(b, k)).astype(np.float32)
            assert np.array_equal(x, y), (k, float(np.abs(x.astype(np.float64) - y).max()))
            n += 1
    return n


def _assert_poison_outside(objs, cp, c1, c2):
    """Rows of columns outside c1..c2 (1-based) and of their packed layers still hold the poison."""
    lo_l = int(cp.istartlay[c1 - 1]) - 1
    hi_l = int(cp.istartlay[c2 - 1]) - 1 + int(cp.nlay[c2 - 1])
    n = 0
    for o in objs:
        for k, v in vars(o).items():
            if v is None or isinstance(v, (int, float)):
                continue
            x = _host(v)
            lo, hi = (c1 - 1, c2) if x.shape[0] == cp.ncol else (lo_l, hi_l)
            assert np.all(x[:lo] == POISON) and np.all(x[hi:] == POISON), k
            n += 1
    assert n > 0


def _device_pair(cfg, cp, sw, lw, c1=None, c2=None, outputs=None):
    """radsurf_sp on float32 CUDA tensors (ssb200_radsurf_device_sp) and radsurf on the widened float64
    tensors (ssb200_radsurf_device); returns the float32 output objects after checking them."""
    import torch
    ins32 = [to_single(o) if o is not None else None for o in (cp, sw, lw)]
    bc, fl = outputs if outputs is not None else _poisoned(cfg, cp.ncol, cp.ntotlay)
    out64 = [_dev(o, np.float64) for o in [bc] + fl]
    out32 = [_dev(o, np.float32) for o in [bc] + fl]
    assert radsurf(cfg, *[_dev(o, np.float64) for o in ins32], out64[0], c1, c2, *out64[1:]) == 0
    assert radsurf_sp(cfg, *[_dev(o, np.float32) for o in ins32], out32[0], c1, c2, *out32[1:]) == 0
    torch.cuda.synchronize()
    assert _assert_cast_equal(out32, out64) > 0
    return [o for o in out32 if o is not None]


def _fluxes_pair(cfg, cp, sw, lw, c1, c2, drv):
    """radsurf_fluxes_sp on float32 host arrays against radsurf_fluxes on the widened inputs."""
    cp32, sw32, lw32 = to_single(cp), to_single(sw), to_single(lw)
    drv32 = {k: np.ascontiguousarray(v.astype(np.float32)) for k, v in drv.items()}
    res = {}
    for single in (True, False):
        bc, fl = _poisoned(cfg, cp.ncol, cp.ntotlay)
        sw_flux, lw_flux = fl[0], fl[2]
        if single:
            bc, sw_flux, lw_flux = to_single(bc), to_single(sw_flux), to_single(lw_flux)
            rc = radsurf_fluxes_sp(cfg, cp32, sw32, lw32, bc, c1, c2, sw_flux, lw_flux, **drv32)
        else:
            rc = radsurf_fluxes(cfg, _wide(cp32), _wide(sw32), _wide(lw32), bc, c1, c2, sw_flux, lw_flux,
                                **{k: v.astype(np.float64) for k, v in drv32.items()})
        assert rc == 0
        res[single] = [bc, sw_flux, lw_flux]
    assert _assert_cast_equal(res[True], res[False]) > 10
    return res[True]


def _no_simple_urban(cp):
    """The mixed case with its SimpleUrban / InfiniteStreet columns made single-layer Urban columns:
    every per-layer read then goes through the staging."""
    out = copy.copy(cp)
    rep = cp.i_representation
    out.i_representation = np.where((rep == ITileSimpleUrban) | (rep == ITileInfiniteStreet), ITileUrban,
                                    rep).astype(np.int32)
    return out


# ---------------------------------------------------------------------------------------------------
# ssb200_radsurf_fluxes_sp
# ---------------------------------------------------------------------------------------------------
def test_fluxes_sp_synthetic_defaults_and_temperatures():
    """70,000 columns x 4 layers (several pipeline blocks); the members read_input would default and the
    emission / Planck members are NULL, the temperatures are given (one air temperature for three)."""
    cfg = _cfg()
    ncol = 70000
    cp, sw, lw = make_synthetic(cfg, ncol, 4)
    cp.veg_contact_fraction = None
    sw.air_ext = sw.air_ssa = sw.wall_specular_frac = sw.roof_albedo_dir = None
    lw.air_ext = lw.air_ssa = None
    for k in ("ground_emission", "roof_emission", "wall_emission", "clear_air_planck", "veg_planck", "veg_air_planck"):
        setattr(lw, k, None)
    rng = np.random.default_rng(11)
    top_sw = rng.uniform(200.0, 900.0, size=(ncol, 1))
    t_air = rng.uniform(270.0, 300.0, size=cp.ntotlay).astype(np.float32)
    drv = dict(top_flux_dn_sw=top_sw, top_flux_dn_direct_sw=top_sw * rng.uniform(0.2, 0.9, size=(ncol, 1)),
               top_flux_dn_lw=rng.uniform(250.0, 400.0, size=(ncol, 1)),
               ground_temperature=rng.uniform(270.0, 300.0, size=ncol),
               roof_temperature=rng.uniform(270.0, 300.0, size=cp.ntotlay),
               wall_temperature=rng.uniform(270.0, 300.0, size=cp.ntotlay))
    drv = {k: v.astype(np.float32) for k, v in drv.items()}
    drv32 = dict(drv, clear_air_temperature=t_air, veg_temperature=t_air, veg_air_temperature=t_air)
    _fluxes_pair(cfg, cp, sw, lw, None, None, drv32)


def test_fluxes_sp_mixed_tiles_sub_range():
    """Ragged layers, night columns, nsw = 2 and nlw = 3 with explicit emission members; a column
    sub-range leaves the poison of every other column and layer in place."""
    cfg = mixed_config(2).consolidate()
    cp, sw, lw = make_mixed(cfg, ncol=400)
    rng = np.random.default_rng(5)
    top_sw = rng.uniform(200.0, 900.0, size=(cp.ncol, cfg.nsw))
    drv = dict(top_flux_dn_sw=top_sw, top_flux_dn_direct_sw=top_sw * 0.6,
               top_flux_dn_lw=rng.uniform(250.0, 400.0, size=(cp.ncol, cfg.nlw)))
    for c1, c2 in ((None, None), (37, 311)):
        out = _fluxes_pair(cfg, cp, sw, lw, c1, c2, drv)
        if c1 is not None:
            _assert_poison_outside(out, cp, c1, c2)


# ---------------------------------------------------------------------------------------------------
# ssb200_radsurf_device_sp
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("streams,nsw,nlw", [(1, 1, 1), (2, 1, 1), (4, 1, 1), (8, 1, 1), (2, 2, 3)])
def test_device_sp_synthetic(streams, nsw, nlw):
    """1, 2 and 4 streams take the staged route, 8 streams (generic kernels) the fallback; nsw = 2,
    nlw = 3 runs the tiled gather / scatter with a float caller side."""
    cfg = _cfg(streams, nsw, nlw)
    cp, sw, lw = make_synthetic(cfg, 3000, NLAY)
    _device_pair(cfg, cp, sw, lw)


@pytest.mark.parametrize("variant", ["mixed", "mixed_staged"])
def test_device_sp_mixed_tiles(variant):
    """The mixed-tile case has SimpleUrban / InfiniteStreet columns (fallback route); without them it
    takes the staged route with ragged layers, night columns and several spectral intervals."""
    cfg = mixed_config(2).consolidate()
    cp, sw, lw = make_mixed(cfg, ncol=400)
    if variant == "mixed_staged":
        cp = _no_simple_urban(cp)
    _device_pair(cfg, cp, sw, lw)
    out = _device_pair(cfg, cp, sw, lw, 37, 311)
    _assert_poison_outside(out, cp, 37, 311)


@pytest.mark.parametrize("streams", [2, 4])
def test_device_sp_degenerate_regions(streams):
    cfg, cp, sw, lw = make_degenerate(streams)
    _device_pair(cfg, cp, sw, lw)
    out = _device_pair(cfg, cp, sw, lw, 13, 70)
    _assert_poison_outside(out, cp, 13, 70)


@pytest.mark.parametrize("case", golden_io.list_cases())
def test_device_sp_golden(case):
    r, _ = golden_io.load_case(case, legendre_gauss_init=load().ssb200_legendre_gauss_init)
    cfg = r.config
    outs = [r.bc_out, r.sw_norm_dir, r.sw_norm_diff, r.lw_internal, r.lw_norm]
    _poison(outs)
    _device_pair(cfg, r.canopy_props, r.sw_spectral_props if cfg.do_sw else None,
                 r.lw_spectral_props if cfg.do_lw else None, outputs=(outs[0], outs[1:]))


@pytest.mark.parametrize("name,value", [(b"stage_layers", 0), (b"fast_kernels", 0), (b"sort_columns", 0),
                                        (b"scratch_budget_bytes", 4 << 20)])
def test_device_sp_under_options(options, name, value):
    """Each option changes the route or the chunking of both entries alike: still bit-equal."""
    options(name, value)
    cfg = _cfg(2)
    cp, sw, lw = make_synthetic(cfg, 3000, NLAY)
    _device_pair(cfg, cp, sw, lw)
    cfgm = mixed_config(2).consolidate()
    cpm, swm, lwm = make_mixed(cfgm, ncol=400)
    _device_pair(cfgm, _no_simple_urban(cpm), swm, lwm)


def test_device_sp_status_and_stream_ordering():
    """status_out is written on the call's stream; a device_sp call on one torch stream followed by a
    radsurf_device call on another (shared context) gives the results of the same calls made serially."""
    import torch
    lib = load()
    cfg = _cfg(2)
    cpa, swa, lwa = (to_single(o) for o in make_synthetic(cfg, 20_000, 16))
    cpb, swb, lwb = make_synthetic(cfg, 20_000, 16, col_offset=50_000)
    a_in = [_dev(o, np.float32) for o in (cpa, swa, lwa)]
    b_in = [_dev(o, np.float64) for o in (cpb, swb, lwb)]

    def outs(dtype, cp):
        bc, fl = _poisoned(cfg, cp.ncol, cp.ntotlay)
        return [_dev(o, dtype) for o in [bc] + fl]

    serial_a, serial_b = outs(np.float32, cpa), outs(np.float64, cpb)
    conc_a, conc_b = outs(np.float32, cpa), outs(np.float64, cpb)
    torch.cuda.synchronize()
    assert radsurf_sp(cfg, *a_in, serial_a[0], None, None, *serial_a[1:]) == 0
    torch.cuda.synchronize()
    assert radsurf(cfg, *b_in, serial_b[0], None, None, *serial_b[1:]) == 0
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    status = torch.full((1,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    structs = marshal(cfg, *a_in, conc_a[0], *conc_a[1:], ptr=f32_ptr(True, "test"))
    for _ in range(3):  # back to back, alternating streams, no host synchronisation in between
        with torch.cuda.stream(s1):
            status.fill_(-1)
        rc = call_radsurf(lib.ssb200_radsurf_device_sp, structs, None, None,
                          extra=(C.c_void_p(s1.cuda_stream), C.cast(status.data_ptr(), C.POINTER(C.c_int32))))
        assert rc == 0
        assert radsurf(cfg, *b_in, conc_b[0], None, None, *conc_b[1:], stream=s2.cuda_stream) == 0
    s1.synchronize()
    assert int(status.item()) == 0
    torch.cuda.synchronize()
    assert _assert_cast_equal(conc_a, serial_a) > 0  # (float32 against float32: plain equality)
    for a, b in zip(conc_b, serial_b):
        for k, v in vars(a).items():
            if hasattr(v, "cpu"):
                assert torch.equal(v, getattr(b, k)), k
    lib.ssb200_release()


# ---------------------------------------------------------------------------------------------------
# wrapper argument checks
# ---------------------------------------------------------------------------------------------------
def test_sp_wrappers_refuse_wrong_dtypes_and_mixed_members():
    import torch
    cfg = _cfg(2)
    cp, sw, lw = make_synthetic(cfg, 64, 4)
    cp32, sw32, lw32 = to_single(cp), to_single(sw), to_single(lw)
    bc, fl = _poisoned(cfg, cp.ncol, cp.ntotlay)
    bc32, fl32 = to_single(bc), [to_single(f) for f in fl]
    # a float64 member, on the host and on the device
    bad = copy.copy(sw32)
    bad.air_ext = sw.air_ext
    with pytest.raises(RadsurfError):
        radsurf_sp(cfg, cp32, bad, lw32, bc32, None, None, *fl32)
    dev32 = [_dev(o, np.float32) for o in (cp32, sw32, lw32)]
    dout = [_dev(o, np.float32) for o in [bc32] + fl32]
    bad_dev = copy.copy(dev32[1])
    bad_dev.air_ext = bad_dev.air_ext.double()
    with pytest.raises(RadsurfError):
        radsurf_sp(cfg, dev32[0], bad_dev, dev32[2], dout[0], None, None, *dout[1:])
    # numpy and torch members in one call
    with pytest.raises(RadsurfError):
        radsurf_sp(cfg, dev32[0], sw32, dev32[2], dout[0], None, None, *dout[1:])
    # radsurf_fluxes_sp: float64 member, top flux, temperature; a torch member
    top = np.full((cp.ncol, 1), 500.0, dtype=np.float32)
    t = np.full(cp.ntotlay, 290.0, dtype=np.float32)
    good = dict(top_flux_dn_sw=top, top_flux_dn_direct_sw=top, top_flux_dn_lw=top)
    for kw, obj in ((good, bad), (dict(good, top_flux_dn_lw=top.astype(np.float64)), sw32),
                    (dict(good, roof_temperature=t.astype(np.float64)), sw32), (good, dev32[1])):
        with pytest.raises(RadsurfError):
            radsurf_fluxes_sp(cfg, cp32, obj, lw32, bc32, None, None, fl32[0], fl32[2], **kw)
    # the double-precision entries still refuse float32 tensors
    with pytest.raises((AssertionError, RadsurfError)):
        radsurf(cfg, *dev32, dout[0], None, None, *dout[1:])
    torch.cuda.synchronize()
