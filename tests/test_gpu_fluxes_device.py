"""GPU tests of ssb200_radsurf_fluxes_device: the reference driver's calc_simple_spectrum_lw + radsurf + scale
+ sum on device arrays.  Every output must be bit-equal to ssb200_radsurf_fluxes (host arrays) on the same
inputs: each comparison is np.array_equal over whole arrays.  Outputs start from a finite poison value, so
columns outside istartcol..iendcol and layers no selected column owns are checked too.  Both routes run:
the staged route (summing scatter, register-resident kernels of 1-4 streams) and the fallback route
(generic kernels, stage_layers = 0, single-layer urban columns)."""
import copy
import ctypes as C

import numpy as np
import pytest

import golden_io
from degenerate_case import make_degenerate
from mixed_case import mixed_config, make_mixed
from spartacus_surface_b200 import (RadsurfError, config_type, canopy_flux_type, boundary_conds_out_type, radsurf)
from spartacus_surface_b200 import _abi
from spartacus_surface_b200._lib import load
from spartacus_surface_b200.radsurf_canopy_flux import ALL_FIELDS
from spartacus_surface_b200.radsurf_canopy_properties import ITileForest, ITileUrban, ITileSimpleUrban, ITileInfiniteStreet
from spartacus_surface_b200.radsurf_interface import f64_cuda_ptr, marshal, radsurf_fluxes
from spartacus_surface_b200.synthetic import make_synthetic

pytestmark = pytest.mark.gpu

POISON = 7.0
NLAY = 9  # istartlay - 1 + l0 is not always a multiple of 4: vector and scalar branch of k_stage1 both run
SSB200_ERR_ARG = -1
DRV_KEYS = ("top_flux_dn_sw", "top_flux_dn_direct_sw", "top_flux_dn_lw", "ground_temperature", "roof_temperature",
            "wall_temperature", "clear_air_temperature", "veg_temperature", "veg_air_temperature")

# library defaults (include/spartacus_b200.h, ssb200_set_option)
DEFAULTS = {b"stage_layers": 1, b"fast_kernels": 1, b"sort_columns": 1, b"concurrent_passes": 1,
            b"scratch_budget_bytes": 0}


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


def _cfg(streams=2, nsw=1, nlw=1, **kw):
    return config_type(nsw=nsw, nlw=nlw, n_vegetation_region_urban=2, n_vegetation_region_forest=2,
                       n_stream_sw_urban=streams, n_stream_lw_urban=streams, n_stream_sw_forest=streams,
                       n_stream_lw_forest=streams, **kw).consolidate()


def _dev(obj):
    """Copy with every float64 numpy member as a torch CUDA tensor."""
    import torch
    if obj is None:
        return None
    if isinstance(obj, np.ndarray):
        return torch.from_numpy(np.ascontiguousarray(obj)).cuda()
    out = copy.copy(obj)
    for k, v in vars(obj).items():
        if isinstance(v, np.ndarray) and v.dtype == np.float64:
            setattr(out, k, torch.from_numpy(np.ascontiguousarray(v)).cuda())
    return out


def _host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else a


def _outputs(cfg, ncol, ntot, profiles=True):
    bc = boundary_conds_out_type().allocate(ncol, cfg.nsw, cfg.nlw)
    sw_flux = canopy_flux_type().allocate(cfg, ncol, ntot, cfg.nsw, use_direct=True, do_save_flux_profile=profiles)
    lw_flux = canopy_flux_type().allocate(cfg, ncol, ntot, cfg.nlw, use_direct=False, do_save_flux_profile=profiles)
    for o in (sw_flux, lw_flux):
        o.fill(POISON)
    for v in vars(bc).values():
        if isinstance(v, np.ndarray):
            v[...] = POISON
    return [bc, sw_flux, lw_flux]


def _tops(cfg, ncol, seed):
    rng = np.random.default_rng(seed)
    top_sw = rng.uniform(200.0, 900.0, size=(ncol, cfg.nsw))
    return dict(top_flux_dn_sw=top_sw, top_flux_dn_direct_sw=np.ascontiguousarray(top_sw * rng.uniform(0.2, 0.9, size=(ncol, cfg.nsw))),
                top_flux_dn_lw=rng.uniform(250.0, 400.0, size=(ncol, cfg.nlw)))


def _defaulted(cfg, ncol, nlay, seed=3):
    """Synthetic canopy with every member read_input would default and every emission / Planck member
    None, and the temperatures and top-of-canopy fluxes of the driver."""
    cp, sw, lw, temps = make_synthetic(cfg, ncol, nlay, with_temperatures=True)
    cp.veg_contact_fraction = None
    sw.air_ext = sw.air_ssa = sw.wall_specular_frac = sw.roof_albedo_dir = None
    lw.air_ext = lw.air_ssa = None
    for k in ("ground_emission", "roof_emission", "wall_emission", "clear_air_planck", "veg_planck", "veg_air_planck"):
        setattr(lw, k, None)
    return cp, sw, lw, dict(_tops(cfg, ncol, seed), **temps)


def _assert_equal(got, ref):
    n = 0
    for a, b in zip(got, ref):
        for k, v in vars(b).items():
            if not isinstance(v, np.ndarray) or v.dtype != np.float64:
                continue
            x = _host(getattr(a, k))
            assert np.array_equal(x, v), (k, float(np.abs(x - v).max()))
            n += 1
    assert n > 0
    return n


def _pair(cfg, cp, sw, lw, drv, c1=None, c2=None, profiles=True):
    """radsurf_fluxes on device tensors against radsurf_fluxes on the same host arrays; returns the device
    outputs copied to the host."""
    import torch
    ref = _outputs(cfg, cp.ncol, cp.ntotlay, profiles)
    assert radsurf_fluxes(cfg, cp, sw, lw, ref[0], c1, c2, ref[1], ref[2], **drv) == 0
    got = [_dev(o) for o in _outputs(cfg, cp.ncol, cp.ntotlay, profiles)]
    assert radsurf_fluxes(cfg, _dev(cp), _dev(sw), _dev(lw), got[0], c1, c2, got[1], got[2],
                          **{k: _dev(v) for k, v in drv.items()}) == 0
    torch.cuda.synchronize()
    _assert_equal(got, ref)
    return got


def _assert_poison_outside(objs, cp, c1, c2):
    """Rows of columns outside c1..c2 (1-based) and of their packed layers still hold the poison."""
    lo_l = int(cp.istartlay[c1 - 1]) - 1
    hi_l = int(cp.istartlay[c2 - 1]) - 1 + int(cp.nlay[c2 - 1])
    for o in objs:
        for k, v in vars(o).items():
            if not hasattr(v, "cpu"):
                continue
            x = _host(v)
            lo, hi = (c1 - 1, c2) if x.shape[0] == cp.ncol else (lo_l, hi_l)
            assert np.all(x[:lo] == POISON) and np.all(x[hi:] == POISON), k


def _no_simple_urban(cp):
    out = copy.copy(cp)
    rep = cp.i_representation
    out.i_representation = np.where((rep == ITileSimpleUrban) | (rep == ITileInfiniteStreet), ITileUrban,
                                    rep).astype(np.int32)
    return out


# ---------------------------------------------------------------------------------------------------
# workloads and routes
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("streams,nsw,nlw", [(1, 1, 1), (2, 1, 1), (4, 1, 1), (8, 1, 1), (2, 2, 3)])
def test_synthetic(streams, nsw, nlw):
    """1, 2 and 4 streams take the staged route (k_stage1 summing scatter), 8 streams the fallback;
    nsw = 2, nlw = 3 the tiled summing scatter (k_stage).  Every member explicit."""
    cfg = _cfg(streams, nsw, nlw)
    cp, sw, lw = make_synthetic(cfg, 3000, NLAY)
    _pair(cfg, cp, sw, lw, _tops(cfg, cp.ncol, streams))


@pytest.mark.parametrize("streams", [2, 8])
def test_defaults_and_temperatures(streams):
    """Every member read_input would default and every emission / Planck member None, the temperatures
    given (one air temperature for clear air, vegetation and the air in vegetation), on both routes."""
    cfg = _cfg(streams)
    _pair(cfg, *_defaulted(cfg, 5000, NLAY))


@pytest.mark.parametrize("variant", ["mixed", "mixed_staged"])
def test_mixed_tiles(variant):
    """With SimpleUrban / InfiniteStreet columns the fallback route, without them the staged route:
    ragged layers, Flat tiles, night columns, several spectral intervals; a column sub-range leaves every
    other column and layer alone."""
    cfg = mixed_config(2).consolidate()
    cp, sw, lw = make_mixed(cfg, ncol=400)
    if variant == "mixed_staged":
        cp = _no_simple_urban(cp)
    drv = _tops(cfg, cp.ncol, 5)
    _pair(cfg, cp, sw, lw, drv)
    _assert_poison_outside(_pair(cfg, cp, sw, lw, drv, 37, 311), cp, 37, 311)


@pytest.mark.parametrize("streams", [2, 4])
def test_degenerate_regions(streams):
    cfg, cp, sw, lw = make_degenerate(streams)
    drv = _tops(cfg, cp.ncol, 6)
    _pair(cfg, cp, sw, lw, drv)
    _assert_poison_outside(_pair(cfg, cp, sw, lw, drv, 13, 70), cp, 13, 70)


@pytest.mark.parametrize("case", golden_io.list_cases())
def test_golden(case):
    r, _ = golden_io.load_case(case, legendre_gauss_init=load().ssb200_legendre_gauss_init)
    cfg = r.config
    _pair(cfg, r.canopy_props, r.sw_spectral_props if cfg.do_sw else None,
          r.lw_spectral_props if cfg.do_lw else None, _tops(cfg, r.canopy_props.ncol, len(case)))


@pytest.mark.parametrize("name,value", [(b"stage_layers", 0), (b"fast_kernels", 0), (b"sort_columns", 0),
                                        (b"concurrent_passes", 0), (b"scratch_budget_bytes", 4 << 20)])
def test_under_options(options, name, value):
    """Each option changes the route, the column order or the chunking: still bit-equal."""
    options(name, value)
    cfg = _cfg(2)
    _pair(cfg, *_defaulted(cfg, 3000, NLAY))
    cfgm = mixed_config(2).consolidate()
    cpm, swm, lwm = make_mixed(cfgm, ncol=400)
    _pair(cfgm, _no_simple_urban(cpm), swm, lwm, _tops(cfgm, cpm.ncol, 8))


def test_member_subsets():
    """No flux profiles; do_urban off (Forest tiles); do_vegetation off (Urban tiles)."""
    for kw, rep in ((dict(), None), (dict(do_urban=False), ITileForest), (dict(do_vegetation=False), ITileUrban)):
        cfg = _cfg(2, **kw)
        cp, sw, lw = make_synthetic(cfg, 2000, NLAY)
        if rep is not None:
            cp.i_representation[:] = rep
        _pair(cfg, cp, sw, lw, _tops(cfg, cp.ncol, 9), profiles=False)


@pytest.mark.parametrize("streams", [2, 8])
def test_non_contiguous_packed_layers(streams):
    """The packed layers of the columns in reverse column order (the host entry refuses such ranges): the
    device entry on the permuted layout equals the host entry on the contiguous one, row for row, and the
    layers of columns outside a sub-range keep the poison."""
    import torch
    cfg = _cfg(streams)
    ncol = 1200
    cp, sw, lw, drv = _defaulted(cfg, ncol, NLAY)
    perm_start = ((ncol - 1 - np.arange(ncol)) * NLAY + 1).astype(np.int32)
    rows = (perm_start[:, None] - 1 + np.arange(NLAY)[None, :]).reshape(-1)  # new row of every old row
    inv = np.empty_like(rows)
    inv[rows] = np.arange(rows.size)

    def permuted(obj):
        out = copy.copy(obj)
        for k, v in vars(obj).items():
            if isinstance(v, np.ndarray) and v.dtype == np.float64 and v.shape[0] == cp.ntotlay:
                setattr(out, k, np.ascontiguousarray(v[inv]))
        return out
    pcp = permuted(cp)
    pcp.istartlay = perm_start
    pdrv = {k: (np.ascontiguousarray(v[inv]) if v.shape[0] == cp.ntotlay else v) for k, v in drv.items()}
    for c1, c2 in ((None, None), (101, 977)):
        ref = _outputs(cfg, ncol, cp.ntotlay)
        assert radsurf_fluxes(cfg, cp, sw, lw, ref[0], c1, c2, ref[1], ref[2], **drv) == 0
        got = [_dev(o) for o in _outputs(cfg, ncol, cp.ntotlay)]
        assert radsurf_fluxes(cfg, _dev(pcp), _dev(permuted(sw)), _dev(permuted(lw)), got[0], c1, c2, got[1], got[2],
                              **{k: _dev(v) for k, v in pdrv.items()}) == 0
        torch.cuda.synchronize()
        back = [got[0]] + [copy.copy(o) for o in got[1:]]
        for o in back[1:]:
            for k in ALL_FIELDS:
                v = getattr(o, k)
                if v is not None and v.shape[0] == cp.ntotlay:
                    setattr(o, k, v[torch.from_numpy(rows).cuda()])
        _assert_equal(back, ref)


def test_equals_composed_device_sequence():
    """Against the device entries composed as a GPU-resident caller would have to: radsurf_device on zeroed
    normalised objects, 3 scales and 2 sums (canopy_flux_type.scale / .sum on tensors)."""
    import torch
    cfg = _cfg(2)
    cp, sw, lw = make_synthetic(cfg, 4000, NLAY)
    drv = _tops(cfg, cp.ncol, 12)
    d = {k: _dev(v) for k, v in drv.items()}
    bc = _dev(boundary_conds_out_type().allocate(cp.ncol, 1, 1))
    norm = [canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, 1, use_direct=u, device="cuda")
            for u in (True, True, False, False)]
    assert radsurf(cfg, _dev(cp), _dev(sw), _dev(lw), bc, None, None, *norm) == 0
    norm[0].scale(cp.nlay, d["top_flux_dn_direct_sw"])
    norm[1].scale(cp.nlay, d["top_flux_dn_sw"] - d["top_flux_dn_direct_sw"])
    norm[3].scale(cp.nlay, d["top_flux_dn_lw"])
    sw_ref = canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, 1, use_direct=True, device="cuda")
    lw_ref = canopy_flux_type().allocate(cfg, cp.ncol, cp.ntotlay, 1, use_direct=False, device="cuda")
    sw_ref.sum(norm[0], norm[1])
    lw_ref.sum(norm[2], norm[3])
    got = [_dev(o) for o in _outputs(cfg, cp.ncol, cp.ntotlay)]
    assert radsurf_fluxes(cfg, _dev(cp), _dev(sw), _dev(lw), got[0], None, None, got[1], got[2], **d) == 0
    torch.cuda.synchronize()
    for a, b in ((got[1], sw_ref), (got[2], lw_ref)):
        for k in ALL_FIELDS:
            if getattr(b, k) is not None:
                assert torch.equal(getattr(a, k), getattr(b, k)), k
    for k in golden_io.BC_FIELDS:
        assert torch.equal(getattr(got[0], k), getattr(bc, k)), k


# ---------------------------------------------------------------------------------------------------
# status, ordering, argument errors
# ---------------------------------------------------------------------------------------------------
def _call(lib, cfg, cp, sw, lw, bc, sw_flux, lw_flux, drv, stream=0, status=None):
    ptr = f64_cuda_ptr("test")
    s = marshal(cfg, cp, sw, lw, bc, ptr=ptr)
    d = _abi.DriverInputs(*[ptr(drv.get(k)) for k in DRV_KEYS])
    fsw = sw_flux.as_struct(ptr) if sw_flux is not None else None
    flw = lw_flux.as_struct(ptr) if lw_flux is not None else None
    ref = lambda x: C.byref(x) if x is not None else None
    st = C.cast(status.data_ptr(), C.POINTER(C.c_int32)) if status is not None else None
    return lib.ssb200_radsurf_fluxes_device(ref(s["config"]), ref(s["canopy"]), ref(s["sw"]), ref(s["lw"]), C.byref(d),
                                            ref(s["bc"]), 0, 0, ref(fsw), ref(flw), C.c_void_p(stream), st)


def test_status_and_stream_ordering():
    """status_out equals the host entry's return value; a fluxes_device call on one stream right after a
    radsurf_device call on another (one shared context) gives the results of the same calls made serially."""
    import torch
    lib = load()
    cfg = _cfg(2)
    cpa, swa, lwa, drva = _defaulted(cfg, 20_000, 16)
    cpb, swb, lwb = make_synthetic(cfg, 20_000, 16, col_offset=50_000)
    ref = _outputs(cfg, cpa.ncol, cpa.ntotlay)
    host_rc = radsurf_fluxes(cfg, cpa, swa, lwa, ref[0], None, None, ref[1], ref[2], **drva)
    a_in = [_dev(o) for o in (cpa, swa, lwa)]
    da = {k: _dev(v) for k, v in drva.items()}
    b_in = [_dev(o) for o in (cpb, swb, lwb)]

    def b_outs():
        bc = _dev(boundary_conds_out_type().allocate(cpb.ncol, 1, 1))
        return [bc] + [canopy_flux_type().allocate(cfg, cpb.ncol, cpb.ntotlay, 1, use_direct=u, device="cuda")
                       for u in (True, True, False, False)]
    serial_b, conc_b = b_outs(), b_outs()
    assert radsurf(cfg, *b_in, serial_b[0], None, None, *serial_b[1:]) == 0
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    status = torch.full((1,), -1, dtype=torch.int32, device="cuda")
    got = [_dev(o) for o in _outputs(cfg, cpa.ncol, cpa.ntotlay)]
    torch.cuda.synchronize()
    for _ in range(3):  # back to back, alternating streams, no host synchronisation in between
        assert radsurf(cfg, *b_in, conc_b[0], None, None, *conc_b[1:], stream=s1.cuda_stream) == 0
        with torch.cuda.stream(s2):
            status.fill_(-1)
        assert _call(lib, cfg, *a_in, got[0], got[1], got[2], da, s2.cuda_stream, status) == 0
    s2.synchronize()
    assert int(status.item()) == host_rc
    torch.cuda.synchronize()
    _assert_equal(got, ref)
    for a, b in zip(conc_b, serial_b):
        for k, v in vars(a).items():
            if hasattr(v, "cpu"):
                assert torch.equal(v, getattr(b, k)), k
    lib.ssb200_release()


def test_argument_errors():
    """Missing top-of-canopy flux, a missing flux object and nlw > 1 with a NULL emission member return
    SSB200_ERR_ARG before any launch; the wrapper refuses mixed numpy / tensor members and float32 tensors."""
    import torch
    lib = load()
    cfg = _cfg(2)
    cp, sw, lw = make_synthetic(cfg, 256, 4)
    drv = _tops(cfg, cp.ncol, 1)
    ins = [_dev(o) for o in (cp, sw, lw)]
    out = [_dev(o) for o in _outputs(cfg, cp.ncol, cp.ntotlay)]
    d = {k: _dev(v) for k, v in drv.items()}
    for k in ("top_flux_dn_sw", "top_flux_dn_direct_sw", "top_flux_dn_lw"):
        assert _call(lib, cfg, *ins, out[0], out[1], out[2], dict(d, **{k: None})) == SSB200_ERR_ARG
    assert _call(lib, cfg, *ins, out[0], None, out[2], d) == SSB200_ERR_ARG
    assert _call(lib, cfg, *ins, out[0], out[1], None, d) == SSB200_ERR_ARG
    cfg3 = _cfg(2, 1, 3)
    cp3, sw3, lw3 = make_synthetic(cfg3, 256, 4)
    lw3.roof_emission = None
    out3 = [_dev(o) for o in _outputs(cfg3, cp3.ncol, cp3.ntotlay)]
    assert _call(lib, cfg3, _dev(cp3), _dev(sw3), _dev(lw3), out3[0], out3[1], out3[2],
                 {k: _dev(v) for k, v in _tops(cfg3, cp3.ncol, 2).items()}) == SSB200_ERR_ARG
    torch.cuda.synchronize()
    for o in out:
        for k, v in vars(o).items():
            if hasattr(v, "cpu"):
                assert torch.all(v == POISON), k  # nothing was written
    # the wrapper: numpy and tensors mixed (a member, a top-of-canopy flux, a temperature), float32 tensors
    t = np.full(cp.ntotlay, 290.0)
    for args, kw in (((ins[0], sw, ins[2]), d), ((*ins,), dict(d, top_flux_dn_lw=drv["top_flux_dn_lw"])),
                     ((*ins,), dict(d, roof_temperature=t))):
        with pytest.raises(RadsurfError):
            radsurf_fluxes(cfg, *args, out[0], None, None, out[1], out[2], **kw)
    bad = copy.copy(ins[1])
    bad.veg_ssa = bad.veg_ssa.float()
    with pytest.raises(RadsurfError):
        radsurf_fluxes(cfg, ins[0], bad, ins[2], out[0], None, None, out[1], out[2], **d)
    with pytest.raises(RadsurfError):
        radsurf_fluxes(cfg, *ins, out[0], None, None, out[1], out[2], **dict(d, top_flux_dn_sw=d["top_flux_dn_sw"].float()))
    torch.cuda.synchronize()
