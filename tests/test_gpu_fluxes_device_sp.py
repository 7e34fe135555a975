"""GPU tests of ssb200_radsurf_fluxes_device_sp: the reference driver's calc_simple_spectrum_lw + radsurf + scale
+ sum on float32 device arrays.  Every output must equal, bit for bit, the float64 driver sequence on the
widened inputs rounded to float32, and (contiguous layouts) ssb200_radsurf_fluxes_sp on the same float32 host
arrays: each comparison is np.array_equal over whole arrays.  Outputs start from a finite poison value, so
columns outside istartcol..iendcol and layers no selected column owns are checked too.  Both routes run: the
staged route (float gather, rounding summing scatter, register-resident kernels of 1-4 streams) and the
fallback route (8 streams, generic kernels, stage_layers = 0, column-resident kernels, single-layer urban
columns)."""
import copy
import ctypes as C

import numpy as np
import pytest

import golden_io
from degenerate_case import make_degenerate
from mixed_case import mixed_config, make_mixed
from spartacus_surface_b200 import RadsurfError, boundary_conds_out_type, canopy_flux_type, radsurf
from spartacus_surface_b200 import _abi
from spartacus_surface_b200._lib import load
from spartacus_surface_b200.radsurf_canopy_flux import ALL_FIELDS
from spartacus_surface_b200.radsurf_canopy_properties import ITileForest, ITileUrban
from spartacus_surface_b200.radsurf_interface import f32_ptr, marshal, radsurf_fluxes, radsurf_fluxes_sp, to_single
from spartacus_surface_b200.synthetic import make_synthetic
from test_gpu_fluxes_device import (POISON, NLAY, SSB200_ERR_ARG, DRV_KEYS, _cfg, _outputs, _tops, _defaulted,
                                    _no_simple_urban)

pytestmark = pytest.mark.gpu

DEFAULTS = {b"stage_layers": 1, b"fast_kernels": 1, b"fused_kernels": 0, b"sort_columns": 1,
            b"concurrent_passes": 1, b"scratch_budget_bytes": 0}


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


def _single(obj):
    if obj is None or isinstance(obj, np.ndarray):
        return None if obj is None else np.ascontiguousarray(obj.astype(np.float32))
    return to_single(obj)


def _wide(obj):
    """Copy with every float32 numpy member widened to float64 (exact)."""
    if obj is None or isinstance(obj, np.ndarray):
        return None if obj is None else obj.astype(np.float64)
    out = copy.copy(obj)
    for k, v in vars(obj).items():
        if isinstance(v, np.ndarray) and v.dtype == np.float32:
            setattr(out, k, v.astype(np.float64))
    return out


def _dev(obj):
    """Copy with every float32 numpy member as a torch CUDA tensor."""
    import torch
    if obj is None:
        return None
    if isinstance(obj, np.ndarray):
        return torch.from_numpy(np.ascontiguousarray(obj)).cuda()
    out = copy.copy(obj)
    for k, v in vars(obj).items():
        if isinstance(v, np.ndarray) and v.dtype == np.float32:
            setattr(out, k, torch.from_numpy(np.ascontiguousarray(v)).cuda())
    return out


def _host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else a


def _assert_equal(got, want):
    """got: float32 outputs (tensors or arrays); want: float64 or float32 numpy outputs, rounded here."""
    n = 0
    for a, b in zip(got, want):
        for k, v in vars(b).items():
            if not isinstance(v, np.ndarray) or v.dtype.kind != "f":
                continue
            x = _host(getattr(a, k))
            assert x.dtype == np.float32, k
            y = v.astype(np.float32)
            assert np.array_equal(x, y), (k, float(np.abs(x.astype(np.float64) - y).max()))
            n += 1
    assert n > 0
    return n


def _sp_outputs(cfg, ncol, ntot, profiles=True):
    return [to_single(o) for o in _outputs(cfg, ncol, ntot, profiles)]


def _run_device(cfg, cp, sw, lw, drv, c1=None, c2=None, profiles=True):
    """The new entry on float32 device copies of the float32 inputs; returns the device outputs."""
    import torch
    got = [_dev(o) for o in _sp_outputs(cfg, cp.ncol, cp.ntotlay, profiles)]
    assert radsurf_fluxes_sp(cfg, _dev(cp), _dev(sw), _dev(lw), got[0], c1, c2, got[1], got[2],
                             **{k: _dev(v) for k, v in drv.items()}) == 0
    torch.cuda.synchronize()
    return got


def _pair(cfg, cp, sw, lw, drv, c1=None, c2=None, profiles=True):
    """Inputs rounded to float32; the new entry against the float64 host entry on the widened inputs (cast)
    and against ssb200_radsurf_fluxes_sp on the same float32 host arrays."""
    cp, sw, lw = _single(cp), _single(sw), _single(lw)
    drv = {k: _single(v) for k, v in drv.items()}
    ref = _outputs(cfg, cp.ncol, cp.ntotlay, profiles)
    assert radsurf_fluxes(cfg, _wide(cp), _wide(sw), _wide(lw), ref[0], c1, c2, ref[1], ref[2],
                          **{k: _wide(v) for k, v in drv.items()}) == 0
    host = _sp_outputs(cfg, cp.ncol, cp.ntotlay, profiles)
    assert radsurf_fluxes_sp(cfg, cp, sw, lw, host[0], c1, c2, host[1], host[2], **drv) == 0
    got = _run_device(cfg, cp, sw, lw, drv, c1, c2, profiles)
    _assert_equal(got, ref)
    _assert_equal(got, host)
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


# ---------------------------------------------------------------------------------------------------
# workloads and routes
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("streams,nsw,nlw", [(1, 1, 1), (2, 1, 1), (4, 1, 1), (8, 1, 1), (2, 2, 3)])
def test_synthetic(streams, nsw, nlw):
    """1, 2 and 4 streams take the staged route (k_stage1 rounding summing scatter, float4 and scalar
    branches at 9 layers), 8 streams the fallback; nsw = 2, nlw = 3 the tiled scatter (k_stage)."""
    cfg = _cfg(streams, nsw, nlw)
    cp, sw, lw = make_synthetic(cfg, 3000, NLAY)
    _pair(cfg, cp, sw, lw, _tops(cfg, cp.ncol, streams))


@pytest.mark.parametrize("streams", [1, 2, 4, 8])
def test_defaults_and_temperatures(streams):
    """Every member read_input would default and every emission / Planck member None, the temperatures given:
    the defaults, sigma T^4 and the default contact fraction stay float64 next to the staged float arrays."""
    cfg = _cfg(streams)
    _pair(cfg, *_defaulted(cfg, 5000, NLAY))


@pytest.mark.parametrize("variant", ["mixed", "mixed_staged"])
def test_mixed_tiles(variant):
    """With SimpleUrban / InfiniteStreet columns the fallback route, without them the staged route: ragged
    layers, Flat tiles, night columns, several spectral intervals; a column sub-range leaves every other
    column and layer alone."""
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


@pytest.mark.parametrize("name,value", [(b"stage_layers", 0), (b"fast_kernels", 0), (b"fused_kernels", 1),
                                        (b"sort_columns", 0), (b"concurrent_passes", 0),
                                        (b"scratch_budget_bytes", 4 << 20)])
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
    """The packed layers of the columns in reverse column order: the new entry on the permuted layout equals
    it on the contiguous one, row for row, and the layers of columns outside a sub-range keep the poison."""
    import torch
    cfg = _cfg(streams)
    ncol = 1200
    cp, sw, lw, drv = _defaulted(cfg, ncol, NLAY)
    cp, sw, lw = _single(cp), _single(sw), _single(lw)
    drv = {k: _single(v) for k, v in drv.items()}
    perm_start = ((ncol - 1 - np.arange(ncol)) * NLAY + 1).astype(np.int32)
    rows = (perm_start[:, None] - 1 + np.arange(NLAY)[None, :]).reshape(-1)  # new row of every old row
    inv = np.empty_like(rows)
    inv[rows] = np.arange(rows.size)

    def permuted(obj):
        out = copy.copy(obj)
        for k, v in vars(obj).items():
            if isinstance(v, np.ndarray) and v.dtype == np.float32 and v.shape[0] == cp.ntotlay:
                setattr(out, k, np.ascontiguousarray(v[inv]))
        return out
    pcp = permuted(cp)
    pcp.istartlay = perm_start
    pdrv = {k: (np.ascontiguousarray(v[inv]) if v.shape[0] == cp.ntotlay else v) for k, v in drv.items()}
    for c1, c2 in ((None, None), (101, 977)):
        ref = _run_device(cfg, cp, sw, lw, drv, c1, c2)
        got = _run_device(cfg, pcp, permuted(sw), permuted(lw), pdrv, c1, c2)
        back = [got[0]] + [copy.copy(o) for o in got[1:]]
        for o in back[1:]:
            for k in ALL_FIELDS:
                v = getattr(o, k)
                if v is not None and v.shape[0] == cp.ntotlay:
                    setattr(o, k, v[torch.from_numpy(rows).cuda()])
        for a, b in zip(back, ref):
            for k, v in vars(b).items():
                if hasattr(v, "cpu"):
                    assert torch.equal(getattr(a, k), v), k


# ---------------------------------------------------------------------------------------------------
# status, ordering, argument errors
# ---------------------------------------------------------------------------------------------------
def _call(lib, cfg, cp, sw, lw, bc, sw_flux, lw_flux, drv, stream=0, status=None):
    ptr = f32_ptr(True, "test")
    s = marshal(cfg, cp, sw, lw, bc, ptr=ptr)
    d = _abi.DriverInputs(*[ptr(drv.get(k)) for k in DRV_KEYS]) if drv is not None else None
    fsw = sw_flux.as_struct(ptr) if sw_flux is not None else None
    flw = lw_flux.as_struct(ptr) if lw_flux is not None else None
    ref = lambda x: C.byref(x) if x is not None else None
    st = C.cast(status.data_ptr(), C.POINTER(C.c_int32)) if status is not None else None
    return lib.ssb200_radsurf_fluxes_device_sp(ref(s["config"]), ref(s["canopy"]), ref(s["sw"]), ref(s["lw"]),
                                               ref(d), ref(s["bc"]), 0, 0, ref(fsw), ref(flw), C.c_void_p(stream), st)


def test_status_and_stream_ordering():
    """status_out equals the host entry's return value; a call on one stream right after a float64
    radsurf_device call on another (one shared context) gives the results of the same calls made serially."""
    import torch
    lib = load()
    cfg = _cfg(2)
    cpa, swa, lwa, drva = _defaulted(cfg, 20_000, 16)
    cpa, swa, lwa = _single(cpa), _single(swa), _single(lwa)
    drva = {k: _single(v) for k, v in drva.items()}
    cpb, swb, lwb = make_synthetic(cfg, 20_000, 16, col_offset=50_000)
    host = _sp_outputs(cfg, cpa.ncol, cpa.ntotlay)
    host_rc = radsurf_fluxes_sp(cfg, cpa, swa, lwa, host[0], None, None, host[1], host[2], **drva)
    a_in = [_dev(o) for o in (cpa, swa, lwa)]
    da = {k: _dev(v) for k, v in drva.items()}

    def d64(obj):
        out = copy.copy(obj)
        for k, v in vars(obj).items():
            if isinstance(v, np.ndarray) and v.dtype == np.float64:
                setattr(out, k, torch.from_numpy(np.ascontiguousarray(v)).cuda())
        return out
    b_in = [d64(o) for o in (cpb, swb, lwb)]

    def b_outs():
        bc = d64(boundary_conds_out_type().allocate(cpb.ncol, 1, 1))
        return [bc] + [canopy_flux_type().allocate(cfg, cpb.ncol, cpb.ntotlay, 1, use_direct=u, device="cuda")
                       for u in (True, True, False, False)]
    serial_b, conc_b = b_outs(), b_outs()
    assert radsurf(cfg, *b_in, serial_b[0], None, None, *serial_b[1:]) == 0
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    status = torch.full((1,), -1, dtype=torch.int32, device="cuda")
    got = [_dev(o) for o in _sp_outputs(cfg, cpa.ncol, cpa.ntotlay)]
    torch.cuda.synchronize()
    for _ in range(3):  # back to back, alternating streams, no host synchronisation in between
        assert radsurf(cfg, *b_in, conc_b[0], None, None, *conc_b[1:], stream=s1.cuda_stream) == 0
        with torch.cuda.stream(s2):
            status.fill_(-1)
        assert _call(lib, cfg, *a_in, got[0], got[1], got[2], da, s2.cuda_stream, status) == 0
    s2.synchronize()
    assert int(status.item()) == host_rc
    torch.cuda.synchronize()
    _assert_equal(got, host)
    for a, b in zip(conc_b, serial_b):
        for k, v in vars(a).items():
            if hasattr(v, "cpu"):
                assert torch.equal(v, getattr(b, k)), k
    lib.ssb200_release()


def test_argument_errors():
    """NULL driver_inputs, a missing top-of-canopy flux or flux object, and an unknown tile code return
    SSB200_ERR_ARG with nothing written; the wrapper refuses mixed numpy / tensor members and float64 tensors."""
    import torch
    lib = load()
    cfg = _cfg(2)
    cp, sw, lw = (_single(o) for o in make_synthetic(cfg, 256, 4))
    drv = {k: _single(v) for k, v in _tops(cfg, cp.ncol, 1).items()}
    ins = [_dev(o) for o in (cp, sw, lw)]
    out = [_dev(o) for o in _sp_outputs(cfg, cp.ncol, cp.ntotlay)]
    d = {k: _dev(v) for k, v in drv.items()}
    assert _call(lib, cfg, *ins, out[0], out[1], out[2], None) == SSB200_ERR_ARG
    for k in ("top_flux_dn_sw", "top_flux_dn_direct_sw", "top_flux_dn_lw"):
        assert _call(lib, cfg, *ins, out[0], out[1], out[2], dict(d, **{k: None})) == SSB200_ERR_ARG
    assert _call(lib, cfg, *ins, out[0], None, out[2], d) == SSB200_ERR_ARG
    assert _call(lib, cfg, *ins, out[0], out[1], None, d) == SSB200_ERR_ARG
    bad_cp = copy.copy(ins[0])
    bad_cp.i_representation = cp.i_representation.copy()
    bad_cp.i_representation[17] = 99
    assert _call(lib, cfg, bad_cp, ins[1], ins[2], out[0], out[1], out[2], d) == SSB200_ERR_ARG
    torch.cuda.synchronize()
    for o in out:
        for k, v in vars(o).items():
            if hasattr(v, "cpu"):
                assert torch.all(v == POISON), k  # nothing was written
    # the device is still usable: a valid call succeeds
    assert _call(lib, cfg, *ins, out[0], out[1], out[2], d) == 0
    torch.cuda.synchronize()
    # the wrapper: numpy and tensors mixed (a member, a top-of-canopy flux, a temperature), float64 tensors
    t = np.full(cp.ntotlay, 290.0, dtype=np.float32)
    for args, kw in (((ins[0], sw, ins[2]), d), ((*ins,), dict(d, top_flux_dn_lw=drv["top_flux_dn_lw"])),
                     ((*ins,), dict(d, roof_temperature=t))):
        with pytest.raises(RadsurfError):
            radsurf_fluxes_sp(cfg, *args, out[0], None, None, out[1], out[2], **kw)
    bad = copy.copy(ins[1])
    bad.veg_ssa = bad.veg_ssa.double()
    with pytest.raises(RadsurfError):
        radsurf_fluxes_sp(cfg, ins[0], bad, ins[2], out[0], None, None, out[1], out[2], **d)
    with pytest.raises(RadsurfError):
        radsurf_fluxes_sp(cfg, *ins, out[0], None, None, out[1], out[2],
                          **dict(d, top_flux_dn_sw=d["top_flux_dn_sw"].double()))
    # the float64 entry still refuses float32 tensors
    with pytest.raises(RadsurfError):
        radsurf_fluxes(cfg, *ins, out[0], None, None, out[1], out[2], **d)
    torch.cuda.synchronize()
