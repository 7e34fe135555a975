"""The configuration matrix of tests/coverage_case.py through the host build of the solver bodies
(tests/hostcheck) against the oracle and its _Float128 truth: every register-resident shape
(pass x NREG 1-3 x NS 1-4 x URBAN) and every generic stream count 5-8, on inputs whose regions and
boundary conditions cannot be confused with one another.  Also checks that the matrix reaches what
it claims to reach and that the inputs really are asymmetric, and pins the truth on the branches
(isolation factor, asymmetric vegetation scale, scattering air, distinct Planck functions) with the
independent implementation of tests/bvp_reference.py."""
import numpy as np
import pytest

import coverage_case as cc
import hostcheck_lib
import oracle_lib
import parity

NAMES = [s["name"] for s in cc.SPECS]


def _identical(a, b):
    for name, fields in b.items():
        for k, v in fields.items():
            assert np.array_equal(a[name][k], v), (name, k, np.abs(a[name][k] - v).max())


def _check(got, status, name, factor=parity.REF_FACTOR):
    o = cc.oracle_runs(name)
    assert status == 0
    assert not cc.poison_mismatches(got, o["fma"]), cc.poison_mismatches(got, o["fma"])
    ref = o["fma"]
    return parity.check(cc.unpoison(got, ref), cc.unpoison(o["quad"], ref), cc.unpoison(o["fma"], ref),
                        cc.unpoison(o["nofma"], ref), factor=factor)


# ---- what the matrix reaches -------------------------------------------------------------------

def test_matrix_reaches_every_kernel_shape():
    reached = set().union(*(cc.shapes(s) for s in cc.SPECS))
    assert reached == cc.full_shape_set(), sorted(cc.full_shape_set() - reached)
    generic = set().union(*(cc.generic_uses(s) for s in cc.SPECS))
    for ns in cc.GENERIC_NS:
        for p in ("sw", "lw"):
            assert any(g[0] == p and g[1] == ns for g in generic), (p, ns)
        for urban in (0, 1):
            assert any(g[1] == ns and g[2] == urban for g in generic), (ns, urban)


def test_matrix_covers_the_configurations():
    default = cc.BY_NAME[cc.DEFAULT]
    assert all(default[f"n_stream_{p}_{k}"] == 4 for p in ("sw", "lw") for k in ("forest", "urban"))
    assert default["n_vegetation_region_forest"] == default["n_vegetation_region_urban"] == 1
    assert any(s["n_vegetation_region_forest"] != s["n_vegetation_region_urban"]
               and all(s[f"n_stream_{p}_forest"] != s[f"n_stream_{p}_urban"] for p in ("sw", "lw")) for s in cc.SPECS)
    assert any(s[f"n_stream_sw_{k}"] != s[f"n_stream_lw_{k}"] for s in cc.SPECS for k in ("forest", "urban"))
    for iso in (0.5, 1.0):
        assert any(s.get("vegetation_isolation_factor_forest") == iso and s["n_vegetation_region_forest"] == 2
                   for s in cc.SPECS), iso
        assert any(s.get("vegetation_isolation_factor_urban") == iso and s["n_vegetation_region_urban"] == 2
                   for s in cc.SPECS), iso
    assert any(s.get("use_symmetric_vegetation_scale_forest") is False
               and s.get("use_symmetric_vegetation_scale_urban") is False for s in cc.SPECS)
    assert sum(s.get("use_sw_direct_albedo", True) for s in cc.SPECS) > len(cc.SPECS) // 2
    for s in cc.SPECS:
        cfg, cp, _, _ = cc.make_case(s)
        assert cp.ncol <= 48 and int(cp.nlay.max()) <= 9
        for urban, nreg in cc.classes(s):
            assert cc.columns(cp, urban, nreg, s).size > 0, (s["name"], urban, nreg)


# ---- the inputs are asymmetric ---------------------------------------------------------------

def _truth(cfg, cp, sw, lw):
    out, status = cc.run(cfg, cp, sw, lw, oracle_lib.make_solver(quad=True))
    assert status == 0
    return out


def _moved(a, b, obj, keys=None):
    """Largest relative change of the fields of `obj` between two runs."""
    worst = 0.0
    for k, v in a[obj].items():
        if keys is not None and k not in keys:
            continue
        scale = max(float(np.abs(v).max()), 1e-300)
        worst = max(worst, float(np.abs(v - b[obj][k]).max()) / scale)
    return worst


def test_inputs_break_the_symmetries():
    """Each perturbation of make_case changes the truth: a kernel that confused the two inputs it
    separates would fail the parity tests."""
    spec = cc.BY_NAME["r3_s2_iso05_asym"]
    base = cc.oracle_runs(spec["name"])["quad"]
    # vegetation and vegetation-air Planck functions swapped
    cfg, cp, sw, lw = cc.make_case(spec)
    lw.veg_planck, lw.veg_air_planck = lw.veg_air_planck, lw.veg_planck
    assert _moved(base, _truth(cfg, cp, sw, lw), "bc", ("lw_emission",)) > 1e-3
    # longwave air does not scatter
    cfg, cp, sw, lw = cc.make_case(spec)
    lw.air_ssa = np.zeros_like(lw.air_ssa)
    t = _truth(cfg, cp, sw, lw)
    assert min(_moved(base, t, "lw_internal"), _moved(base, t, "lw_norm")) > 1e-6
    # direct roof albedo equal to the diffuse one
    cfg, cp, sw, lw = cc.make_case(spec)
    sw.roof_albedo_dir = sw.roof_albedo.copy()
    assert _moved(base, _truth(cfg, cp, sw, lw), "bc", ("sw_albedo_dir",)) > 1e-6
    # no isolation: the three-region columns of both tile kinds move
    cfg, cp, sw, lw = cc.make_case(dict(spec, vegetation_isolation_factor_forest=0.0,
                                        vegetation_isolation_factor_urban=0.0))
    t = _truth(cfg, cp, sw, lw)
    for urban in (0, 1):
        cols = cc.columns(cp, urban, 3, spec)
        for k in ("sw_albedo", "lw_emission"):
            a, b = base["bc"][k][cols], t["bc"][k][cols]
            assert np.abs(a - b).max() > 1e-6 * np.abs(a).max(), (urban, k)
    # the perturbations themselves
    cfg, cp, sw, lw = cc.make_case(spec)
    for a, b in ((lw.veg_planck, lw.veg_air_planck), (lw.veg_planck, lw.clear_air_planck),
                 (lw.veg_air_planck, lw.clear_air_planck), (sw.ground_albedo_dir, sw.ground_albedo)):
        assert np.all(a != b)
    assert np.all((sw.wall_specular_frac > 0.0) & (sw.wall_specular_frac < 1.0))


# ---- per spec: the host build of the kernels' bodies ---------------------------------------

@pytest.mark.parametrize("name", NAMES)
def test_generic_bodies_bit_identical_to_nofma_oracle(name):
    got, status = cc.run(*cc.make_case(cc.BY_NAME[name]), hostcheck_lib.make_solver())
    assert status == 0
    _identical(got, cc.oracle_runs(name)["nofma"])


MODES = {"interface_sweeps": dict(fast=True), "interface_sweeps_unstaged": dict(fast=True, stage=False),
         "record_sweeps": dict(records=True)}


@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("name", NAMES)
def test_register_resident_bodies_vs_truth(name, mode):
    """The register-resident bodies (generic ones for 5-8 streams) against the _Float128 truth with
    the rule of tests/parity.py."""
    spec = cc.BY_NAME[name]
    if mode == "record_sweeps" and not any(s[2] <= 2 for s in cc.shapes(spec)):
        pytest.skip("record sweeps exist for 1 and 2 streams only")
    got, status = cc.run(*cc.make_case(spec), hostcheck_lib.make_solver(**MODES[mode]))
    ok, worst, lines = _check(got, status, name)
    assert ok, "\n".join(lines)


@pytest.mark.parametrize("name", NAMES)
def test_generic_device_formulation_vs_truth(name):
    """The generic bodies as the device builds them (symmetrised Jacobi eigen-systems), factor 4."""
    got, status = cc.run(*cc.make_case(cc.BY_NAME[name]), hostcheck_lib.make_solver(generic_jacobi=True))
    ok, worst, lines = _check(got, status, name, factor=4.0)
    o = cc.oracle_runs(name)
    if not ok and parity.max_err(cc.unpoison(o["fma"], o["fma"]), cc.unpoison(o["quad"], o["fma"])) > 1e-2:
        pytest.skip("reference arithmetic order has no correct digit on this case (LU without pivoting)")
    assert ok, "\n".join(lines)


# ---- the truth itself on the new branches ------------------------------------------------------

def test_truth_pinned_on_isolation_asymmetric_scale_and_scattering_air():
    """One vegetated-urban column of the matrix (3 regions, 2 streams, isolation 0.5, asymmetric
    vegetation scale, distinct Planck functions, scattering longwave air) through the independent
    operators of tests/bvp_reference.py and the reference's sweep recurrences (mode "sic", as in
    test_bvp_pin.py): every field of both passes within 1e-11 of the _Float128 oracle.  The forest
    isolation branch (csrc/ssb_geometry.cuh) has no independent implementation: bvp_reference.py
    solves urban and vegetated-urban tiles only."""
    import bvp_reference as bvp
    spec = cc.BY_NAME["r3_s2_iso05_asym"]
    cfg, cp, sw, lw = cc.make_case(spec)
    assert cfg.vegetation_isolation_factor_urban == 0.5 and not cfg.use_symmetric_vegetation_scale_urban
    assert cfg.n_vegetation_region_urban == 2 and cfg.n_stream_sw_urban == cfg.n_stream_lw_urban == 2
    cols = [j for j in cc.columns(cp, 1, 3, spec) if 2 <= cp.nlay[j] <= 4 and cp.cos_sza[j] > 0.0]
    icol = int(cols[0])
    il1, L = int(cp.istartlay[icol]) - 1, int(cp.nlay[icol])
    assert np.all(cp.veg_fraction[il1:il1 + L] > 0.0) and cp.cos_sza[icol] > 0.0
    truth = cc.oracle_runs(spec["name"])["quad"]
    for band, spectral, nspec in (("sw", sw, cfg.nsw), ("lw", lw, cfg.nlw)):
        for g in range(nspec):
            out = bvp.solve_column(cfg, cp, spectral, icol, g, band, mode="sic")
            for obj, fields in out.items():
                scale = 1.0 if obj == "bc" else max(abs(float(truth[obj][k][icol, g]))
                                                    for k in ("top_dn", "top_net", "ground_dn", "ground_net"))
                for k, v in fields.items():
                    t = truth[obj][k]
                    if isinstance(v, list):
                        tv, bv = t[il1:il1 + L, g], np.array([float(x) for x in v])
                    else:
                        tv, bv = np.array([t[icol, g]]), np.array([float(v)])
                    err = float(np.abs(bv - tv).max() / max(np.abs(tv).max(), 1e-3 * scale))
                    assert err <= 1e-11, (band, g, obj, k, err)
