"""ssb200_radsurf_fluxes_device against what a GPU-resident caller runs without it, on the default synthetic
workload (1,048,576 columns x 16 layers, nreg 3, 2 streams, one SW and one LW interval; flux profiles on),
in one invocation.  Three arms on arrays resident in HBM, alternating, timed with CUDA events:

  radsurf_device  ssb200_radsurf_device alone: the four normalised flux objects (bench.py's device step);
  composed        the driver sequence from the separate device entries: ssb200_calc_simple_spectrum_lw_device,
                  ssb200_radsurf_device, 3 x ssb200_canopy_flux_scale_device, 2 x ssb200_canopy_flux_sum_device,
                  with every member read_input would default built by the caller as a full array;
  fluxes_device   ssb200_radsurf_fluxes_device with the NULL-member pattern of bench.py's e2e block.

`--reps` repetitions of `--steps` calls each; median and spread (min, max) of the per-call time.  For each arm:
the HBM the caller allocates (every distinct tensor the arm's calls take) and the bytes per step of the caller's
arrays computed from the shapes (every array an entry reads counted once per entry, every array it writes once;
the solver's scratch and level-major staging traffic, which the three arms share, is not counted).  The outputs of
the composed and the fluxes_device arm are compared bit for bit on a seeded sample of columns.  The card name and
power limit are read in the same run.  Writes <out>/fluxes_device.json.

    python profiles/fluxes_device.py --out <dir>
"""
import argparse
import copy
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from sp_entries import card, stats  # noqa: E402


def tensors(objs):
    """Distinct real tensors of API objects / dicts / tensors."""
    seen = {}
    for o in objs:
        vals = [o] if hasattr(o, "data_ptr") else (o.values() if isinstance(o, dict) else vars(o).values())
        for v in vals:
            if hasattr(v, "data_ptr") and v.is_floating_point():
                seen[v.data_ptr()] = v
    return list(seen.values())


def nbytes(objs):
    return int(sum(t.numel() * t.element_size() for t in tensors(objs)))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--ncol", type=int, default=1 << 20)
    ap.add_argument("--nlay", type=int, default=16)
    ap.add_argument("--streams", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=3, help="calls per repetition")
    ap.add_argument("--no-profiles", dest="profiles", action="store_false", help="flux objects without profiles")
    ap.add_argument("--sample", type=int, default=65536, help="columns in the bit-equality sample")
    args = ap.parse_args()
    import torch
    from spartacus_surface_b200 import radsurf, config_type, canopy_flux_type, boundary_conds_out_type
    from spartacus_surface_b200._lib import load
    from spartacus_surface_b200.radsurf_interface import radsurf_fluxes
    from spartacus_surface_b200.synthetic import make_synthetic
    if not torch.cuda.is_available():
        raise SystemExit("fluxes_device.py needs a CUDA device")
    lib = load()
    lib.ssb200_set_device(0)
    ncol, nlay, dev = args.ncol, args.nlay, "cuda:0"
    cfg = config_type(do_sw=True, do_lw=True, nsw=1, nlw=1, n_vegetation_region_urban=2, n_vegetation_region_forest=2,
                      n_stream_sw_urban=args.streams, n_stream_lw_urban=args.streams,
                      n_stream_sw_forest=args.streams, n_stream_lw_forest=args.streams).consolidate()
    cp, sw, lw, temps = make_synthetic(cfg, ncol, nlay, device=dev, with_temperatures=True)
    ntot = cp.ntotlay
    g = torch.Generator(device="cpu").manual_seed(7)
    top_sw = (200.0 + 700.0 * torch.rand((ncol, 1), generator=g, dtype=torch.float64)).to(dev)
    tops = {"top_flux_dn_sw": top_sw,
            "top_flux_dn_direct_sw": (top_sw * (0.2 + 0.7 * torch.rand((ncol, 1), generator=g, dtype=torch.float64)
                                                .to(dev))).contiguous(),
            "top_flux_dn_lw": (250.0 + 150.0 * torch.rand((ncol, 1), generator=g, dtype=torch.float64)).to(dev)}
    flux = lambda d: canopy_flux_type().allocate(cfg, ncol, ntot, 1, use_direct=d, do_save_flux_profile=args.profiles,
                                                 device=dev)
    bc_of = lambda: boundary_conds_out_type().allocate(ncol, 1, 1, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    dp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None

    # radsurf_device: every member explicit (make_synthetic builds them all)
    a_bc, a_norm = bc_of(), [flux(d) for d in (True, True, False, False)]

    def arm_radsurf():
        assert radsurf(cfg, cp, sw, lw, a_bc, None, None, *a_norm, stream=stream) == 0

    # composed: the caller holds emission arrays filled from the temperatures, the four normalised objects and
    # the two summed ones
    b_bc, b_norm, b_sw, b_lw = bc_of(), [flux(d) for d in (True, True, False, False)], flux(True), flux(False)
    lw_b = copy.copy(lw)
    for k in ("ground_emission", "roof_emission", "wall_emission", "clear_air_planck", "veg_planck", "veg_air_planck"):
        setattr(lw_b, k, torch.empty_like(getattr(lw, k)))
    lw_b_struct = lw_b.as_struct()
    diff_factor = torch.empty_like(tops["top_flux_dn_sw"])

    def arm_composed():
        rc = lib.ssb200_calc_simple_spectrum_lw_device(
            C.byref(lw_b_struct), ncol, ntot, 0, 0, 0, ntot, dp(temps["ground_temperature"]), dp(temps["roof_temperature"]),
            dp(temps["wall_temperature"]), dp(temps["clear_air_temperature"]), dp(temps["veg_temperature"]),
            dp(temps["veg_air_temperature"]), C.c_void_p(stream))
        assert rc == 0
        assert radsurf(cfg, cp, sw, lw_b, b_bc, None, None, *b_norm, stream=stream) == 0
        torch.sub(tops["top_flux_dn_sw"], tops["top_flux_dn_direct_sw"], out=diff_factor)
        b_norm[0].scale(cp.nlay, tops["top_flux_dn_direct_sw"])
        b_norm[1].scale(cp.nlay, diff_factor)
        b_norm[3].scale(cp.nlay, tops["top_flux_dn_lw"])
        b_sw.sum(b_norm[0], b_norm[1])
        b_lw.sum(b_norm[2], b_norm[3])

    # fluxes_device: NULL members as in bench.py's e2e block
    cp_c, sw_c, lw_c = copy.copy(cp), copy.copy(sw), copy.copy(lw)
    cp_c.veg_contact_fraction = None
    sw_c.air_ext = sw_c.air_ssa = sw_c.wall_specular_frac = sw_c.roof_albedo_dir = None
    lw_c.air_ext = lw_c.air_ssa = None
    for k in ("ground_emission", "roof_emission", "wall_emission", "clear_air_planck", "veg_planck", "veg_air_planck"):
        setattr(lw_c, k, None)
    c_bc, c_sw, c_lw = bc_of(), flux(True), flux(False)

    def arm_fluxes():
        assert radsurf_fluxes(cfg, cp_c, sw_c, lw_c, c_bc, None, None, c_sw, c_lw, stream=stream, **tops, **temps) == 0

    ins = [cp, sw, lw]
    arms = {
        "radsurf_device": dict(fn=arm_radsurf, call="ssb200_radsurf_device",
                               caller=[cp, sw, lw, a_bc] + a_norm,
                               step=nbytes(ins) + nbytes([a_bc] + a_norm)),
        "composed": dict(fn=arm_composed,
                         call="calc_simple_spectrum_lw_device + radsurf_device + 3 scale_device + 2 sum_device",
                         caller=[cp, sw, lw_b, temps, tops, diff_factor, b_bc, b_sw, b_lw] + b_norm,
                         # emission: temperatures and emissivities read, emission written; radsurf; scales read
                         # and write 3 objects; sums read 4, write 2
                         step=(nbytes([temps, lw.ground_emissivity, lw.roof_emissivity, lw.wall_emissivity])
                               + nbytes([lw_b.ground_emission, lw_b.roof_emission, lw_b.wall_emission,
                                         lw_b.clear_air_planck, lw_b.veg_planck, lw_b.veg_air_planck])
                               + nbytes([cp, sw, lw_b]) + nbytes([b_bc] + b_norm)
                               + 2 * nbytes([b_norm[0], b_norm[1], b_norm[3]]) + nbytes(list(tops.values()))
                               + nbytes(b_norm) + nbytes([b_sw, b_lw]))),
        "fluxes_device": dict(fn=arm_fluxes, call="ssb200_radsurf_fluxes_device",
                              caller=[cp_c, sw_c, lw_c, temps, tops, c_bc, c_sw, c_lw],
                              step=nbytes([cp_c, sw_c, lw_c, temps, tops]) + nbytes([c_bc, c_sw, c_lw])),
    }
    for a in arms.values():
        a["fn"]()  # warm-up: plan, scratch, context buffers
        a["ms"] = []
    torch.cuda.synchronize()
    for _ in range(args.reps):
        for a in arms.values():  # alternating arms
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                a["fn"]()
            e1.record()
            torch.cuda.synchronize()
            a["ms"].append(e0.elapsed_time(e1) / args.steps)

    # bit-equality of the composed and the fluxes_device outputs on a seeded column sample
    seed = 20261020
    cols = np.sort(np.random.default_rng(seed).choice(ncol, size=min(args.sample, ncol), replace=False))
    rows = np.concatenate([np.arange(cp.istartlay[c] - 1, cp.istartlay[c] - 1 + cp.nlay[c]) for c in cols])
    checked, bad = 0, []
    for name, x, y in (("bc", b_bc, c_bc), ("sw_flux", b_sw, c_sw), ("lw_flux", b_lw, c_lw)):
        for k, v in vars(x).items():
            if not hasattr(v, "cpu"):
                continue
            idx = torch.from_numpy(cols if v.shape[0] == ncol else rows).to(dev)
            p, q = v[idx], getattr(y, k)[idx]
            checked += p.numel()
            if not torch.equal(p, q):
                bad.append(f"{name}.{k}")
    result = {"card": card(),
              "workload": {"ncol": ncol, "nlay": nlay, "nreg": 3, "streams": args.streams, "nsw": 1, "nlw": 1,
                           "flux_profiles": args.profiles, "reps": args.reps, "calls_per_rep": args.steps},
              "timing": "CUDA events on the launch stream per call; arrays resident in HBM (no PCIe)",
              "bytes_per_step": "caller arrays only, from shapes: each array an entry reads or writes counted once "
                                "per entry (scratch and staging traffic of the solve not counted)",
              "check": {"sample_columns": int(cols.size), "seed": seed, "values_compared": checked,
                        "composed_vs_fluxes_device_bit_equal": not bad, "mismatching_members": bad}}
    for tag, a in arms.items():
        result[tag] = dict(call=a["call"], caller_hbm_bytes=nbytes(a["caller"]), bytes_per_step=int(a["step"]),
                           **stats(a["ms"]))
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "fluxes_device.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("card", "check")}))
    for tag in arms:
        r = result[tag]
        print(tag, round(r["median_ms"], 2), "ms", f"caller HBM {r['caller_hbm_bytes'] / 1e9:.2f} GB",
              f"step {r['bytes_per_step'] / 1e9:.2f} GB")
    lib.ssb200_release()
    if bad:
        raise SystemExit("fluxes_device outputs differ from the composed device sequence")


if __name__ == "__main__":
    main()
