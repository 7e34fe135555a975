"""ssb200_radsurf_fluxes_device_sp against its float64 twin ssb200_radsurf_fluxes_device, on the default synthetic
workload (1,048,576 columns x 16 layers, nreg 3, 2 streams, one SW and one LW interval; flux profiles on) with
the NULL-member pattern of bench.py's e2e block, in one invocation.  Two arms on arrays resident in HBM,
alternating, timed with CUDA events:

  fluxes_device     ssb200_radsurf_fluxes_device on float64 tensors (the float32 inputs widened);
  fluxes_device_sp  ssb200_radsurf_fluxes_device_sp on the float32 tensors.

`--reps` repetitions of `--steps` calls each; median and spread (min, max) of the per-call time.  For each arm
the HBM the caller allocates (every distinct tensor the arm's call takes).  The float32 outputs are compared
bit for bit with the float64 outputs cast to float32 on a seeded sample of columns.  The card name and power
limit are read in the same run.  Writes <out>/fluxes_device_sp.json.

    python profiles/fluxes_device_sp.py --out <dir>
"""
import argparse
import copy
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from fluxes_device import nbytes  # noqa: E402
from sp_entries import card, stats  # noqa: E402


def converted(obj, fn):
    """Copy of an API object or dict with every floating tensor member mapped by fn."""
    out = dict(obj) if isinstance(obj, dict) else copy.copy(obj)
    items = obj.items() if isinstance(obj, dict) else vars(obj).items()
    for k, v in items:
        if hasattr(v, "data_ptr") and v.is_floating_point():
            if isinstance(out, dict):
                out[k] = fn(v)
            else:
                setattr(out, k, fn(v))
    return out


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
    from spartacus_surface_b200 import config_type, canopy_flux_type, boundary_conds_out_type
    from spartacus_surface_b200._lib import load
    from spartacus_surface_b200.radsurf_interface import radsurf_fluxes, radsurf_fluxes_sp
    from spartacus_surface_b200.synthetic import make_synthetic
    if not torch.cuda.is_available():
        raise SystemExit("fluxes_device_sp.py needs a CUDA device")
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
    # NULL members as in bench.py's e2e block
    cp.veg_contact_fraction = None
    sw.air_ext = sw.air_ssa = sw.wall_specular_frac = sw.roof_albedo_dir = None
    lw.air_ext = lw.air_ssa = None
    for k in ("ground_emission", "roof_emission", "wall_emission", "clear_air_planck", "veg_planck", "veg_air_planck"):
        setattr(lw, k, None)
    # float32 inputs, and the float64 inputs of the twin: the same values widened
    single = [converted(o, lambda t: t.float().contiguous()) for o in (cp, sw, lw, temps, tops)]
    del cp, sw, lw, temps, tops, top_sw
    wide = [converted(o, lambda t: t.double().contiguous()) for o in single]
    flux = lambda d, dt: converted(canopy_flux_type().allocate(cfg, ncol, ntot, 1, use_direct=d,
                                                               do_save_flux_profile=args.profiles, device=dev),
                                   lambda t: t.to(dt).contiguous())
    bc_of = lambda dt: converted(boundary_conds_out_type().allocate(ncol, 1, 1, device=dev), lambda t: t.to(dt))
    d_out = [bc_of(torch.float64), flux(True, torch.float64), flux(False, torch.float64)]
    s_out = [bc_of(torch.float32), flux(True, torch.float32), flux(False, torch.float32)]
    stream = torch.cuda.current_stream().cuda_stream

    def arm_double():
        cp_, sw_, lw_, t_, f_ = wide
        assert radsurf_fluxes(cfg, cp_, sw_, lw_, d_out[0], None, None, d_out[1], d_out[2], stream=stream,
                              **f_, **t_) == 0

    def arm_single():
        cp_, sw_, lw_, t_, f_ = single
        assert radsurf_fluxes_sp(cfg, cp_, sw_, lw_, s_out[0], None, None, s_out[1], s_out[2], stream=stream,
                                 **f_, **t_) == 0

    arms = {
        "fluxes_device": dict(fn=arm_double, call="ssb200_radsurf_fluxes_device (float64)", caller=wide + d_out),
        "fluxes_device_sp": dict(fn=arm_single, call="ssb200_radsurf_fluxes_device_sp (float32)",
                                 caller=single + s_out),
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

    # bit-equality: float32 outputs against the float64 outputs cast to float32, on a seeded column sample
    cp_w = wide[0]
    seed = 20261021
    cols = np.sort(np.random.default_rng(seed).choice(ncol, size=min(args.sample, ncol), replace=False))
    rows = np.concatenate([np.arange(cp_w.istartlay[c] - 1, cp_w.istartlay[c] - 1 + cp_w.nlay[c]) for c in cols])
    checked, bad = 0, []
    for name, x, y in zip(("bc", "sw_flux", "lw_flux"), d_out, s_out):
        for k, v in vars(x).items():
            if not hasattr(v, "cpu"):
                continue
            idx = torch.from_numpy(cols if v.shape[0] == ncol else rows).to(dev)
            p, q = v[idx].float(), getattr(y, k)[idx]
            checked += p.numel()
            if not torch.equal(p, q):
                bad.append(f"{name}.{k}")
    result = {"card": card(),
              "workload": {"ncol": ncol, "nlay": nlay, "nreg": 3, "streams": args.streams, "nsw": 1, "nlw": 1,
                           "flux_profiles": args.profiles, "null_members": "bench.py e2e pattern",
                           "reps": args.reps, "calls_per_rep": args.steps},
              "timing": "CUDA events on the launch stream per call; arrays resident in HBM (no PCIe)",
              "check": {"sample_columns": int(cols.size), "seed": seed, "values_compared": checked,
                        "sp_equals_double_cast": not bad, "mismatching_members": bad}}
    for tag, a in arms.items():
        result[tag] = dict(call=a["call"], caller_hbm_bytes=nbytes(a["caller"]), **stats(a["ms"]))
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "fluxes_device_sp.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("card", "check")}))
    for tag in arms:
        r = result[tag]
        print(tag, round(r["median_ms"], 2), "ms", f"[{r['min_ms']:.2f}, {r['max_ms']:.2f}]",
              f"caller HBM {r['caller_hbm_bytes'] / 1e9:.2f} GB")
    lib.ssb200_release()
    if bad:
        raise SystemExit("fluxes_device_sp outputs differ from the float64 entry cast to float32")


if __name__ == "__main__":
    main()
