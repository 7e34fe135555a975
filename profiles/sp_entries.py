"""Single-precision entries against their double-precision twins on the default synthetic workload
(1,048,576 columns x 16 layers, nreg 3, 2 streams, one SW and one LW interval), in one invocation:

  e2e     ssb200_radsurf_fluxes vs ssb200_radsurf_fluxes_sp: pinned host buffers, the NULL-member
          pattern of bench.py's e2e block (read_input's defaults and sigma T^4 evaluated on the device),
          host wall clock around calls that return with the outputs on the host;
  device  ssb200_radsurf_device on float64 vs ssb200_radsurf_device_sp on float32 tensors, CUDA events.

The two arms of each pair alternate, `--reps` repetitions of `--steps` calls each; median and spread
(min, max) of the per-call time are reported.  Both arms take the same values: the double arm's inputs
are the float32 inputs widened, so the check that every sampled sp output equals the double output cast
to float32 bit for bit runs on the timed results.  Bytes per step are computed from the shapes (as
bench.py does: every input array up, every output array down).  The card name and power limit are read
in the same run.  Writes <out>/sp_entries.json.

    python profiles/sp_entries.py --out <dir>
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (x.strip() for x in q.split(","))
        return {"name": name, "power_limit": power, "clocks_max_sm": clock}
    except (OSError, ValueError, subprocess.SubprocessError):
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "not read", "clocks_max_sm": "not read"}


def stats(ms):
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)),
            "per_call_ms": [round(float(x), 3) for x in ms]}


def real_members(objs):
    for o in objs:
        vals = o.values() if isinstance(o, dict) else vars(o).values()
        for v in vals:
            if isinstance(v, np.ndarray) and v.dtype.kind == "f":
                yield v


def nbytes(objs):
    seen, total = set(), 0
    for v in real_members(objs):
        if v.ctypes.data not in seen:
            seen.add(v.ctypes.data)
            total += v.nbytes
    return int(total)


def pinned(obj, dtype, keep):
    """Copy of an API object (or dict) whose real members are pinned host arrays of `dtype`."""
    import torch
    out = dict(obj) if isinstance(obj, dict) else copy.copy(obj)
    items = obj.items() if isinstance(obj, dict) else vars(obj).items()
    done = {}
    for k, v in items:
        if isinstance(v, np.ndarray) and v.dtype.kind == "f":
            if id(v) not in done:  # one array given for several members stays one array
                t = torch.from_numpy(np.ascontiguousarray(v.astype(dtype))).pin_memory()
                keep.append(t)
                done[id(v)] = t.numpy()
            if isinstance(out, dict):
                out[k] = done[id(v)]
            else:
                setattr(out, k, done[id(v)])
    return out


def on_device(obj, dtype):
    import torch
    out = copy.copy(obj)
    for k, v in vars(obj).items():
        if isinstance(v, np.ndarray) and v.dtype.kind == "f":
            setattr(out, k, torch.from_numpy(np.ascontiguousarray(v.astype(dtype))).cuda())
    return out


def compare_rows(a32, a64, cols, rows_of_cols, ncol):
    """Sampled rows of every member: sp equals double cast to float32 bit for bit."""
    n, bad = 0, []
    for k, v in vars(a32).items():
        if v is None or isinstance(v, (int, float)):
            continue
        x = v.cpu().numpy() if hasattr(v, "cpu") else v
        y = getattr(a64, k)
        y = y.cpu().numpy() if hasattr(y, "cpu") else y
        idx = cols if x.shape[0] == ncol else rows_of_cols
        xs, ys = x[idx], y[idx].astype(np.float32)
        n += xs.size
        if not np.array_equal(xs, ys):
            bad.append(k)
    return n, bad


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--ncol", type=int, default=1 << 20)
    ap.add_argument("--nlay", type=int, default=16)
    ap.add_argument("--streams", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=3, help="calls per repetition")
    ap.add_argument("--sample", type=int, default=65536, help="columns in the bit-equality sample")
    args = ap.parse_args()
    import torch
    from spartacus_surface_b200 import radsurf, config_type, canopy_flux_type, boundary_conds_out_type
    from spartacus_surface_b200._lib import load
    from spartacus_surface_b200.radsurf_interface import radsurf_fluxes, radsurf_fluxes_sp, radsurf_sp, to_single
    from spartacus_surface_b200.synthetic import make_synthetic, to_host
    if not torch.cuda.is_available():
        raise SystemExit("sp_entries.py needs a CUDA device")
    lib = load()
    lib.ssb200_set_device(0)
    ncol, nlay = args.ncol, args.nlay
    cfg = config_type(do_sw=True, do_lw=True, nsw=1, nlw=1, n_vegetation_region_urban=2, n_vegetation_region_forest=2,
                      n_stream_sw_urban=args.streams, n_stream_lw_urban=args.streams,
                      n_stream_sw_forest=args.streams, n_stream_lw_forest=args.streams).consolidate()
    cp, sw, lw, temps = make_synthetic(cfg, ncol, nlay, device="cuda:0", with_temperatures=True)
    cp, sw, lw = (to_single(to_host(o)) for o in (cp, sw, lw))  # the values both arms solve
    temps = {k: np.ascontiguousarray(v.cpu().numpy().astype(np.float32)) for k, v in temps.items()}
    temps["veg_temperature"] = temps["veg_air_temperature"] = temps["clear_air_temperature"]
    torch.cuda.empty_cache()
    rng = np.random.default_rng(7)
    top_sw = rng.uniform(200.0, 900.0, size=(ncol, 1))
    tops = {"top_flux_dn_sw": top_sw, "top_flux_dn_direct_sw": top_sw * rng.uniform(0.2, 0.9, size=(ncol, 1)),
            "top_flux_dn_lw": rng.uniform(250.0, 400.0, size=(ncol, 1))}
    tops = {k: v.astype(np.float32) for k, v in tops.items()}
    cols = np.sort(np.random.default_rng(20261020).choice(ncol, size=min(args.sample, ncol), replace=False))
    rows = np.concatenate([np.arange(cp.istartlay[c] - 1, cp.istartlay[c] - 1 + cp.nlay[c]) for c in cols])
    result = {"card": card(), "workload": {"ncol": ncol, "nlay": nlay, "nreg": 3, "streams": args.streams,
                                            "nsw": 1, "nlw": 1, "reps": args.reps, "calls_per_rep": args.steps},
              "check": {"sample_columns": int(cols.size), "seed": 20261020}}

    # ---- end to end, pinned host buffers ----------------------------------------------------------------
    cp2, sw2, lw2 = copy.copy(cp), copy.copy(sw), copy.copy(lw)
    cp2.veg_contact_fraction = None
    sw2.air_ext = sw2.air_ssa = sw2.wall_specular_frac = sw2.roof_albedo_dir = None
    lw2.air_ext = lw2.air_ssa = None
    for k in ("ground_emission", "roof_emission", "wall_emission", "clear_air_planck", "veg_planck", "veg_air_planck"):
        setattr(lw2, k, None)
    keep = []
    e2e = {}
    for tag, dtype, fn in (("double", np.float64, radsurf_fluxes), ("single", np.float32, radsurf_fluxes_sp)):
        ins = [pinned(o, dtype, keep) for o in (cp2, sw2, lw2, temps, tops)]
        bc = pinned(boundary_conds_out_type().allocate(ncol, 1, 1), dtype, keep)
        sfl = pinned(canopy_flux_type().allocate(cfg, ncol, cp.ntotlay, 1, use_direct=True, do_save_flux_profile=False),
                     dtype, keep)
        lfl = pinned(canopy_flux_type().allocate(cfg, ncol, cp.ntotlay, 1, use_direct=False, do_save_flux_profile=False),
                     dtype, keep)
        e2e[tag] = dict(fn=fn, ins=ins, outs=(bc, sfl, lfl), ms=[],
                        h2d=nbytes(ins), d2h=nbytes([bc, sfl, lfl]))

    def call_e2e(a):
        cp_, sw_, lw_, t_, top_ = a["ins"]
        bc, sfl, lfl = a["outs"]
        assert a["fn"](cfg, cp_, sw_, lw_, bc, None, None, sfl, lfl, **top_, **t_) == 0

    for a in e2e.values():
        call_e2e(a)  # warm-up: device mirrors, plan
    for _ in range(args.reps):
        for a in e2e.values():  # alternating arms
            t0 = time.perf_counter()
            for _ in range(args.steps):
                call_e2e(a)  # returns when the outputs are on the host
            a["ms"].append(1e3 * (time.perf_counter() - t0) / args.steps)
    checked, bad = 0, []
    for o32, o64 in zip(e2e["single"]["outs"], e2e["double"]["outs"]):
        n, b = compare_rows(o32, o64, cols, rows, ncol)
        checked, bad = checked + n, bad + b
    result["e2e"] = {tag: dict(call=("ssb200_radsurf_fluxes" if tag == "double" else "ssb200_radsurf_fluxes_sp"),
                               h2d_bytes_per_step=a["h2d"], d2h_bytes_per_step=a["d2h"], **stats(a["ms"]))
                     for tag, a in e2e.items()}
    result["e2e"]["timing"] = "host wall clock per call, pinned host buffers, calls return with outputs on the host"
    result["check"]["e2e"] = {"values_compared": checked, "bit_equal": not bad, "mismatching_members": bad}
    del e2e, keep
    lib.ssb200_release()

    # ---- device-resident ----------------------------------------------------------------------------------
    dev = {}
    for tag, dtype, fn in (("double", np.float64, radsurf), ("single", np.float32, radsurf_sp)):
        ins = [on_device(o, dtype) for o in (cp, sw, lw)]
        bc = boundary_conds_out_type().allocate(ncol, 1, 1)
        fl = [canopy_flux_type().allocate(cfg, ncol, cp.ntotlay, 1, use_direct=d, do_save_flux_profile=False)
              for d in (True, True, False, False)]
        size = np.dtype(dtype).itemsize  # (cp, sw, lw hold float32, the fresh outputs float64)
        host_bytes = nbytes([cp, sw, lw]) // 4 * size, nbytes([bc] + fl) // 8 * size
        dev[tag] = dict(fn=fn, ins=ins, outs=[on_device(o, dtype) for o in [bc] + fl], ms=[],
                        input_bytes=int(host_bytes[0]), output_bytes=int(host_bytes[1]))
    stream = torch.cuda.current_stream().cuda_stream

    def call_dev(a):
        o = a["outs"]
        assert a["fn"](cfg, *a["ins"], o[0], None, None, *o[1:], stream=stream) == 0

    for a in dev.values():
        call_dev(a)
    torch.cuda.synchronize()
    for _ in range(args.reps):
        for a in dev.values():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                call_dev(a)
            e1.record()
            torch.cuda.synchronize()
            a["ms"].append(e0.elapsed_time(e1) / args.steps)
    checked, bad = 0, []
    for o32, o64 in zip(dev["single"]["outs"], dev["double"]["outs"]):
        n, b = compare_rows(o32, o64, cols, rows, ncol)
        checked, bad = checked + n, bad + b
    result["device"] = {tag: dict(call=("ssb200_radsurf_device" if tag == "double" else "ssb200_radsurf_device_sp"),
                                  h2d_bytes_per_step=0, d2h_bytes_per_step=0,
                                  caller_input_bytes=a["input_bytes"], caller_output_bytes=a["output_bytes"],
                                  **stats(a["ms"]))
                        for tag, a in dev.items()}
    result["device"]["timing"] = "CUDA events on the launch stream per call; arrays resident in HBM (no PCIe)"
    result["check"]["device"] = {"values_compared": checked, "bit_equal": not bad, "mismatching_members": bad}
    result["check"]["bit_equal"] = result["check"]["e2e"]["bit_equal"] and result["check"]["device"]["bit_equal"]
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "sp_entries.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("card", "check")}))
    for part in ("e2e", "device"):
        print(part, {t: round(result[part][t]["median_ms"], 2) for t in ("double", "single")})
    if not result["check"]["bit_equal"]:
        raise SystemExit("single-precision outputs differ from the cast double outputs")


if __name__ == "__main__":
    main()
