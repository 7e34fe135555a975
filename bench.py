#!/usr/bin/env python
"""bench.py - throughput of the SPARTACUS-Surface solver hot path on B200.

Metric (BASELINE.json): column·g·layers / s, SW+LW, on the synthetic vegetated-urban canopy of
SURVEY.md §8(d): 1,048,576 columns x 16 layers, nreg = 3, one SW and one LW interval (g = 2),
FP64.  One "step" = one radsurf pass over all columns.  Columns are independent, so with N GPUs
the 1,048,576 columns are SHARDED into N contiguous blocks (SURVEY §8e: 131,072 per GPU at N = 8;
"scaling": "strong"), no collective in the path; `--weak` gives every rank its own 1,048,576
columns instead, and at N > 1 the default run reports that figure as the extra key `weak_scaling`.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--streams 2|4] [--columns C] [--weak]
  python bench.py --impl reference ...   # CPU oracle (restatement of the Fortran) on the host cores
  python bench.py --dump-outputs DIR ... # also write the outputs of the last timed step (see dump_outputs)

Prints ONE JSON line (rank 0).  Keys beyond the base contract:
  roofline          dominant kernel on the SURVEY §8(d) FP64 flop count (frac, frac_segment_aware),
                    its DRAM traffic from the committed ncu capture and traffic / algorithmic bytes;
                    roofline.whole_step = the same for the whole step
  e2e               the driver sequence of the reference (calc_simple_spectrum_lw, radsurf, scale, sum:
                    driver/spartacus_surface_driver.F90:206-261) through ssb200_radsurf_fluxes with
                    pinned HOST buffers; e2e.radsurf_only = plain ssb200_radsurf (all four normalised
                    flux objects returned to the host)
  parity_vs_truth   error of the GPU result against the oracle's _Float128 ground truth on a subsample,
                    beside the error of the reference's own FP64 arithmetic (tests/parity.py rule)
  extra.s4          the reference-default 4-stream configuration on a smaller column count
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NLAY = 16
FULL_COLUMNS = 1 << 20
UNIT = "column*g*layers/s"
METRIC = "column_g_layers_per_s_SW+LW"
# kernel families timed by the library (CUDA events on the launch stream); the last one holds the surface
# kernels (flat / single-layer tiles) and the gather / scatter passes of the level-major staging
FAMILIES = ["sw_layer", "sw_sweep", "lw_layer", "lw_sweep", "surface_and_staging"]
FLUX_NAMES = ("sw_norm_dir", "sw_norm_diff", "lw_internal", "lw_norm")

# Compulsory HBM bytes per (column, layer): 25 input + 40 output doubles + per-column terms (SURVEY §8d)
ALGO_BYTES_PER_COL_LAYER = 540.0


# Algorithmic FLOPs per (column, layer) (SURVEY.md section 8d / App. C closed form).  "full": every layer
# charged the full-size (nreg = 3) count, the agreed numerator of SURVEY 8d; "seg": layers that solve only
# a sub-block of their regions (no vegetation in the layer: clear region only) charged with the order they
# actually solve - the reference does the same - while the sweeps stay full size.
def _layer_flops(n, d):
    N = 2 * n + d
    sw = 25 * n**3 + (38.67 + 8 * d) * n**3 + 2 / 3 * N**3 + 2 * N * N * d + 4 * n * N * d + 8 * d * n * n
    lw = 25 * n**3 + 34.67 * n**3 + 16 * n * n
    return sw, lw


def flop_table(ns, f_full, f_clear, f_veg):
    """per (column, layer): kernel family -> (flops "full" count, flops segment-aware)"""
    n, d, m = 3 * ns, 3, 4 * ns
    sw_full, lw_full = _layer_flops(n, d)
    sw_c, lw_c = _layer_flops(ns, 1)
    sw_v, lw_v = _layer_flops(2 * ns, 2)
    sw_sweep = 10.67 * n**3 + 22 * n * n + 4 * m * m + 6 * n * n * d
    lw_sweep = 10.67 * n**3 + 26 * n * n + 4 * m * m
    return {"sw_layer": (sw_full, f_full * sw_full + f_clear * sw_c + f_veg * sw_v),
            "lw_layer": (lw_full, f_full * lw_full + f_clear * lw_c + f_veg * lw_v),
            "sw_sweep": (sw_sweep, sw_sweep), "lw_sweep": (lw_sweep, lw_sweep)}


def make_config(streams):
    from spartacus_surface_b200 import config_type
    cfg = config_type(do_sw=True, do_lw=True, nsw=1, nlw=1, n_vegetation_region_urban=2,
                      n_vegetation_region_forest=2, n_stream_sw_urban=streams, n_stream_lw_urban=streams,
                      n_stream_sw_forest=streams, n_stream_lw_forest=streams)
    return cfg


def allocate_outputs(cfg, ncol, ntotlay, device=None):
    from spartacus_surface_b200 import canopy_flux_type, boundary_conds_out_type
    bc = boundary_conds_out_type().allocate(ncol, 1, 1, device=device)
    fl = [canopy_flux_type().allocate(cfg, ncol, ntotlay, 1, use_direct=d, do_save_flux_profile=False, device=device)
          for d in (True, True, False, False)]
    return bc, fl


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t_begin=None, t_end=None):
        """Median SM clock and throttle reasons of the samples that arrived in [t_begin, t_end]
        (the timed region); if the region was too short to catch one, of the samples since the
        sampler started (it starts before the warm-up steps, so those are under the same load)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [r for t, r in self.rows if t_begin is None or t_begin <= t <= (t_end or t) + 0.15]
        window = "timed region" if inside else "warm-up and timed region"
        for r in (inside or [r for _, r in self.rows]):
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


def host_threads():
    """Host cores this process may use (torchrun sets OMP_NUM_THREADS=1: ask the scheduler instead)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def bind_near_gpu(index):
    """Run this rank's host side (pinned staging buffers are first-touched by it) on the cores of the
    GPU's own NUMA node.  Returns (description, previous affinity to restore)."""
    try:
        prev = os.sched_getaffinity(0)
    except AttributeError:
        return "unchanged (no sched_getaffinity)", None
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        near = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        want = near & prev
        if want and want != prev:
            os.sched_setaffinity(0, want)
            return f"{len(want)} cores of the GPU's NUMA node (of {len(prev)} allowed)", prev
        return f"unchanged: the {len(prev)} allowed cores are all on the GPU's NUMA node", prev
    except Exception as exc:  # noqa: BLE001 - affinity is an optimisation only
        return f"unchanged ({type(exc).__name__})", prev


def workload_config(args, total_columns, world, per_gpu, weak):
    shard = (f"every GPU its own {per_gpu} columns" if weak else
             f"sharded over {world} GPU(s) in contiguous column blocks ({per_gpu} per GPU)")
    return {"workload": f"synthetic vegetated-urban canopy, {total_columns} columns x {NLAY} layers x (1 SW + 1 LW) "
                        f"intervals, nreg=3, {args.streams} streams per hemisphere, {shard}",
            "columns_total": total_columns, "columns_per_gpu": per_gpu, "layers": NLAY, "streams": args.streams,
            "nreg": 3, "parallelism": "independent column shards, no collective",
            "l2": "inputs + outputs + scratch of one step (> 1 GB even at 131072 columns per GPU) exceed the "
                  "126 MB L2; no flush needed"}


def run_reference(args, rank, world):
    """CPU arm: the oracle (C++ restatement of the Fortran solver; the Fortran itself cannot be
    built: no Fortran compiler in the image) on all host threads, bounded sample per step."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    from spartacus_surface_b200.synthetic import make_synthetic
    cfg = make_config(args.streams).consolidate(oracle_lib.legendre_gauss_init)
    ncol = args.cpu_columns
    cp, sw, lw = make_synthetic(cfg, ncol, NLAY)
    bc, fl = allocate_outputs(cfg, ncol, cp.ntotlay)
    threads = host_threads()
    solver = oracle_lib.make_solver(nthreads=threads, nblocksize=16)
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        rc = solver(cfg, cp, sw, lw, bc, None, None, *fl)
        dt = time.perf_counter() - t0
        assert rc == 0
        if it >= args.warmup:
            times.append(dt)
    units = ncol * NLAY * 2
    total = sum(times)
    value = units * len(times) / total
    sample = (f"each step solves the first {ncol} of the {args.columns} synthetic columns (same generator and seed; "
              f"columns are independent, throughput is per unit), OpenMP blocks of 16 columns")
    conf = workload_config(args, args.columns, 1, args.columns, False)
    conf["workload"] += f"; CPU arm: bounded sample of {ncol} columns per step"
    conf["columns_solved_per_step"] = ncol
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": conf,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def head_to_host(obj, nc, ncol):
    """Host copy of the first `nc` columns of an API object whose double members live on the device."""
    import copy
    import numpy as np
    out = copy.copy(obj)
    for k, v in vars(obj).items():
        if type(v).__module__.startswith("torch"):
            rows = nc if v.shape[0] == ncol else nc * NLAY
            setattr(out, k, np.ascontiguousarray(v[:rows].cpu().numpy()))
        elif isinstance(v, np.ndarray) and v.shape and v.shape[0] == ncol:
            setattr(out, k, np.ascontiguousarray(v[:nc]))
    if hasattr(out, "ncol"):
        out.ncol, out.ntotlay = nc, nc * NLAY
    return out


def fields_of(fl, rows_col=None, ncol=None):
    """{object: {field: numpy}} of four flux objects (torch or numpy members), first rows_col columns."""
    import numpy as np
    from spartacus_surface_b200.radsurf_canopy_flux import ALL_FIELDS
    out = {}
    for n, f in zip(FLUX_NAMES, fl):
        d = {}
        for k in ALL_FIELDS:
            v = getattr(f, k)
            if v is None:
                continue
            if rows_col is not None:
                v = v[:rows_col * (NLAY if v.shape[0] != ncol else 1)]
            d[k] = v.cpu().numpy() if type(v).__module__.startswith("torch") else np.asarray(v)
        out[n] = d
    return out


class Solve:
    """One device-resident problem: inputs, outputs and the timed step."""

    def __init__(self, lib, streams, ncol, col_offset, device):
        import torch
        from spartacus_surface_b200.synthetic import make_synthetic
        self.lib, self.ncol, self.device = lib, ncol, device
        self.cfg = make_config(streams).consolidate()
        self.cp, self.sw, self.lw, self.temps = make_synthetic(self.cfg, ncol, NLAY, col_offset=col_offset,
                                                                device=device, with_temperatures=True)
        self.bc, self.fl = allocate_outputs(self.cfg, ncol, self.cp.ntotlay, device=device)
        self.stream = torch.cuda.current_stream().cuda_stream

    def step(self):
        from spartacus_surface_b200 import radsurf
        rc = radsurf(self.cfg, self.cp, self.sw, self.lw, self.bc, None, None, *self.fl, stream=self.stream)
        assert rc == 0, rc

    def timed(self, steps, warmup, barrier, all_max, sampler=None):
        """W warm-up steps, then K steps between barrier + synchronize; CUDA events on the launch
        stream; max over ranks.  Returns (ms for the K steps, launches, clocks)."""
        import torch
        for _ in range(warmup):
            self.step()
        barrier()
        launches0 = self.lib.ssb200_kernel_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_begin = time.time()
        e0.record()
        for _ in range(steps):
            self.step()
        e1.record()
        torch.cuda.synchronize()
        t_end = time.time()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop(t_begin, t_end) if sampler else None
        launches = self.lib.ssb200_kernel_launch_count() - launches0
        barrier()
        return all_max(ms), int(launches), clocks

    def kernel_times(self):
        """Per kernel family: launch durations of ONE step, CUDA events on the launch stream (library)."""
        import torch
        self.lib.ssb200_set_profiling(1)
        for _ in range(2):  # (the first profiled step may grow a scratch buffer: passes run serially here)
            self.step()
            torch.cuda.synchronize()
        tms, cnt = (C.c_double * 5)(), (C.c_int64 * 5)()
        self.lib.ssb200_last_kernel_times_ms(tms)
        self.lib.ssb200_last_kernel_counts(cnt)
        self.lib.ssb200_set_profiling(0)
        return {FAMILIES[i]: {"ms": tms[i], "launches": int(cnt[i])} for i in range(5)}

    def segment_mix(self):
        vfr, bfr = self.cp.veg_fraction, self.cp.building_fraction
        min_veg = self.cfg.min_vegetation_fraction
        f_clear = float((vfr <= min_veg).double().mean().item())
        f_veg = float(((vfr > min_veg) & ((1.0 - bfr - vfr) <= min_veg)).double().mean().item())
        return 1.0 - f_clear - f_veg, f_clear, f_veg

    def residuals(self):
        import torch
        res = {}
        for name, f in zip(FLUX_NAMES, self.fl):
            r = torch.zeros(self.ncol, dtype=torch.float64, device=self.device)
            s, cps = f.as_struct(), self.cp.as_struct()
            rc = self.lib.ssb200_canopy_flux_check_device(C.byref(s), C.byref(cps), C.c_void_p(r.data_ptr()), None)
            assert rc == 0, rc
            torch.cuda.synchronize()
            denom = (f.top_dn if name != "lw_internal" else f.top_net)[:, 0].abs().clamp_min(1e-30)
            res[name] = float((r.abs() / denom).max().item())
        nonfinite = int(sum((~torch.isfinite(getattr(f, k))).sum().item() for f in self.fl
                            for k in ("ground_net", "top_net", "clear_air_abs", "veg_abs", "wall_net", "roof_net")))
        return res, nonfinite

    def parity_vs_truth(self, ncols, threads):
        """GPU result of the first `ncols` columns against the oracle's _Float128 build on the same
        inputs, beside the two FP64 builds of the oracle (tests/parity.py rule)."""
        import numpy as np
        import oracle_lib
        import parity
        ns_ = min(ncols, self.ncol)
        scp, ssw, slw = (head_to_host(o, ns_, self.ncol) for o in (self.cp, self.sw, self.lw))
        outs = []
        for kw in ({"quad": True}, {}, {"nofma": True}):
            sbc, sfl = allocate_outputs(self.cfg, ns_, scp.ntotlay)
            oracle_lib.make_solver(nthreads=threads, **kw)(self.cfg, scp, ssw, slw, sbc, None, None, *sfl)
            outs.append(fields_of(sfl))
        got = fields_of(self.fl, ns_, self.ncol)
        ok, worst, lines = parity.check(got, outs[0], outs[1], outs[2])
        summ = parity.summary(got, outs[0], outs[1], outs[2])
        # elementwise relative error of every flux-scale field (the north_star's measure)
        elem_gpu = elem_ref = 0.0
        for n in outs[0]:
            for k in parity.SCALE_FIELDS:
                if k in outs[0][n]:
                    t = outs[0][n][k]
                    den = np.maximum(np.abs(t), 1e-300)
                    elem_gpu = max(elem_gpu, float((np.abs(got[n][k] - t) / den).max()))
                    elem_ref = max(elem_ref, float((np.abs(outs[1][n][k] - t) / den).max()))
        return {"within_rule": bool(ok), "rule": "err(gpu, truth) <= max(1e-9, 2 err(reference_fp64, truth)) per field "
                                                 "(tests/parity.py)",
                "columns": ns_, "truth": "oracle built with _Float128 scalars (oracle/_build/liboracle_quad.so)",
                "err_gpu_vs_truth": summ["err_gpu"], "err_gpu_field": summ["err_gpu_field"],
                "err_reference_fp64_vs_truth": summ["err_ref_fp64"], "worst_err_over_bound": worst,
                "fields_above_1e-9": summ["fields_above_1e-9"], "violations": lines[:4],
                "elementwise_rel_err_flux_fields": {"gpu": elem_gpu, "reference_fp64": elem_ref}}


DUMP_COLUMNS = 8192       # 5.4 KB of outputs per column: 44 MB in all
DUMP_LIMIT_BYTES = 64 << 20
DUMP_SEED = 20190605


def dump_outputs(prob, out_dir):
    """Write what the last step returned to its caller - bc_out and the four normalised flux
    objects - as out_dir/<object>.<field>.npy (float64, the solver's type).  Every member is
    restricted to the same fixed, seeded sample of min(DUMP_COLUMNS, ncol) columns (all layers of
    each), in column order.  The synthetic inputs are a pure function of the column index, so two
    builds run with the same arguments can be compared output for output."""
    import numpy as np
    import torch
    from spartacus_surface_b200.radsurf_canopy_flux import ALL_FIELDS
    n = min(DUMP_COLUMNS, prob.ncol)
    cols = np.sort(np.random.default_rng(DUMP_SEED).choice(prob.ncol, n, replace=False))
    col_idx = torch.from_numpy(cols).to(prob.device)
    lay_idx = (col_idx[:, None] * NLAY + torch.arange(NLAY, device=prob.device)[None, :]).reshape(-1)
    members = [("bc", k, getattr(prob.bc, k)) for k in ("sw_albedo", "sw_albedo_dir", "lw_emissivity", "lw_emission")]
    members += [(name, k, getattr(f, k)) for name, f in zip(FLUX_NAMES, prob.fl) for k in ALL_FIELDS]
    arrays = {}
    for name, k, v in members:
        if v is None:
            continue
        assert v.shape[0] in (prob.ncol, prob.ncol * NLAY), (name, k, tuple(v.shape))
        idx = col_idx if v.shape[0] == prob.ncol else lay_idx
        arrays[f"{name}.{k}"] = v.index_select(0, idx).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, total
    os.makedirs(out_dir, exist_ok=True)
    for key, a in arrays.items():
        np.save(os.path.join(out_dir, key + ".npy"), a)


def pinned_copy(obj, pin):
    """numpy view of pinned copies of every float64 member."""
    import numpy as np
    import torch
    for k, v in list(vars(obj).items()):
        if isinstance(v, np.ndarray) and v.dtype == np.float64:
            tt = torch.from_numpy(v).pin_memory()
            pin.append(tt)
            setattr(obj, k, tt.numpy())
    return obj


def nbytes(*objs):
    import numpy as np
    seen, total = set(), 0
    for obj in objs:
        vals = obj.values() if isinstance(obj, dict) else vars(obj).values()
        for v in vals:
            if isinstance(v, np.ndarray) and v.dtype == np.float64 and v.ctypes.data not in seen:
                seen.add(v.ctypes.data)
                total += v.nbytes
    return total


def run_e2e(prob, steps, barrier, all_max, world, gpu_index):
    """End to end with pinned HOST buffers on every rank at once.  Primary: the reference driver's
    sequence in one call (ssb200_radsurf_fluxes: only inputs that carry information go up, only the
    two summed flux objects come down).  Secondary: plain ssb200_radsurf."""
    import copy
    import numpy as np
    import torch
    from spartacus_surface_b200 import radsurf, canopy_flux_type, boundary_conds_out_type
    from spartacus_surface_b200.radsurf_interface import radsurf_fluxes
    from spartacus_surface_b200.synthetic import to_host
    affinity, prev = bind_near_gpu(gpu_index)
    cfg, ncol = prob.cfg, prob.ncol
    units = ncol * NLAY * 2
    pin = []
    hcp, hsw, hlw = (pinned_copy(to_host(o), pin) for o in (prob.cp, prob.sw, prob.lw))
    out = {}
    # ---- driver sequence ------------------------------------------------------------------------
    temps = {k: v.cpu().numpy() for k, v in prob.temps.items() if k in ("ground_temperature", "roof_temperature",
                                                                         "wall_temperature", "clear_air_temperature")}
    temps = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in temps.items()}
    pin.extend(temps.values())
    temps = {k: v.numpy() for k, v in temps.items()}
    temps["veg_temperature"] = temps["veg_air_temperature"] = temps["clear_air_temperature"]
    rng = np.random.default_rng(7)
    tops = {"top_flux_dn_sw": rng.uniform(200.0, 900.0, size=(ncol, 1))}
    tops["top_flux_dn_direct_sw"] = tops["top_flux_dn_sw"] * rng.uniform(0.2, 0.9, size=(ncol, 1))
    tops["top_flux_dn_lw"] = rng.uniform(250.0, 400.0, size=(ncol, 1))
    tops = {k: torch.from_numpy(v).pin_memory() for k, v in tops.items()}
    pin.extend(tops.values())
    tops = {k: v.numpy() for k, v in tops.items()}
    cp2, sw2, lw2 = copy.copy(hcp), copy.copy(hsw), copy.copy(hlw)
    cp2.veg_contact_fraction = None  # read_input's default, evaluated on the device
    sw2.air_ext = sw2.air_ssa = sw2.wall_specular_frac = sw2.roof_albedo_dir = None
    lw2.air_ext = lw2.air_ssa = None
    for k in ("ground_emission", "roof_emission", "wall_emission", "clear_air_planck", "veg_planck", "veg_air_planck"):
        setattr(lw2, k, None)
    bc2 = pinned_copy(boundary_conds_out_type().allocate(ncol, 1, 1), pin)
    sw_flux = pinned_copy(canopy_flux_type().allocate(cfg, ncol, hcp.ntotlay, 1, use_direct=True,
                                                      do_save_flux_profile=False), pin)
    lw_flux = pinned_copy(canopy_flux_type().allocate(cfg, ncol, hcp.ntotlay, 1, use_direct=False,
                                                      do_save_flux_profile=False), pin)

    def fluxes():
        rc = radsurf_fluxes(cfg, cp2, sw2, lw2, bc2, None, None, sw_flux, lw_flux, **tops, **temps)
        assert rc == 0, rc

    fluxes()  # warm-up (allocates the device mirrors)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        fluxes()  # returns when the outputs are on the host
    dt = all_max(time.perf_counter() - t0)
    h2d = nbytes(cp2, sw2, lw2, temps, tops)
    d2h = nbytes(bc2, sw_flux, lw_flux)
    out = {"value": world * units * steps / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d) * world,
           "d2h_bytes_per_step": int(d2h) * world, "ms_per_step": 1e3 * dt / steps,
           "call": "ssb200_radsurf_fluxes: the reference driver's sequence for a block of columns "
                   "(calc_simple_spectrum_lw, radsurf, scale by the top-of-canopy fluxes, sum) in one call; pinned "
                   "host arrays on every rank at once; H2D of every input that carries information (read_input's "
                   "constant defaults and sigma T^4 are evaluated on the device), kernels, D2H of bc_out and of the "
                   "two summed flux objects; host wall clock, max over ranks; bytes summed over ranks",
           "host_affinity": affinity}
    # the summed fluxes equal scale + sum of the device-resident normalised result (same kernels)
    f0, f1 = prob.fl[0], prob.fl[1]
    nchk = min(4096, ncol)
    ref = (f0.top_net[:nchk, 0].cpu().numpy() * tops["top_flux_dn_direct_sw"][:nchk, 0]
           + f1.top_net[:nchk, 0].cpu().numpy() * (tops["top_flux_dn_sw"][:nchk, 0] - tops["top_flux_dn_direct_sw"][:nchk, 0]))
    assert np.allclose(ref, sw_flux.top_net[:nchk, 0], rtol=1e-13, atol=0.0), "device and host entry disagree"
    del bc2, sw_flux, lw_flux
    # ---- plain drop-in entry ------------------------------------------------------------------------
    hbc, hfl = allocate_outputs(cfg, ncol, hcp.ntotlay)
    for obj in [hbc] + hfl:
        pinned_copy(obj, pin)
    radsurf(cfg, hcp, hsw, hlw, hbc, None, None, *hfl)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        rc = radsurf(cfg, hcp, hsw, hlw, hbc, None, None, *hfl)
        assert rc == 0
    dt = all_max(time.perf_counter() - t0)
    out["radsurf_only"] = {"value": world * units * steps / dt, "unit": UNIT,
                           "h2d_bytes_per_step": int(nbytes(hcp, hsw, hlw)) * world,
                           "d2h_bytes_per_step": int(nbytes(hbc, *hfl)) * world, "ms_per_step": 1e3 * dt / steps,
                           "call": "ssb200_radsurf: every input array up, all four normalised flux objects down"}
    dev_top = prob.fl[0].top_net[:nchk, 0].cpu().numpy()
    assert np.array_equal(dev_top, hfl[0].top_net[:nchk, 0]), "device and host entry disagree"
    if prev is not None:
        os.sched_setaffinity(0, prev)
    return out


def load_profile_json(name):
    try:
        return json.load(open(os.path.join(ROOT, "profiles", name)))
    except (OSError, ValueError):
        return {}


def roofline_report(prob, kt, step_ms, streams, fp64_peak, hbm_peak, peaks_present):
    """SURVEY §8(d): FP64 roofline on the algorithmic flop count, per kernel family and whole step."""
    ncol = prob.ncol
    f_full, f_clear, f_veg = prob.segment_mix()
    fl_tab = flop_table(streams, f_full, f_clear, f_veg)
    traffic_tab = load_profile_json("r02_dram_traffic.json") or load_profile_json("r01_dram_traffic.json")
    traffic_file = "profiles/r02_dram_traffic.json" if load_profile_json("r02_dram_traffic.json") else \
        "profiles/r01_dram_traffic.json"
    total_flops = sum(v[0] for v in fl_tab.values())
    kernels = {}
    for k in ("sw_layer", "lw_layer", "sw_sweep", "lw_sweep"):
        if kt[k]["launches"] == 0 or kt[k]["ms"] <= 0.0:
            continue
        n_l = kt[k]["launches"]
        per_ms = kt[k]["ms"] / n_l
        units = ncol * NLAY / n_l  # (column, layer) pairs of one launch (one chunk of columns)
        tf_full = fl_tab[k][0] * units / (per_ms * 1e-3) / 1e12
        tf_seg = fl_tab[k][1] * units / (per_ms * 1e-3) / 1e12
        tr = traffic_tab.get(f"{k}_s{streams}")
        # the compulsory 540 B per (column, layer) of the whole path, apportioned by algorithmic flops
        algo_bytes = ALGO_BYTES_PER_COL_LAYER * fl_tab[k][0] / total_flops
        ent = {"avg_launch_ms": per_ms, "launches_per_step": n_l, "column_layers_per_launch": units,
               "algorithmic_flops_per_column_layer": fl_tab[k][0],
               "algorithmic_flops_per_column_layer_segment_aware": fl_tab[k][1],
               "fp64_tflops": tf_full, "fp64_frac": tf_full / fp64_peak, "fp64_frac_segment_aware": tf_seg / fp64_peak,
               "share_of_step": kt[k]["ms"] / sum(kt[f]["ms"] for f in FAMILIES),
               "traffic": tr["dram_bytes_per_column_layer"] * units if tr else None,
               "dram_bytes_per_column_layer_ncu": tr["dram_bytes_per_column_layer"] if tr else None,
               "dram_gbs": tr["dram_bytes_per_column_layer"] * units / (per_ms * 1e-3) / 1e9 if tr else None}
        if tr:
            ent["dram_frac_of_hbm_peak"] = ent["dram_gbs"] / hbm_peak
            ent["traffic_over_algorithmic"] = tr["dram_bytes_per_column_layer"] / algo_bytes
        kernels[k] = ent
    dom = max(kernels, key=lambda k: kt[k]["ms"])
    e = kernels[dom]
    all_full = total_flops * ncol * NLAY
    all_seg = sum(v[1] for v in fl_tab.values()) * ncol * NLAY
    traffic_all = sum(kernels[k]["dram_bytes_per_column_layer_ncu"] or 0.0 for k in kernels)
    roofline = {
        "bound": "fp64", "kernel": dom, "achieved": e["fp64_tflops"], "peak": fp64_peak, "unit": "TFLOP/s",
        "frac": e["fp64_frac"], "frac_segment_aware": e["fp64_frac_segment_aware"], "traffic": e["traffic"],
        "traffic_over_algorithmic": e.get("traffic_over_algorithmic"),
        "avg_launch_ms": e["avg_launch_ms"], "launches_per_step": e["launches_per_step"],
        "flops_note": "achieved = SURVEY 8(d) algorithmic flops per (column, layer) of this kernel family x pairs per "
                      "launch / average launch duration (CUDA events on the launch stream); SURVEY charges every layer "
                      "the full nreg=3 count - frac_segment_aware charges layers without vegetation the order they "
                      "solve; traffic = ncu dram bytes per launch; traffic_over_algorithmic: against this family's "
                      "share (by flops) of the compulsory 540 B per (column, layer)",
        "segment_mix": {"all_regions": f_full, "clear_only": f_clear, "vegetated_only": f_veg},
        "fp64_peak_source": "measured in this run: register-resident independent DFMA chains on all SMs "
                            "(ssb200_measure_fp64_peak_tflops; profiles/r02_fp64_peak.json holds a tracked copy); "
                            "MEASURED_PEAKS.json has no FP64 entry",
        "hbm_peak": hbm_peak, "hbm_peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks_present else "fallback 6650 GB/s",
        "traffic_source": f"{traffic_file} (ncu --set full dram__bytes_read+write per kernel family, scaled to the launch)",
        "whole_step": {"bound": "fp64", "achieved": all_full / (step_ms * 1e-3) / 1e12,
                       "frac": all_full / (step_ms * 1e-3) / 1e12 / fp64_peak,
                       "frac_segment_aware": all_seg / (step_ms * 1e-3) / 1e12 / fp64_peak,
                       "algorithmic_flops_per_column_layer": total_flops,
                       "algorithmic_bytes_per_column_layer": ALGO_BYTES_PER_COL_LAYER,
                       "dram_bytes_per_column_layer_ncu": traffic_all or None,
                       "traffic_over_algorithmic": traffic_all / ALGO_BYTES_PER_COL_LAYER if traffic_all else None,
                       "hbm_frac_on_algorithmic_bytes": ALGO_BYTES_PER_COL_LAYER * ncol * NLAY / (step_ms * 1e-3) / 1e9
                       / hbm_peak,
                       "note": "SURVEY 8(d) flop count of the reference formulation / step time"},
    }
    return roofline, kernels


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=2, choices=[1, 2, 3, 4, 8])
    ap.add_argument("--columns", type=int, default=FULL_COLUMNS, help="columns of the whole job")
    ap.add_argument("--weak", action="store_true", help="every rank solves --columns columns of its own")
    ap.add_argument("--cpu-columns", type=int, default=131072, help="columns of the bounded CPU sample")
    ap.add_argument("--truth-columns", type=int, default=256, help="columns checked against the _Float128 oracle")
    ap.add_argument("--s4-columns", type=int, default=131072, help="columns of the 4-stream secondary (0: skip)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-weak-extra", action="store_true", help="N > 1: skip the extra weak-scaling measurement")
    ap.add_argument("--generic", action="store_true", help="force the generic kernels (test-only path)")
    ap.add_argument("--opt", action="append", default=[], help="tuning: name=value passed to ssb200_set_option")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one for a fixed sample of columns "
                         "(of rank 0) as DIR/<object>.<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    from spartacus_surface_b200._lib import load

    lib = load()
    if not torch.cuda.is_available() or lib.ssb200_device_count() <= 0:
        raise SystemExit("bench.py needs a CUDA device: the solver has no CPU fallback")
    torch.cuda.set_device(local_rank)
    lib.ssb200_set_device(local_rank)
    device = torch.device("cuda", local_rank)
    # stdout carries exactly one JSON line: whatever libraries print there (the NCCL version
    # banner under torchrun) goes to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    if args.generic:
        lib.ssb200_set_option(b"fast_kernels", 0)
    for kv in args.opt:
        k, v = kv.split("=")
        assert lib.ssb200_set_option(k.encode(), int(v)) == 0, kv

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- the measured problem: `columns` sharded over the ranks (strong) or per rank (weak) ----------
    from spartacus_surface_b200.sharding import shard_columns
    import numpy as np
    if args.weak:
        col0, ncol = rank * args.columns, args.columns
        total_columns = world * args.columns
    else:
        c0, c1 = shard_columns(np.full(args.columns, NLAY), world)[rank]
        col0, ncol = c0, c1 - c0
        total_columns = args.columns
    prob = Solve(lib, args.streams, ncol, col0, device)
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_max, launches, clocks = prob.timed(args.steps, args.warmup, barrier, all_max, sampler)
    if args.dump_outputs and rank == 0:
        dump_outputs(prob, args.dump_outputs)
    value = total_columns * NLAY * 2 * args.steps / (ms_max * 1e-3)
    step_ms = ms_max / args.steps
    res, nonfinite = prob.residuals()

    e2e = run_e2e(prob, args.e2e_steps, barrier, all_max, world, local_rank) if args.e2e_steps > 0 else None

    # ---- N > 1: the weak-scaling figure beside the sharded one ------------------------------------
    weak = None
    if world > 1 and not args.weak and not args.no_weak_extra:
        del prob
        torch.cuda.empty_cache()
        wprob = Solve(lib, args.streams, args.columns, rank * args.columns, device)
        wms, _, _ = wprob.timed(args.steps, args.warmup, barrier, all_max)
        weak = {"value": world * args.columns * NLAY * 2 * args.steps / (wms * 1e-3), "unit": UNIT,
                "ms_per_step": wms / args.steps, "columns_per_gpu": args.columns,
                "note": "every rank solves its own full-size problem (the round-1 measurement)"}
        prob = wprob if rank == 0 else None
        if rank != 0:
            del wprob

    out = None
    if rank == 0:
        kt = prob.kernel_times()
        fp64_peak = lib.ssb200_measure_fp64_peak_tflops(1 << 15)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        kstep_ms = step_ms if weak is None else weak["ms_per_step"]
        roofline, roofline_kernels = roofline_report(prob, kt, kstep_ms, args.streams, fp64_peak, hbm_peak, bool(peaks))
        if weak is not None:
            roofline["note"] = "per-kernel times and roofline taken on the full-size (weak) problem of rank 0"
        fp64_rec = load_profile_json("r02_fp64_peak.json")

        # ---- CPU baseline beside it (oracle on the host cores, bounded sample) and parity -----------
        cpu = parity_truth = parity_sample = flops_measured = None
        if not args.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib
            import parity
            nc = min(args.cpu_columns, prob.ncol)
            ccp, csw, clw = (head_to_host(o, nc, prob.ncol) for o in (prob.cp, prob.sw, prob.lw))
            cbc, cfl = allocate_outputs(prob.cfg, nc, ccp.ntotlay)
            cpu_threads = host_threads()
            solver = oracle_lib.make_solver(nthreads=cpu_threads)
            solver(prob.cfg, ccp, csw, clw, cbc, None, 256, *cfl)  # touch pages / warm caches
            t0 = time.perf_counter()
            rc = solver(prob.cfg, ccp, csw, clw, cbc, None, None, *cfl)
            dt = time.perf_counter() - t0
            assert rc == 0
            cpu = {"value": nc * NLAY * 2 / dt, "unit": UNIT, "cores": cpu_threads, "kind": "port",
                   "sample": f"first {nc} of the {prob.ncol} columns of rank 0, one pass, OpenMP dynamic blocks of 16 "
                             f"columns ({dt:.1f} s); C++ restatement of the reference (no Fortran compiler in the image)"}
            errs = parity.field_errors(fields_of(prob.fl, nc, prob.ncol), fields_of(cfl))
            parity_sample = {"columns": nc, "against": "FP64 oracle (not the truth: carries the reference's own rounding)",
                             "max_err_fluxes": max(v for k, v in errs.items() if "sunlit" not in k[1]),
                             "max_err_sunlit_fractions": max([v for k, v in errs.items() if "sunlit" in k[1]] or [0.0]),
                             "measure": "tests/parity.py field_errors"}
            parity_truth = prob.parity_vs_truth(args.truth_columns, cpu_threads)
            # instrumented flop counter of the oracle next to the closed form (SURVEY App. C)
            olib = oracle_lib.load()
            nf = min(2048, nc)
            olib.oracle_flops_enable(1)
            solver(prob.cfg, ccp, csw, clw, cbc, None, nf, *cfl)
            flops_measured = {"per_column_layer": olib.oracle_flops_read() / (nf * NLAY),
                              "closed_form_full": roofline["whole_step"]["algorithmic_flops_per_column_layer"],
                              "closed_form_segment_aware": sum(v[1] for v in flop_table(args.streams, *prob.segment_mix()).values()),
                              "columns": nf,
                              "note": "counted in the oracle's radtool routines while solving the first columns (the "
                                      "reference skips the vegetated regions of layers without vegetation, so compare "
                                      "with the segment-aware closed form)"}
            olib.oracle_flops_enable(0)

        # ---- secondary: the reference-default 4 streams --------------------------------------------
        extra = {}
        if args.s4_columns > 0 and args.streams != 4 and world == 1:
            ncol_total = prob.ncol
            del prob
            torch.cuda.empty_cache()
            p4 = Solve(lib, 4, args.s4_columns, 0, device)
            ms4, l4, _ = p4.timed(max(2, min(args.steps, 3)), 3, barrier, all_max)
            k4 = max(2, min(args.steps, 3))
            kt4 = p4.kernel_times()
            r4, rk4 = roofline_report(p4, kt4, ms4 / k4, 4, fp64_peak, hbm_peak, bool(peaks))
            res4, nonfinite4 = p4.residuals()
            s4 = {"value": args.s4_columns * NLAY * 2 * k4 / (ms4 * 1e-3), "unit": UNIT, "ms_per_step": ms4 / k4,
                  "columns": args.s4_columns, "steps": k4, "warmup": 3, "gpu_launches": l4,
                  "config": "same synthetic canopy, 4 streams per hemisphere (radsurf_config.F90:61-64 default; "
                            "test/rami5/config.nam)",
                  "roofline": r4, "kernel_times_one_step": kt4,
                  "conservation_max_abs_residual_over_top_flux": res4, "nonfinite_outputs": nonfinite4}
            if not args.no_cpu_baseline:
                s4["parity_vs_truth"] = p4.parity_vs_truth(min(64, args.truth_columns), host_threads())
            extra["s4"] = s4
            del p4

        conf = workload_config(args, total_columns, world, ncol, args.weak)
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak" if args.weak else "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": conf,
            "roofline": roofline, "roofline_kernels": roofline_kernels, "kernel_times_one_step": kt,
            "fp64_tflops_measured": {"this_run": fp64_peak, "tracked": fp64_rec or None},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "conservation_max_abs_residual_over_top_flux": res, "nonfinite_outputs": nonfinite,
            "parity_vs_truth": parity_truth, "parity_vs_oracle_fp64_sample": parity_sample,
            "oracle_flops_measured": flops_measured, "weak_scaling": weak, "extra": extra,
            "library": lib.ssb200_version().decode(),
            "kernels": "generic (test-only)" if args.generic else "register-resident layer / sweep kernels on level-major staged arrays, columns ordered by segment pattern, SW and LW passes on two streams",
        }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(out) + "\n").encode())


if __name__ == "__main__":
    main()
