"""Scratch bytes per (column, layer) of the register-resident sweeps on the benchmark canopy.

Counts, from the element offsets and the load / store sites of csrc/ssb_sweep_blocks.cuh and
csrc/ssb_fast_sweeps.cuh, the doubles each (column, interval) moves through the two scratch areas:

  * interface scratch: stored by the upward pass (the state a_above, d_above / source_above at every
    level, pruned to what the consumer layer reads, interface_store_pruned; in the `with_lu_in_scratch`
    column also the NA^2 LU factors of D_AA = I - a_AA R_AA, which the downward pass now rebuilds) and
    loaded by the downward pass;
  * layer scratch: written by the layer kernels (block of each segment type, geometry block not
    counted) and read by the upward and the downward pass (each element counted once per pass).

A layer solves all regions (segment 0), only the clear one (1) or only the vegetated ones (2); the
segment of every layer comes from the benchmark's synthetic canopy (bench.py: 16 layers, nreg 3,
vegetated urban, no flux profiles, so the pruned interface store applies).  The result is a count of
the bytes the code asks for, not a DRAM measurement: re-reads served by L1 / L2 are not counted twice,
evictions are not modelled.

    python profiles/scratch_bytes.py [--streams 2] [--columns 65536]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def block(seg, nreg, ns):
    """(NA, I0) of the stream block a layer of segment `seg` solves."""
    n = nreg * ns
    if nreg == 1 or seg == 0:
        return n, 0
    if seg == 1:
        return ns, 0
    return n - ns, ns


def interface_counts(seg, first, nreg, ns, lw, with_lu):
    """(stored, loaded) interface doubles at the level below a layer of segment `seg`
    (`first`: the ground level, always stored in full, every row read)."""
    n, d = nreg * ns, nreg
    na, _ = block(seg, nreg, ns)
    da = na // ns
    vec_full = n if lw else n * d
    full = first or na == n
    if full:
        stored = n * n + vec_full
        loaded = n * n + (n if lw else n * da)  # every row of a_above; the block's DA columns of d_above
    else:
        a_part = na * n + (n - na) * na       # rows and columns of a_above that touch the block
        v_part = na * (1 if lw else da)       # block rows of source_above / d_above
        stored = loaded = a_part + v_part
    if with_lu:
        stored += na * na
        loaded += na * na
    return stored, loaded


def layer_counts(seg, nreg, ns, lw):
    """(written by the layer kernels, read by the upward pass, read by the downward pass)."""
    n, d = nreg * ns, nreg
    na, _ = block(seg, nreg, ns)
    da = na // ns
    if lw:
        book = 3 * d + 1
        written = 3 * na * na + 2 * na + book
        up = 2 * na * na + na                         # R, T, source
        down = 3 * na * na + 2 * na + book + 7        # T, R, int_flux, source, int_source, bookkeeping, geometry
    else:
        written = 3 * na * na + 3 * na * da + 2 * da * da
        up = 2 * na * na + 2 * na * da + da * da + 1  # R, T, S_up, S_dn, E, segment
        down = 3 * na * na + 3 * na * da + 2 * da * da + 8
    return written, up, down


def canopy_segments(ncol, streams):
    import bench
    from spartacus_surface_b200.synthetic import make_synthetic
    import oracle_lib
    cfg = bench.make_config(streams).consolidate(oracle_lib.legendre_gauss_init)
    cp, _, _ = make_synthetic(cfg, ncol, bench.NLAY)
    vf, bf = np.asarray(cp.veg_fraction), np.asarray(cp.building_fraction)
    mv = cfg.min_vegetation_fraction
    seg = np.where(vf <= mv, 1, np.where(1.0 - bf - vf <= mv, 2, 0))
    return seg.reshape(ncol, bench.NLAY), cfg


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=2)
    ap.add_argument("--columns", type=int, default=65536)
    args = ap.parse_args()
    seg, cfg = canopy_segments(args.columns, args.streams)
    nreg, ns = 3, args.streams
    ncl = seg.size
    out = {"canopy": f"bench.py synthetic canopy, first {args.columns} columns x {seg.shape[1]} layers, nreg {nreg}, "
                     f"{ns} streams, no flux profiles",
           "segment_mix": {k: float((seg == v).mean()) for k, v in (("all_regions", 0), ("clear_only", 1),
                                                                    ("vegetated_only", 2))},
           "unit": "bytes per (column, layer) and interval"}
    for lw in (False, True):
        res = {}
        for tag, with_lu in (("with_lu_in_scratch", True), ("lu_rebuilt", False)):
            st = ld = 0
            for l in range(seg.shape[1]):
                for s in (0, 1, 2):
                    cnt = int((seg[:, l] == s).sum())
                    if cnt:
                        a, b = interface_counts(s, l == 0, nreg, ns, lw, with_lu)
                        st += cnt * a
                        ld += cnt * b
            lw_, lu_, ldn = 0, 0, 0
            for s in (0, 1, 2):
                cnt = int((seg == s).sum())
                w, u, dn = layer_counts(s, nreg, ns, lw)
                lw_ += cnt * w
                lu_ += cnt * u
                ldn += cnt * dn
            res[tag] = {"interface_written": 8 * st / ncl, "interface_read": 8 * ld / ncl,
                        "layer_written": 8 * lw_ / ncl, "layer_read_by_sweeps": 8 * (lu_ + ldn) / ncl,
                        "sweeps_total": 8 * (st + ld + lu_ + ldn) / ncl}
        out["lw" if lw else "sw"] = res
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
