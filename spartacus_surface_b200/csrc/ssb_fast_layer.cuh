// ssb_fast_layer.cuh - register-resident layer problems: one thread per
// (column, interval, layer) with compile-time (NREG regions, NS streams).
// Same inputs, outputs and scratch layout as layer_problem_sw/_lw of
// ssb_solver.cuh (radsurf_urban_sw.F90:335-585, radsurf_urban_lw.F90:296-546
// and the forest equivalents); the layer matrices come from ssb_layer_math.cuh.
#pragma once
#include "ssb_layer_math.cuh"
#include "ssb_solver.cuh"

namespace ssb {

struct LayerOptics {
  double ext[3], ssa[3], planck[3];
  double wall_ext, wall_factor;
  double zcos, cos_sza, tan0, sin0, dz;
  double vssa, vplanck, vaplanck, ve;
};

// scalar description of the Gamma matrices of the solved block (regions R0 .. R0+NR-1)
template <int NREG, int NS, int NR, int R0>
SSB_HDI void fill_layer_coef(const ClassArgs &a, const LayerGeom &gm, const LayerOptics &op, LayerCoef<NR, NS> &k) {
  k.set_streams(&a.lg);
  SSB_UNROLL
  for (int rf = 0; rf < NR; ++rf) {
    const int Rf = R0 + rf;
    double loss = 0.0;
    SSB_UNROLL
    for (int Rt = 0; Rt < NREG; ++Rt) {
      if (Rt == Rf) continue;
      const double fx = gm.f_exchange[Rt + 3 * Rf];
      loss += fx;
      if (Rt >= R0 && Rt < R0 + NR) k.dx[(Rt - R0) + NR * rf] = fx;
    }
    k.loss[rf] = loss;
    k.ext[rf] = op.ext[Rf];
    k.es[rf] = op.ext[Rf] * op.ssa[Rf];
    k.fw[rf] = a.cfg.urban ? gm.f_wall[Rf] : 0.0;
    k.frac[rf] = (NR == 1) ? 1.0 : gm.frac[Rf];
    k.rfrac[rf] = (NR == 1) ? 1.0 : 1.0 / gm.frac[Rf];
  }
  k.wall_ext = op.wall_ext;
  k.wall_factor = op.wall_factor;
}

template <int NREG, int NS, int NR, int R0>
SSB_HDI void fast_sw_branch(const ClassArgs &a, int q, int lev, const LayerGeom &gm, const LayerOptics &op,
                            const StateMem &st) {
  LayerCoef<NR, NS> k;
  fill_layer_coef<NREG, NS, NR, R0>(a, gm, op, k);
  k.tan0 = op.tan0;
  k.sin0 = op.sin0;
  k.rcos = 1.0 / (a.cfg.urban ? op.zcos : op.cos_sza);
  double *P = a.layer + layer_sidx(a, 0, lev, q);
  const bool ok = layer_sw_solve<NREG, NS, NR, R0>(k, op.dz, P, st);
  count_failure(a.status, ok ? 0 : 1);
}

SSB_HDI void load_geometry_inputs(const ClassArgs &a, int il, double &bf, double &bs, double &vf, double &vs,
                                  double &ve, double &vcf, double &vfsd) {
  const SolveCfg &c = a.cfg;
  const bool veg = c.nreg > 1 || !c.urban;
  bf = c.urban ? a.cp.building_fraction[il] : 0.0;
  bs = c.urban ? a.cp.building_scale[il] : 0.0;
  vf = (veg && a.cp.veg_fraction) ? a.cp.veg_fraction[il] : 0.0;
  vs = (veg && a.cp.veg_scale) ? a.cp.veg_scale[il] : 1.0;
  ve = (veg && a.cp.veg_ext) ? a.cp.veg_ext[il] : 0.0;
  vcf = (c.urban && c.nreg > 1 && a.cp.veg_contact_fraction) ? a.cp.veg_contact_fraction[il] : 0.0;
  vfsd = (c.nreg == 3) ? a.cp.veg_fsd[il] : 0.0;
}

// layer geometry from the geometry block of the layer scratch (written by fast_prepare_level)
template <int NREG>
SSB_HDI void load_layer_geom(const ClassArgs &a, int q, int lev, LayerGeom &gm) {
  const double *P = a.layer + layer_sidx(a, a.ne_layer_geo, lev, q);
  SSB_UNROLL
  for (int i = 0; i < 9; ++i) gm.f_exchange[i] = 0.0;
  SSB_UNROLL
  for (int r = 0; r < 3; ++r) {
    gm.f_wall[r] = P[(size_t)r * kScratchTile];
    gm.od_scaling[r] = P[(size_t)(3 + r) * kScratchTile];
    gm.frac[r] = P[(size_t)(8 + r) * kScratchTile];
    gm.norm_perim_wall[r] = P[(size_t)(17 + r) * kScratchTile];
    gm.norm_perim[r] = 0.0;  // (only used to derive the exchange rates)
  }
  if (NREG > 1) {
    SSB_UNROLL
    for (int i = 0; i < 6; ++i) gm.f_exchange[geo_exchange_index(i)] = P[(size_t)(11 + i) * kScratchTile];
  }
  gm.f_wall_dir_clear = P[(size_t)6 * kScratchTile];
  const int seg = (int)P[(size_t)7 * kScratchTile];
  gm.r0 = (seg == 2) ? 1 : 0;
  gm.nr = (seg == 0) ? NREG : (seg == 1 ? 1 : NREG - 1);
}

// which sub-block of regions a layer solves: 0 = all regions, 1 = clear region only,
// 2 = vegetated regions only (radsurf_urban_sw.F90:512-583)
SSB_HDI int branch_segment(const LayerGeom &gm, int nreg) {
  if (gm.nr == nreg) return 0;
  return gm.r0 == 0 ? 1 : 2;
}

// inputs of one shortwave layer problem; false when the problem is skipped
template <int NREG, int NS>
SSB_HDI bool fast_sw_prepare(const ClassArgs &a, int q, int lev, LayerGeom &gm, LayerOptics &op) {
  const SolveCfg &c = a.cfg;
  const int nspec = c.nspec;
  const int ic = q / nspec, g = q % nspec;
  const int col = a.cols[ic];
  if (lev >= a.nlay[col]) return false;
  op.cos_sza = a.cp.cos_sza[col];
  if (!(op.cos_sza > 0.0)) return false;
  const int il = layer_index(a, ic, col, lev);
  op.zcos = c.urban ? dmax(op.cos_sza, 1.0e-6) : op.cos_sza;
  op.sin0 = 0.0;
  if (c.urban) {
    op.sin0 = sqrt(1.0 - op.zcos * op.zcos);
    op.tan0 = op.sin0 / op.zcos;
  } else {
    op.tan0 = sqrt(1.0 - op.cos_sza * op.cos_sza) / dmax(op.cos_sza, 1.0e-6);
  }
  op.dz = a.cp.dz[il];
  load_layer_geom<NREG>(a, q, lev, gm);
  const double ve = ((NREG > 1 || !c.urban) && a.cp.veg_ext) ? a.cp.veg_ext[il] : 0.0;
  op.ext[0] = SSB_LAY(a.sw.air_ext, g, il);
  op.ssa[0] = SSB_LAY(a.sw.air_ssa, g, il);
  SSB_UNROLL
  for (int r = 1; r < NREG; ++r) {
    const double vssa = SSB_LAY(a.sw.veg_ssa, g, il);
    const double od = (NREG == 2) ? 1.0 : gm.od_scaling[r];
    op.ext[r] = op.ext[0] + od * ve;
    op.ssa[r] = (op.ext[0] * op.ssa[0] + od * ve * vssa) / dmax(op.ext[r], 1.0e-8);
  }
  op.wall_ext = 0.0;
  op.wall_factor = 0.0;
  if (c.urban) {
    const double wa = SSB_LAY(a.sw.wall_albedo, g, il), wsf = SSB_LAY(a.sw.wall_specular_frac, g, il);
    op.wall_ext = 1.0 - wa * wsf;
    op.wall_factor = wa * (1.0 - wsf);
  }
  return true;
}

template <int NREG, int NS>
SSB_HD inline void fast_layer_problem_sw(const ClassArgs &a, int q, int lev, const StateMem &st) {
  LayerGeom gm;
  LayerOptics op;
  if (!fast_sw_prepare<NREG, NS>(a, q, lev, gm, op)) return;
  const int seg = branch_segment(gm, NREG);
  if (seg == 0) {
    fast_sw_branch<NREG, NS, NREG, 0>(a, q, lev, gm, op, st);
  } else if (seg == 1) {
    fast_sw_branch<NREG, NS, 1, 0>(a, q, lev, gm, op, st);  // vegetation-free layer: clear region only
  } else {
    if (NREG > 1) fast_sw_branch<NREG, NS, (NREG > 1 ? NREG - 1 : 1), (NREG > 1 ? 1 : 0)>(a, q, lev, gm, op, st);
  }
}

// one pre-classified problem: SEG is known at compile time, so only one sub-block size is instantiated
template <int NREG, int NS, int SEG>
SSB_HDI void fast_layer_problem_sw_seg(const ClassArgs &a, int q, int lev, const StateMem &st) {
  LayerGeom gm;
  LayerOptics op;
  if (!fast_sw_prepare<NREG, NS>(a, q, lev, gm, op)) return;
  constexpr int NR = (SEG == 0) ? NREG : (SEG == 1 ? 1 : (NREG > 1 ? NREG - 1 : 1));
  constexpr int R0 = (SEG == 2 && NREG > 1) ? 1 : 0;
  fast_sw_branch<NREG, NS, NR, R0>(a, q, lev, gm, op, st);
}

template <int NREG, int NS, int NR, int R0>
SSB_HDI void fast_lw_branch(const ClassArgs &a, int q, int lev, const LayerGeom &gm, const LayerOptics &op,
                            double wall_emission, const StateMem &st) {
  constexpr int N = NR * NS;
  LayerCoef<NR, NS> k;
  fill_layer_coef<NREG, NS, NR, R0>(a, gm, op, k);
  k.tan0 = k.sin0 = k.rcos = 0.0;
  double brate[N];
  SSB_UNROLL
  for (int r = 0; r < NR; ++r) {
    const int Rr = R0 + r;
    const double volume_emiss = gm.frac[Rr] * (op.ext[Rr] * (1.0 - op.ssa[Rr]) * op.planck[Rr]);
    const double wall_emiss = a.cfg.urban ? gm.norm_perim_wall[Rr] * a.lg.vadjustment * wall_emission : 0.0;
    SSB_UNROLL
    for (int js = 0; js < NS; ++js)
      brate[js + r * NS] = (a.lg.hweight[js] / a.lg.mu[js]) * volume_emiss + (0.5 * a.lg.vweight[js]) * wall_emiss;
  }
  double *P = a.layer + layer_sidx(a, 0, lev, q);
  const bool ok = layer_lw_solve<NREG, NS, NR, R0>(k, brate, op.dz, P, st);
  count_failure(a.status, ok ? 0 : 1);
}

// inputs of one longwave layer problem (also writes the emission bookkeeping terms); SEG < 0: dispatch at run time
template <int NREG, int NS, int SEG>
SSB_HDI void fast_layer_problem_lw_impl(const ClassArgs &a, int q, int lev, const StateMem &st) {
  const SolveCfg &c = a.cfg;
  const int nspec = c.nspec;
  const int ic = q / nspec, g = q % nspec;
  const int col = a.cols[ic];
  if (lev >= a.nlay[col]) return;
  const int il = layer_index(a, ic, col, lev);
  LayerOptics op;
  op.dz = a.cp.dz[il];
  LayerGeom gm;
  load_layer_geom<NREG>(a, q, lev, gm);
  const double ve = ((NREG > 1 || !c.urban) && a.cp.veg_ext) ? a.cp.veg_ext[il] : 0.0;
  op.ext[0] = SSB_LAY(a.lw.air_ext, g, il);
  op.ssa[0] = SSB_LAY(a.lw.air_ssa, g, il);
  op.planck[0] = SSB_LAY(a.lw.clear_air_planck, g, il);
  double vssa = 0.0, vplanck = 0.0, vaplanck = 0.0;
  if (NREG > 1) {
    vssa = SSB_LAY(a.lw.veg_ssa, g, il);
    vplanck = SSB_LAY(a.lw.veg_planck, g, il);
    vaplanck = SSB_LAY(a.lw.veg_air_planck, g, il);
  }
  SSB_UNROLL
  for (int r = 1; r < NREG; ++r) {
    const double od = (NREG == 2) ? 1.0 : gm.od_scaling[r];
    op.ext[r] = op.ext[0] + od * ve;
    op.ssa[r] = (op.ext[0] * op.ssa[0] + od * ve * vssa) / dmax(op.ext[r], 1.0e-8);
    op.planck[r] = (op.ext[0] * (1.0 - op.ssa[0]) * vaplanck + od * ve * (1.0 - vssa) * vplanck) /
                   dmax(op.ext[r] * (1.0 - op.ssa[r]), 1.0e-8);
  }
  op.wall_ext = 1.0;
  op.wall_factor = c.urban ? 1.0 - SSB_LAY(a.lw.wall_emissivity, 0, il) : 0.0;
  const double wall_emission = c.urban ? SSB_LAY(a.lw.wall_emission, g, il) : 0.0;

  // bookkeeping terms of urban_lw:447-476 for all regions (same as the generic path)
  constexpr int n = NREG * NS, d = NREG;
  double emiss_factor = 0.0;
  SSB_UNROLL
  for (int js = 0; js < NS; ++js) emiss_factor += a.lg.hweight[js] / a.lg.mu[js];
  emiss_factor = 2.0 * emiss_factor;
  const int e_book = 3 * n * n + 2 * n;
  double wsum = 0.0;
  SSB_UNROLL
  for (int Rr = 0; Rr < NREG; ++Rr) {
    const double volume_emiss = gm.frac[Rr] * (op.ext[Rr] * (1.0 - op.ssa[Rr]) * op.planck[Rr]);
    a.layer[layer_sidx(a, e_book + Rr, lev, q)] = emiss_factor * volume_emiss;
    double e_air = 0.0, e_veg = 0.0;
    if (Rr > 0) {
      e_air = emiss_factor * gm.frac[Rr] * op.ext[0] * (1.0 - op.ssa[0]) * vaplanck;
      e_veg = emiss_factor * gm.frac[Rr] * ve * (1.0 - vssa) * vplanck * gm.od_scaling[Rr];
    }
    a.layer[layer_sidx(a, e_book + d + Rr, lev, q)] = e_air;
    a.layer[layer_sidx(a, e_book + 2 * d + Rr, lev, q)] = e_veg;
    wsum += gm.norm_perim_wall[Rr];
  }
  a.layer[layer_sidx(a, e_book + 3 * d, lev, q)] = c.urban ? (wsum * a.lg.vadjustment) * wall_emission : 0.0;

  if (SEG >= 0) {
    constexpr int NR = (SEG <= 0) ? NREG : (SEG == 1 ? 1 : (NREG > 1 ? NREG - 1 : 1));
    constexpr int R0 = (SEG == 2 && NREG > 1) ? 1 : 0;
    fast_lw_branch<NREG, NS, NR, R0>(a, q, lev, gm, op, wall_emission, st);
    return;
  }
  const int seg = branch_segment(gm, NREG);
  if (seg == 0) {
    fast_lw_branch<NREG, NS, NREG, 0>(a, q, lev, gm, op, wall_emission, st);
  } else if (seg == 1) {
    fast_lw_branch<NREG, NS, 1, 0>(a, q, lev, gm, op, wall_emission, st);
  } else {
    if (NREG > 1)
      fast_lw_branch<NREG, NS, (NREG > 1 ? NREG - 1 : 1), (NREG > 1 ? 1 : 0)>(a, q, lev, gm, op, wall_emission, st);
  }
}

template <int NREG, int NS>
SSB_HD inline void fast_layer_problem_lw(const ClassArgs &a, int q, int lev, const StateMem &st) {
  fast_layer_problem_lw_impl<NREG, NS, -1>(a, q, lev, st);
}

// Sort key of a column for the register-resident kernels: bit l is set when layer l solves
// only a sub-block of its regions (same rule as layer_geometry: radsurf_urban_sw.F90:512-583).
// Columns with equal keys take the same code path layer by layer, so ordering the columns of
// a launch by this key makes warps uniform: the segment kernels write, and the sweeps skip,
// whole 32-byte sectors.  Night-time columns (shortwave) go last.  T: element type of the
// per-layer fractions (float for the caller's arrays of ssb200_radsurf_device_sp).
template <class T = double>
SSB_HDI unsigned column_segment_key(const ClassArgs &a, int col) {
  const SolveCfg &c = a.cfg;
  if (!c.lw && !(a.cp.cos_sza[col] > 0.0)) return 0xffffffffu;
  const bool veg_branching = c.urban ? (c.nreg > 1) : true;
  if (!veg_branching) return 0u;
  const int nlay = a.nlay[col], il1 = a.istartlay[col] - 1;
  const bool veg = c.nreg > 1 || !c.urban;
  unsigned key = 0u;
  for (int l = 0; l < nlay && l < 31; ++l) {
    const double bf = c.urban ? (double)((const T *)a.cp.building_fraction)[il1 + l] : 0.0;
    const double vf = (veg && a.cp.veg_fraction) ? (double)((const T *)a.cp.veg_fraction)[il1 + l] : 0.0;
    double frac[3];
    region_fractions(c, bf, vf, frac);
    if (vf <= c.min_veg || frac[0] <= c.min_veg) key |= 1u << l;
  }
  return key;
}

// Per layer problem (q, level k) preparation for the register-resident kernels: writes the
// geometry block of the layer scratch and returns the segment of the problem (which
// sub-block of regions it solves), -1 when there is none.
SSB_HDI int fast_prepare_level(const ClassArgs &a, int q, int k) {
  const SolveCfg &c = a.cfg;
  const int ic = q / c.nspec, col = a.cols[ic];
  if (k >= a.nlay[col]) return -1;
  if (!c.lw && !(a.cp.cos_sza[col] > 0.0)) return -1;
  const int il = layer_index(a, ic, col, k);
  double bf, bs, vf, vs, ve, vcf, vfsd;
  load_geometry_inputs(a, il, bf, bs, vf, vs, ve, vcf, vfsd);
  LayerGeom gm;
  layer_geometry(c, bf, bs, vf, vs, vcf, vfsd, c.lw ? a.lg.vadjustment2 : 1.0, gm);
  const int seg = branch_segment(gm, c.nreg);
  double *P = a.layer + layer_sidx(a, a.ne_layer_geo, k, q);
  for (int r = 0; r < 3; ++r) {
    P[(size_t)r * kScratchTile] = gm.f_wall[r];
    P[(size_t)(3 + r) * kScratchTile] = gm.od_scaling[r];
    P[(size_t)(8 + r) * kScratchTile] = gm.frac[r];
    P[(size_t)(17 + r) * kScratchTile] = gm.norm_perim_wall[r];
  }
  for (int i = 0; i < 6; ++i) P[(size_t)(11 + i) * kScratchTile] = gm.f_exchange[geo_exchange_index(i)];
  P[(size_t)6 * kScratchTile] = gm.f_wall_dir_clear;
  P[(size_t)7 * kScratchTile] = (double)seg;
  return seg;
}

}  // namespace ssb
